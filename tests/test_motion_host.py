"""CPU: the moving-object test of include/dca_b200.h section 16 through its numpy restatement
(tests/_motion_restatement.py) on analytic scenes rendered at KITTI intrinsics (a road, a wall at 60 m and a box, the
camera moving 1 m forward per frame), fuse_files / track_files with motion= and the kernels replaced by their
restatements, and the argument checks of the Python API and of the C entry points.

The scene bounds are measured values with a margin; they say nothing about KITTI or any real camera."""
import importlib
import math
import os

import numpy as np
import pytest
import torch
from PIL import Image

import _motion_restatement as R
import _reproject_restatement as RP
import _tsdf_restatement as RT
import dcanet_b200 as d

mo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.motion")
fu = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.fusion")
geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")

F32 = np.float32
K = RP.kitti_scene()
CALIB = geo.StereoCalib(K["fx"], K["fy"], K["cx"], K["cy"], 0.54)
INTR = (CALIB.fx, CALIB.fy, CALIB.cx, CALIB.cy)
H, W = 375, 1242
GROUND, WALL = 1.65, 60.0                    # world: X right, Y down, Z forward; the camera starts at the origin
# 1.8 m wide, 1.8 m tall and 1 m deep, front face at Z = 0: its top is above the camera, so only the front face and the
# sides are seen
BOX = (np.array([-0.9, GROUND - 1.8, 0.0]), np.array([0.9, GROUND, 1.0]))


def pose(i, err=None):
    """camera-to-world of frame i: 1 m forward per frame; err = (translation m, rotation deg) added about the X axis."""
    p = np.eye(4)
    p[2, 3] = float(i)
    if err is not None:
        t, a = err
        c, s = math.cos(math.radians(a)), math.sin(math.radians(a))
        p[:3, :3] = np.array([[1, 0, 0], [0, c, -s], [0, s, c]])
        p[:3, 3] += t / math.sqrt(3)
    return p


def render(cam_to_world, box_at=None, win=(0, 0, W, H)):
    """Float64 ray cast of road, wall and the box moved to box_at (world offset), as float32 depth [h, w]."""
    u0, v0, w, h = win
    u, v = np.meshgrid(np.arange(w) + u0, np.arange(h) + v0)
    dcam = np.stack([(u - INTR[2]) / INTR[0], (v - INTR[3]) / INTR[1], np.ones(u.shape)], -1)
    Rm, C = cam_to_world[:3, :3], cam_to_world[:3, 3]
    dw = dcam @ Rm.T
    best = np.full(u.shape, np.inf)
    with np.errstate(divide="ignore", invalid="ignore"):
        for t in ((GROUND - C[1]) / dw[..., 1], (WALL - C[2]) / dw[..., 2]):
            best = np.where(t > 0, np.minimum(best, t), best)
        if box_at is not None:
            lo, hi = BOX[0] + box_at, BOX[1] + box_at
            t0, t1 = (lo - C) / dw, (hi - C) / dw
            tn, tf = np.minimum(t0, t1).max(-1), np.maximum(t0, t1).min(-1)
            best = np.where((tn <= tf) & (tn > 0), np.minimum(best, tn), best)
    return np.where(np.isfinite(best), best, 0).astype(F32)      # camera Z: the direction's Z component is 1


def box_image(cam_to_world, box_at):
    """Pixel bounds (x_min, y_min, x_max, y_max) of the box's front face."""
    lo, hi = BOX[0] + box_at, BOX[1] + box_at
    Z = lo[2] - cam_to_world[2, 3]
    xs = [INTR[0] * (X - cam_to_world[0, 3]) / Z + INTR[2] for X in (lo[0], hi[0])]
    ys = [INTR[1] * (Y - cam_to_world[1, 3]) / Z + INTR[3] for Y in (lo[1], hi[1])]
    return xs[0], ys[0], xs[1], ys[1]


def run(depth, prev, A, **kw):
    fB = CALIB.focal_baseline
    lab, res = R.labels(depth[None], prev[None], INTR, fB, 0.0, 0, 0, A[None], **{k: v for k, v in kw.items()
                                                                                   if k in ("tau", "tau_rel", "radius")})
    comp = R.components(depth[None], lab, res, INTR, fB, 0.0, 0, 0,
                        **{k: v for k, v in kw.items() if k in ("gate", "min_pixels")})
    return lab[0], res[0], comp


def rel(i, j=None, err=None):
    """T(frame i-1 <- frame i), float32 [12], from the (perturbed) float64 poses."""
    j = i - 1 if j is None else j
    return np.linalg.solve(pose(j), pose(i, err))[:3].reshape(12).astype(F32)


def depth_edges(depth, grow=2):
    disp = CALIB.focal_baseline / np.where(depth > 0, depth, np.inf)
    e = np.zeros(depth.shape, bool)
    e[:, 1:] |= np.abs(np.diff(disp, axis=1)) > 1
    e[1:, :] |= np.abs(np.diff(disp, axis=0)) > 1
    for _ in range(grow):
        e[1:] |= e[:-1]; e[:-1] |= e[1:]; e[:, 1:] |= e[:, :-1]; e[:, :-1] |= e[:, 1:]
    return e


# ---- the two-frame test --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("box", [False, True])
def test_a_static_scene_has_no_moving_object(box):
    at = np.array([1.5, 0.0, 16.0]) if box else None
    prev, cur = render(pose(0), at), render(pose(1), at)
    lab, res, comp = run(cur, prev, rel(1))
    moving = (lab == R.APPEARED) | (lab == R.BEHIND)
    assert not (moving & ~depth_edges(cur)).any()
    assert comp["count"][0] == 0 and comp["dropped"][0] == 0 and (comp["instance"] == 0).all()
    assert (lab == R.STATIC).mean() > 0.95
    assert np.nanmax(np.abs(res[lab == R.STATIC])) < 3.0


def test_background_uncovered_beside_a_near_static_box_is_behind():
    """Two depth maps cannot tell background uncovered by the ego-motion from a surface that moved away: beside a static
    box 8 m ahead, the wall and road that the box hid at t-1 form a BEHIND band as wide as the parallax,
    0.6 m fx (1/8 - 1/9) = 6 px (measured: 3 columns, 168 pixels, one object at the default min_pixels).  Fusion only
    loses those pixels' weight for one frame."""
    at = np.array([1.5, 0.0, 9.0])
    prev, cur = render(pose(0), at), render(pose(1), at)
    lab, _, comp = run(cur, prev, rel(1))
    moving = (lab == R.APPEARED) | (lab == R.BEHIND)
    assert not (moving & ~depth_edges(cur, grow=10)).any() and not (lab == R.APPEARED).any()
    bx = box_image(pose(1), at)
    for k in range(comp["count"][0]):
        n, app, beh, x0, y0, x1, y1, _ = comp["ints"][0, k]
        assert beh == n and n < 400 and x1 < bx[0] and x1 - x0 < 8


def test_the_tracking_error_makes_no_object():
    """The README's tracking error on KITTI: 3.3 mm and 0.02 deg per frame."""
    at = np.array([1.5, 0.0, 16.0])
    prev, cur = render(pose(0), at), render(pose(1), at)
    for err in ((0.0033, 0.02), (-0.0033, -0.02)):
        lab, _, comp = run(cur, prev, rel(1, err=err))
        assert comp["count"][0] == 0, err
        assert (lab == R.STATIC).mean() > 0.95


def _moving_box(start, step):
    """(prev depth, current depth, box offset now) for a box at `start` (world, frame 0) moving `step` per frame."""
    start, step = np.asarray(start, float), np.asarray(step, float)
    return render(pose(0), start), render(pose(1), start + step), start + step


def test_an_approaching_box_appeared():
    prev, cur, at = _moving_box([0.0, 0.0, 10.0], [0.0, 0.0, -2.0])
    lab, _, comp = run(cur, prev, rel(1))
    assert comp["count"][0] == 1
    n, app, beh, x0, y0, x1, y1, _ = comp["ints"][0, 0]
    bx = box_image(pose(1), at)
    assert app > 0.9 * n
    # the lowest rows can pass: there the road of the previous frame held the expected depth (measured: 12 rows)
    assert x0 <= bx[0] + 1 and y0 <= bx[1] + 1 and x1 >= bx[2] - 1 and y1 >= bx[3] - 16
    assert x0 >= bx[0] - 3 and x1 <= bx[2] + 3
    ext = comp["extent"][0, 0]
    assert ext[4] == pytest.approx(at[2] - 1.0, abs=0.01)              # the front face, 1 m behind the camera's move


@pytest.mark.parametrize("step", [2.0, 1.0], ids=["receding", "ego_speed"])
def test_a_receding_or_followed_box_is_behind(step):
    prev, cur, at = _moving_box([0.0, 0.0, 8.0], [0.0, 0.0, step])
    lab, _, comp = run(cur, prev, rel(1))
    assert comp["count"][0] == 1
    n, app, beh = comp["ints"][0, 0, :3]
    assert beh > 0.9 * n
    bx = box_image(pose(1), at)
    x0, y0, x1, y1 = comp["ints"][0, 0, 3:7]
    assert x0 <= bx[0] + 1 and x1 >= bx[2] - 1 and y0 <= bx[1] + 1


def test_a_lateral_mover_has_a_leading_and_a_trailing_part():
    prev, cur, at = _moving_box([-2.0, 0.0, 10.0], [1.0, 0.0, 0.0])
    lab, _, comp = run(cur, prev, rel(1))
    k = comp["count"][0]
    assert k >= 2
    rows = comp["ints"][0, :k]
    lead = [r for r in rows if r[1] == r[0]]
    trail = [r for r in rows if r[2] == r[0]]
    assert len(lead) + len(trail) == k
    bx = box_image(pose(1), at)
    # measured: the front face's leading 1 m (72 columns, 9,576 pixels) and its 1-column side face; the uncovered
    # background on the left (8,635 pixels), 1 m wide at the wall's and the road's disparities
    assert lead and max(r[5] for r in lead) >= bx[2] - 1 and all(r[3] > bx[0] + 50 for r in lead)
    assert trail and all(r[5] < bx[0] + 1 for r in trail) and sum(r[0] for r in trail) > 5000


# ---- the Python API with the restated kernels ----------------------------------------------------------------------
def _restated_labels(depth, prev, intrinsics, fB, doffs, u0, v0, A, tau, tau_rel, radius, label, residual):
    lab, res = R.labels(depth.numpy(), prev.numpy(), intrinsics, fB, doffs, u0, v0, A, tau, tau_rel, radius)
    label.copy_(torch.from_numpy(lab))
    residual.copy_(torch.from_numpy(res))


def _restated_components(depth, label, residual, intrinsics, fB, doffs, u0, v0, gate, min_pixels, instance, objects):
    c = R.components(depth.numpy(), label.numpy(), residual.numpy(), intrinsics, fB, doffs, u0, v0, gate, min_pixels)
    instance.copy_(torch.from_numpy(c["instance"]))
    for name in ("count", "dropped", "ints", "extent", "res_sum"):
        getattr(objects, name).copy_(torch.from_numpy(c[name]))


def _patch(monkeypatch, calls=None):
    def lab(*a):
        if calls is not None:
            calls.append(("labels", a[0].shape[0]))
        _restated_labels(*a)

    def comp(*a):
        if calls is not None:
            calls.append(("components", a[0].shape[0]))
        _restated_components(*a)
    monkeypatch.setattr(mo, "_labels_kernel", lab)
    monkeypatch.setattr(mo, "_components_kernel", comp)


def test_motion_splits_batches_of_16_and_reads_objects_on_request(monkeypatch):
    calls = []
    _patch(monkeypatch, calls)
    win = (0, 500, 120, 200, 150)                         # (y0, x0, h, w, v_origin)
    prev = np.stack([render(pose(0), np.array([0.0, 0.0, 10.0]), (500, 150, 200, 120))] * 18)
    cur = np.stack([render(pose(1), np.array([0.0, 0.0, 8.0]), (500, 150, 200, 120))] * 18)
    A = np.stack([np.linalg.solve(pose(0), pose(1))] * 18)
    m = d.motion(torch.from_numpy(cur)[:, None], torch.from_numpy(prev), CALIB, A, window=win, min_pixels=50)
    assert calls == [("labels", 16), ("labels", 2), ("components", 18)]
    want_l, want_r = R.labels(cur, prev, INTR, CALIB.focal_baseline, 0.0, 500, 150,
                              A[:, :3].reshape(18, 12).astype(F32))
    assert np.array_equal(m.label.numpy(), want_l) and np.array_equal(m.residual.numpy(), want_r, equal_nan=True)
    assert (m.objects.counts() == 1).all()
    o = m.objects.numpy(3)
    assert o["pixels"][0] > 1000 and o["appeared"][0] > 0.9 * o["pixels"][0] and o["box"].shape == (1, 4)
    assert math.isfinite(o["mean_residual"][0]) and o["mean_residual"][0] < -3


def _bad_calls():
    z = torch.ones(1, 8, 10)
    c = CALIB
    yield lambda: d.motion(np.ones((1, 8, 10), F32), z, c, np.eye(4))
    yield lambda: d.motion(z.double(), z, c, np.eye(4))
    yield lambda: d.motion(z, torch.ones(1, 8, 9), c, np.eye(4))
    yield lambda: d.motion(z, z, c, np.eye(4)[None].repeat(2, 0))
    yield lambda: d.motion(z, z, c, np.full((4, 4), np.nan))
    yield lambda: d.motion(z, z, c, np.eye(4) * 1e300)
    yield lambda: d.motion(z, z, c, np.eye(3))
    yield lambda: d.motion(z, z, c, np.eye(4), window=(0, 0, 8, 11, 0))
    yield lambda: d.motion(z, z, c, np.eye(4), tau=-1.0)
    yield lambda: d.motion(z, z, c, np.eye(4), tau=math.nan)
    yield lambda: d.motion(z, z, c, np.eye(4), tau_rel=math.inf)
    yield lambda: d.motion(z, z, c, np.eye(4), radius=5)
    yield lambda: d.motion(z, z, c, np.eye(4), radius=1.0)
    yield lambda: d.motion(z, z, c, np.eye(4), gate=-0.5)
    yield lambda: d.motion(z, z, c, np.eye(4), min_pixels=0)
    yield lambda: d.motion(z, z, c, np.eye(4), min_pixels=True)
    yield lambda: d.motion(torch.ones(0, 8, 10), torch.ones(0, 8, 10), c, np.zeros((0, 4, 4)))
    yield lambda: d.fuse_files(None, [], [], None, c, motion="yes")
    yield lambda: d.fuse_files(None, [], [], None, c, motion=dict(speed=1))
    yield lambda: d.fuse_files(None, [], [], None, c, motion=dict(radius=9))
    yield lambda: d.track_files(None, [], None, c, motion=dict(tau=-1))


@pytest.mark.parametrize("i", range(21))
def test_argument_errors_raise_before_any_launch(i):
    calls = list(_bad_calls())
    assert len(calls) == 21
    before = _lib.LAUNCHES
    with pytest.raises(ValueError):
        calls[i]()
    assert _lib.LAUNCHES == before


def test_cpu_tensors_are_refused():
    with pytest.raises(_lib.DcaError):
        d.motion(torch.ones(1, 8, 10), torch.ones(1, 8, 10), CALIB, np.eye(4))


def test_entry_points_reject_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    A = np.tile(np.eye(4)[:3].reshape(12), (16, 1)).astype(F32)
    nan = float("nan")
    ok = [p, p, 10, 80, 1, 8, 10, 700.0, 700.0, 5.0, 4.0, 0, 0, 380.0, 0.0, A.ctypes.data, 3.0, 0.05, 1, p, p, None]

    def lcall(**kw):
        args = list(ok)
        for k_, v in kw.items():
            args[int(k_[1:])] = v
        return lib.dca_motion_labels(*args)

    for i in (0, 1, 15, 19, 20):
        assert lcall(**{f"a{i}": None}) == -1, i
    assert lcall(a4=0) == lcall(a4=17) == lcall(a5=0) == lcall(a6=0) == lcall(a2=9) == lcall(a3=79) == -1
    assert lcall(a7=0.0) == lcall(a8=nan) == lcall(a9=math.inf) == lcall(a14=nan) == lcall(a13=0.0) == -1
    assert lcall(a16=-1.0) == lcall(a17=nan) == lcall(a18=-1) == lcall(a18=5) == -1
    Abad = A.copy()
    Abad[0, 3] = nan
    assert lcall(a15=Abad.ctypes.data) == -1
    assert lcall(a11=1 << 24) == lcall(a12=-(1 << 24)) == -3
    assert lcall(a6=1 << 24, a2=1 << 24, a3=8 << 24) == -3
    cok = [p, 10, 80, p, p, 1, 8, 10, 700.0, 700.0, 5.0, 4.0, 0, 0, 380.0, 0.0, 1.0, 100, p, p, p, p, p, p, p, None]

    def ccall(**kw):
        args = list(cok)
        for k_, v in kw.items():
            args[int(k_[1:])] = v
        return lib.dca_motion_components(*args)

    for i in (0, 3, 4) + tuple(range(18, 25)):
        assert ccall(**{f"a{i}": None}) == -1, i
    assert ccall(a5=0) == ccall(a5=65536) == ccall(a6=0) == ccall(a7=0) == ccall(a1=9) == ccall(a2=79) == -1
    assert ccall(a8=0.0) == ccall(a11=nan) == ccall(a14=-1.0) == ccall(a15=math.inf) == -1
    assert ccall(a16=-0.1) == ccall(a16=nan) == ccall(a17=0) == -1
    assert ccall(a13=1 << 24) == ccall(a7=1 << 24, a1=1 << 24, a2=8 << 24) == -3


# ---- fusion and tracking with motion= --------------------------------------------------------------------------------
GRID = dict(origin=(-4.0, -1.0, 1.0), voxel_size=0.1, dims=(80, 30, 220), trunc=0.3, colour=False, device="cpu")
N_FRAMES = 5
FWIN = (300, 60, 640, 300)                       # (u0, v0, w, h) of the depth maps


def _box_at(i):
    return np.array([0.0, 0.0, 20.0 - 3.0 * i])       # approaching at 3 m per frame (2 m beyond the ego-motion)


def _patch_pipeline(monkeypatch, integrate_calls):
    """FusePipeline with the analytic depth of each pair in order, and the TSDF integration by its restatement."""
    state = {"i": 0}

    def observe(self, slot, calib, window):
        i = state["i"]
        state["i"] += 1
        depth = torch.from_numpy(render(pose(i), _box_at(i), FWIN))[None]
        u0, v0, w, h = FWIN
        return depth, None, None, (0, u0, h, w, v0)

    def integrate(vol, box, depth, weight, rgb, intr, u0, v0, T, max_depth):
        integrate_calls.append((box, depth.clone(), None if weight is None else weight.clone(), T.copy()))
        RT.integrate(vol.state.numpy(), vol.origin, vol.voxel_size, depth.numpy(), T, intr, u0, v0,
                     weight=None if weight is None else weight.numpy(), trunc=vol.trunc, max_weight=vol.max_weight,
                     max_depth=max_depth, box=box)
    monkeypatch.setattr(fu.FusePipeline, "_observe", observe)
    monkeypatch.setattr(fu, "_integrate_kernel", integrate)
    _patch(monkeypatch)


def _items(tmp_path):
    items = []
    for i in range(N_FRAMES):
        for s in "lr":
            Image.fromarray(np.full((16, 16, 3), 10 * i, np.uint8)).save(tmp_path / f"{s}{i}.png")
        items.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png")))
    return items


class _NoModel(torch.nn.Module):
    def forward(self, *a, **k):
        raise AssertionError("the forward is replaced by the analytic depth")


def _fuse(tmp_path, monkeypatch, motion):
    calls = []
    _patch_pipeline(monkeypatch, calls)
    vol = fu.TSDFVolume(**GRID)
    poses = np.stack([pose(i) for i in range(N_FRAMES)])
    fu.fuse_files(_NoModel(), _items(tmp_path), poses, vol, CALIB, crop=(16, 16), max_depth=30.0, weight=None,
                  motion=motion)
    return vol, calls


def _near_boxes(xyz, frames, margin=0.2):
    """Surface points within `margin` of the box of each frame, above the road (the road under and around the box is
    seen from the other frames, and its crossings lie within the margin of the box's bottom face)."""
    out = []
    above = xyz[:, 1] < GROUND - margin
    for i in frames:
        lo, hi = BOX[0] + _box_at(i) - margin, BOX[1] + _box_at(i) + margin
        out.append(int((((xyz >= lo) & (xyz <= hi)).all(-1) & above).sum()))
    return out


def test_fuse_files_with_motion_leaves_no_ghost(tmp_path, monkeypatch):
    vol, calls = _fuse(tmp_path, monkeypatch, True)
    xyz, _, _ = RT.surface(vol.state.numpy(), vol.origin, vol.voxel_size, 0.5, False, False)
    assert _near_boxes(xyz, range(1, N_FRAMES)) == [0] * (N_FRAMES - 1)
    assert _near_boxes(xyz, [0])[0] > 100                                          # frame 0 has no reference
    assert calls[0][2] is None and all(c[2] is not None for c in calls[1:])
    for c in calls[1:]:
        assert 0 < int((c[2] == 0).sum()) < c[2].numel() // 2 and ((c[2] == 0) | (c[2] == 1)).all()
    ghost, _ = _fuse(tmp_path, monkeypatch, None)
    xyz, _, _ = RT.surface(ghost.state.numpy(), ghost.origin, ghost.voxel_size, 0.5, False, False)
    assert min(_near_boxes(xyz, range(1, N_FRAMES))) > 20
    assert len(xyz) > 5000


def test_motion_none_is_the_current_driver_call_for_call(tmp_path, monkeypatch):
    _, with_none = _fuse(tmp_path, monkeypatch, None)
    called = []
    monkeypatch.setattr(mo, "motion", lambda *a, **k: called.append(1))
    calls = []
    _patch_pipeline(monkeypatch, calls)
    vol = fu.TSDFVolume(**GRID)
    fu.fuse_files(_NoModel(), _items(tmp_path), np.stack([pose(i) for i in range(N_FRAMES)]), vol, CALIB,
                  crop=(16, 16), max_depth=30.0, weight=None)
    assert not called and len(calls) == len(with_none) == N_FRAMES
    for a, b in zip(calls, with_none):
        assert a[0] == b[0] and torch.equal(a[1], b[1]) and a[2] is None and b[2] is None and np.array_equal(a[3], b[3])


def test_track_files_masks_at_the_tracked_poses(tmp_path, monkeypatch):
    """track_files(motion=True): the reference of each frame is the last frame integrated, at its tracked pose; a frame
    that fails to track is not integrated and does not become the reference."""
    tr = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.tracking")
    calls = []
    _patch_pipeline(monkeypatch, calls)
    seen = []
    real = mo.motion

    def spy(depth, prev, calib, A, **kw):
        seen.append(np.asarray(A))
        return real(depth, prev, calib, A, **kw)
    monkeypatch.setattr(mo, "motion", spy)
    tracked = {1: pose(1), 2: None, 3: pose(3), 4: pose(4)}            # frame 2 fails

    def launch(self, depth, weight=None, init=None):
        return init

    def collect(self, guess):
        n = len(seen_frames)
        seen_frames.append(n)
        p = tracked[n + 1]
        return tr.TrackResult(p if p is not None else pose(n + 1), p is not None, np.zeros(1, np.int64), np.zeros(1))
    seen_frames = []
    monkeypatch.setattr(tr.Tracker, "_launch", launch)
    monkeypatch.setattr(tr.Tracker, "_collect", collect)
    vol = fu.TSDFVolume(**GRID)
    traj = tr.track_files(_NoModel(), _items(tmp_path), vol, CALIB, crop=(16, 16), max_depth=30.0, weight=None,
                          motion=True)
    assert list(traj.ok) == [True, True, False, True, True]
    assert len(calls) == 4 and len(seen) == 3
    want = [np.linalg.solve(pose(0), pose(1)), np.linalg.solve(pose(1), pose(3)), np.linalg.solve(pose(3), pose(4))]
    for a, b in zip(seen, want):
        assert np.allclose(a, b, atol=1e-12)
