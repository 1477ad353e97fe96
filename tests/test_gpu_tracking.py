"""GPU: the raycast and ICP tracking (csrc/track.cu) bit-exact against their restatement (tests/_track_restatement.py):
the raycast at odd grids and windows, with and without colour, two min_weights, pitched outputs, a pose outside the grid
and a window that misses the volume; ICP's final pose and every iteration's stats at every level, at a KITTI-sized
window too; no host sync and CUDA-graph capture; Tracker.track's one sync; the synthetic sequence end to end; and
track_files against a serial loop on the real forward."""
import importlib

import numpy as np
import pytest
import torch
from PIL import Image

import _track_restatement as TR
import _tsdf_restatement as R
from test_gpu_tsdf import _used_state
from test_tracking_host import CALIB, TRUNC, _perturbed, _restated_icp, _restated_raycast
from test_tsdf_host import GRID, INTR, WIN, _patch_integrate, fuse, look_at, render, trajectory

pytestmark = pytest.mark.gpu

fu = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.fusion")
tk = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.tracking")
geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")

F32 = np.float32


def _scene(n=6, frames=3):
    poses = trajectory(n)
    s = fuse(np.stack([render(p) for p in poses[:frames]]), poses[:frames])
    return poses, s


def _raycast_raw(state, origin, vs, trunc, min_weight, intr, u0, v0, H, W, M, min_depth, max_depth, pad=0):
    """dca_tsdf_raycast into outputs with `pad` extra elements per row (pitched) -> numpy maps."""
    st = torch.from_numpy(state).cuda()
    P, nz, ny, nx = state.shape
    depth = torch.full((H, W + pad), -5.0, device="cuda")
    vert = torch.full((H, 3 * W + pad), -5.0, device="cuda")
    nrm = torch.full((H, 3 * W + pad), -5.0, device="cuda")
    rgb = torch.full((H, 3 * W + pad), 9, dtype=torch.uint8, device="cuda") if P == 5 else None
    m = np.ascontiguousarray(M, F32).reshape(12)
    _lib.call("dca_tsdf_raycast", st.data_ptr(), P, nx, ny, nz, *[float(F32(o)) for o in origin], float(F32(vs)),
              float(F32(trunc)), float(min_weight), *intr, u0, v0, H, W, m.ctypes.data, float(min_depth),
              float(max_depth), depth.data_ptr(), W + pad, vert.data_ptr(), 3 * W + pad, nrm.data_ptr(), 3 * W + pad,
              0 if rgb is None else rgb.data_ptr(), 3 * W + pad, torch.cuda.current_stream().cuda_stream)
    out = [depth, vert, nrm] + ([rgb] if rgb is not None else [])
    out = [t.cpu().numpy() for t in out]
    if pad:
        assert (out[0][:, W:] == -5).all() and (out[1][:, 3 * W:] == -5).all() and (out[2][:, 3 * W:] == -5).all()
        if rgb is not None:
            assert (out[3][:, 3 * W:] == 9).all()
    d = out[0][:, :W]
    v, n = out[1][:, :3 * W].reshape(H, W, 3), out[2][:, :3 * W].reshape(H, W, 3)
    c = out[3][:, :3 * W].reshape(H, W, 3) if rgb is not None else None
    return d, v, n, c


def _same(got, want):
    for g, w in zip(got, want):
        if w is None:
            assert g is None
        else:
            assert np.array_equal(g, w, equal_nan=True)


@pytest.mark.parametrize("case", ["scene", "scene_colour_pitched", "scene_min_weight", "random_odd", "random_colour",
                                  "outside", "misses"])
def test_raycast_equals_the_restatement_exactly(case):
    rng = np.random.default_rng(len(case))
    if case.startswith("scene"):
        poses, s = _scene()
        if case == "scene_colour_pitched":
            c = R.new_state(GRID["dims"], colour=True)
            c[:2] = s
            c[2:] = rng.uniform(0, 255, c[2:].shape)
            s = c
        origin, vs, trunc = GRID["origin"], GRID["vs"], TRUNC
        mw = 2.5 if case == "scene_min_weight" else 0.5
        u0, v0, w, h = WIN
        M = poses[3][:3]
        intr, md = INTR, 40.0
    else:
        dims, origin, vs, trunc = (37, 23, 41), (-0.3, 0.15, -0.45), 0.125, 0.4
        s = _used_state(rng, dims, case != "random_odd")
        s[1] = np.where(s[1] > 0, s[1] + 0.3, 0)
        mw = 0.5
        intr, u0, v0, h, w, md = (40.0, 38.5, 20.25, 16.0), 11, -3, 29, 45, 12.0
        centre = np.array([2.0, 1.3, 2.1]) if case.startswith("random") else np.array([-3.0, -2.0, -4.0])
        target = np.array([2.3, 1.5, 4.0])
        if case == "misses":
            target = 2 * centre - target                             # outside the grid, looking away from it
        M = look_at(centre, target)[:3]
    M = M.astype(F32)
    want = TR.raycast(s, origin, vs, trunc, mw, intr, u0, v0, h, w, M, 0.25, md)
    got = _raycast_raw(s, origin, vs, trunc, mw, intr, u0, v0, h, w, M, 0.25, md,
                       pad=7 if case in ("scene_colour_pitched", "random_odd") else 0)
    # the march stops at the first back face, frequent in a random tsdf: few hits there
    _same(got, want)
    hits = int((want[0] > 0).sum())
    print("raycast %s: %d of %d pixels hit" % (case, hits, h * w))
    if case == "misses":
        assert hits == 0
    else:
        assert hits > (0.3 * h * w if case.startswith("scene") else 0)


def _icp_raw(depth, weight, intr, u0, v0, md, mvert, mnorm, A0, levels, min_inliers):
    H, W = depth.shape
    d = torch.from_numpy(depth).cuda()
    wt = None if weight is None else torch.from_numpy(weight).cuda()
    model = fu.Rendered(None, torch.from_numpy(mvert).cuda(), torch.from_numpy(mnorm).cuda(), None)
    n = sum(lv[1] for lv in levels)
    ws = torch.empty(tk.workspace_bytes(H, W) // 8, dtype=torch.int64, device="cuda")
    pose = torch.empty(12, dtype=torch.float64, device="cuda")
    stats = torch.empty((n, 4), dtype=torch.float64, device="cuda")
    ok = torch.empty(1, dtype=torch.int32, device="cuda")
    tk._icp_kernel(d, wt, intr, u0, v0, md, model, np.asarray(A0, np.float64).reshape(12), levels, min_inliers, ws,
                   pose, stats, ok)
    return pose.cpu().numpy(), stats.cpu().numpy(), bool(ok.item())


@pytest.mark.parametrize("case", ["constant_velocity", "perturbed_weighted", "degenerate_levels", "kitti_window"])
def test_icp_equals_the_restatement_exactly(case):
    poses, s = _scene(16)
    rng = np.random.default_rng(3)
    u0, v0, w, h = WIN if case != "kitti_window" else (0, 0, 1242, 375)
    levels = tk.LEVELS if case != "degenerate_levels" else ((3, 2, 0.3), (1, 3, 0.05), (5, 1, 16.0))
    M = poses[2][:3].astype(F32)
    model = _raycast_raw(s, GRID["origin"], GRID["vs"], TRUNC, 0.5, INTR, u0, v0, h, w, M, 0.0, 40.0)
    depth = render(poses[3], (u0, v0, w, h))
    depth = (depth * (1 + rng.uniform(-0.01, 0.01, depth.shape))).astype(F32)
    weight = None
    guess = poses[2] @ np.linalg.solve(poses[1], poses[2])
    if case == "perturbed_weighted":
        weight = rng.uniform(-0.2, 1.2, depth.shape).astype(F32)
        weight.reshape(-1)[:5] = np.nan
        guess = _perturbed(poses[3])
    A0 = np.linalg.solve(poses[2], guess)[:3]
    mi = 100 if case != "degenerate_levels" else 6000        # above the 5,408 pixels of the stride-5 grid
    want = TR.icp(depth, weight, INTR, u0, v0, 40.0, model[1], model[2], A0, levels, mi)
    got = _icp_raw(depth, weight, INTR, u0, v0, 40.0, model[1], model[2], A0, levels, mi)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1], equal_nan=True) and got[2] == want[2]
    print("icp %s: ok %s, inliers %s, flags %s" % (case, got[2], got[1][:, 0].astype(int).tolist(),
                                                   got[1][:, 3].astype(int).tolist()))
    if case != "degenerate_levels":
        assert got[2]
    else:
        assert (got[1][:, 3] == TR.FEW_INLIERS).any() and not got[2]


def test_no_host_sync_graph_capture_and_one_sync_per_track():
    poses, s = _scene(16)
    u0, v0, w, h = WIN
    vol = fu.TSDFVolume(GRID["origin"], GRID["vs"], GRID["dims"], trunc=TRUNC, colour=False)
    vol.state.copy_(torch.from_numpy(s))
    depth = torch.from_numpy(render(poses[3])).cuda()
    win = (0, u0, h, w, v0)
    trk = tk.Tracker(vol, CALIB, (h, w), window=win, pose=poses[2])
    A0 = np.linalg.solve(poses[2], poses[2] @ np.linalg.solve(poses[1], poses[2]))[:3].reshape(12)
    pose, stats, ok = trk._views(trk._out)

    def step():
        fu._raycast_kernel(vol, trk.intrinsics, u0, v0, poses[2][:3].reshape(12).astype(F32), 0.5, 0.0, 40.0, trk.model)
        tk._icp_kernel(depth, None, trk.intrinsics, u0, v0, 40.0, trk.model, A0, trk.levels, 100, trk.workspace, pose,
                       stats, ok)

    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        rendered = vol.raycast(poses[2], CALIB, (h, w), window=win)
        step()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    eager = pose.clone()
    assert torch.equal(rendered.depth, trk.model.depth) and torch.equal(rendered.normal.isnan(), trk.model.normal.isnan())
    pose.zero_()
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(st):
        with torch.cuda.graph(g, stream=st):
            step()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(pose, eager) and int(ok.item()) == 1

    class Counting:
        def __init__(self, ev):
            self.ev, self.n = ev, 0

        def record(self, *a):
            self.ev.record(*a)

        def synchronize(self):
            self.n += 1
            self.ev.synchronize()

    trk._done = Counting(trk._done)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        r = trk.track(depth, init=poses[2] @ np.linalg.solve(poses[1], poses[2]))
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert trk._done.n == 1 and r.ok
    A = np.eye(4)
    A[:3] = eager.cpu().numpy().reshape(3, 4)
    assert np.array_equal(r.cam_to_world, poses[2] @ A)


def test_the_synthetic_sequence_equals_the_restatement(monkeypatch):
    """Fuse 2 frames at their true poses, then track and fuse 4 more on the device; the same on the restatement."""
    poses = trajectory(16)
    depths = np.stack([render(p) for p in poses])
    u0, v0, w, h = WIN
    win = (0, u0, h, w, v0)
    runs = {}
    for where in ("cuda", "cpu"):
        if where == "cpu":
            monkeypatch.setattr(fu, "_raycast_kernel", _restated_raycast)
            monkeypatch.setattr(tk, "_icp_kernel", _restated_icp)
            _patch_integrate(monkeypatch)
        vol = fu.TSDFVolume(GRID["origin"], GRID["vs"], GRID["dims"], trunc=TRUNC, colour=False, device=where)
        for b in range(2):
            vol.integrate(torch.from_numpy(depths[b])[None].to(where), CALIB, poses[b], window=win)
        trk = tk.Tracker(vol, CALIB, (h, w), window=win, pose=poses[1])
        trk._accepted = [poses[0], poses[1]]
        out = []
        for f in range(2, 6):
            r = trk.track(torch.from_numpy(depths[f]).to(where))
            out.append(r)
            vol.integrate(torch.from_numpy(depths[f])[None].to(where), CALIB, r.cam_to_world, window=win)
        runs[where] = (out, vol.state.cpu().numpy())
    for a, b in zip(runs["cuda"][0], runs["cpu"][0]):
        assert a.ok and b.ok and np.array_equal(a.cam_to_world, b.cam_to_world)
        assert np.array_equal(a.inliers, b.inliers) and np.array_equal(a.rms, b.rms, equal_nan=True)
    assert np.array_equal(runs["cuda"][1], runs["cpu"][1])


def test_track_files_on_the_forward_equals_a_serial_loop(tmp_path):
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    rng = np.random.default_rng(0)
    calib = geo.StereoCalib(100.0, 100.0, 64.0, 32.0, 0.5)
    items = []
    base = rng.integers(0, 256, (64, 140, 3), dtype=np.uint8)
    for i in range(4):
        left = np.ascontiguousarray(base[:, 2 * i:2 * i + 128])
        right = np.ascontiguousarray(base[:, 2 * i + 4:2 * i + 132])
        Image.fromarray(left).save(tmp_path / f"l{i}.png")
        Image.fromarray(right).save(tmp_path / f"r{i}.png")
        items.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png")))
    grid = dict(origin=(-20.0, -10.0, 0.0), voxel_size=0.5, dims=(80, 40, 100), trunc=1.5)
    kw = dict(levels=((2, 3, 4.0), (1, 3, 2.0)), min_inliers=50)
    vol = fu.TSDFVolume(**grid)
    traj = tk.track_files(net, items, vol, calib, crop=(64, 128), max_depth=45.0, **kw)
    ref = fu.TSDFVolume(**grid)
    trk, poses, oks = None, [], []
    for i, it in enumerate(items):
        pair = io.load_pair(*it)
        left = torch.from_numpy(pair[None, 0:3]).cuda()
        right = torch.from_numpy(pair[None, 3:6]).cuda()
        win = (0, 0, 64, 128, 0)
        with torch.no_grad():
            out = net(left, right, confidence=True)
        pc = geo.reproject(out[0], calib, window=win, max_depth=45.0)
        peak = out[2].peak[:, 0]
        rgb = torch.from_numpy(np.asarray(Image.open(it[0]).convert("RGB")).copy()).cuda()
        if i == 0:
            trk = tk.Tracker(ref, calib, (64, 128), win, max_depth=45.0, **kw)
            pose, ok = np.eye(4), True
        else:
            r = trk.track(pc.depth, weight=peak)
            pose, ok = r.cam_to_world, r.ok
        poses.append(pose)
        oks.append(ok)
        if ok:
            ref.integrate(pc.depth, calib, pose, weight=peak, rgb=rgb[None], window=win, max_depth=45.0)
    print("track_files on the forward: ok %s" % traj.ok.tolist())
    assert traj.ok.tolist() == oks and np.array_equal(traj.poses, np.stack(poses))
    assert torch.equal(vol.state, ref.state) and int((ref.weight > 0).sum()) > 100
