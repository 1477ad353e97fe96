"""CPU: TSDF fusion (fusion.py) through its float32 restatement (tests/_tsdf_restatement.py).  The fused surface of an
analytic scene (ground plane, box, sphere) rendered from six poses against the scene itself (distance, normals, coverage,
noise averaging), the culling box against the whole grid, the frame split, KITTI odometry poses, the PLY with normals,
the entry points' argument codes, and fuse_files against a serial loop with the kernels replaced by their
restatements."""
import importlib
import math
import os

import numpy as np
import pytest
import torch
from PIL import Image

import _reproject_restatement as RP
import _tsdf_restatement as R
from test_kitti_io import _rgb
from test_reproject_host import _FakeStereoFilters, _frame, _read_ply, _restated_kernel

fu = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.fusion")
geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")

F32 = np.float32


# ---- an analytic scene -------------------------------------------------------------------------------------------
# world frame = camera axes of the first frame: X right, Y down, Z forward; the ground is Y = GROUND (below the cameras)
GROUND = 1.65
SPHERE = (np.array([1.2, 0.85, 10.0]), 0.8)
BOX = (np.array([-1.9, 0.6, 9.0]), np.array([-0.5, GROUND, 10.6]))


def scene_sdf(p):
    """Signed distance (float64) to the union of ground, sphere and box; positive in free space."""
    p = np.asarray(p, np.float64)
    ground = GROUND - p[..., 1]
    sphere = np.linalg.norm(p - SPHERE[0], axis=-1) - SPHERE[1]
    c, h = (BOX[0] + BOX[1]) / 2, (BOX[1] - BOX[0]) / 2
    q = np.abs(p - c) - h
    box = np.linalg.norm(np.maximum(q, 0), axis=-1) + np.minimum(q.max(-1), 0)
    return np.minimum(np.minimum(ground, sphere), box)


def scene_normal(p, eps=1e-5):
    g = np.stack([scene_sdf(p + eps * e) - scene_sdf(p - eps * e) for e in np.eye(3)], -1)
    return g / np.linalg.norm(g, axis=-1, keepdims=True)


def look_at(centre, target):
    """camera-to-world [4,4]: camera Z towards target, X right, Y down (world Y down)."""
    z = target - centre
    z = z / np.linalg.norm(z)
    x = np.cross(np.array([0.0, 1.0, 0.0]), z)
    x = x / np.linalg.norm(x)
    y = np.cross(z, x)
    m = np.eye(4)
    m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = x, y, z, centre
    return m


def trajectory(n=6):
    """n poses on a curved path (an arc, the camera height varying slightly), each looking at the scene centre."""
    out = []
    for a in np.linspace(-0.25, 0.25, n):
        c = np.array([7.0 * np.sin(a), 0.1 * np.cos(3 * a), 10.0 - 7.0 * np.cos(a)])
        out.append(look_at(c, np.array([0.0, 1.2, 10.0])))
    return np.stack(out)


KITTI = RP.kitti_scene()
INTR = (KITTI["fx"], KITTI["fy"], KITTI["cx"], KITTI["cy"])
WIN = (360, 100, 520, 260)                       # (u0, v0, w, h): a window of the 1242 x 375 image


def render(pose, win=WIN):
    """Analytic float64 depth (camera Z, 0 = no hit) of the window, as float32 [h, w]."""
    fx, fy, cx, cy = INTR
    u0, v0, w, h = win
    u, v = np.meshgrid(np.arange(w) + u0, np.arange(h) + v0)
    d = np.stack([(u - cx) / fx, (v - cy) / fy, np.ones_like(u, dtype=np.float64)], -1)
    R_, C = pose[:3, :3], pose[:3, 3]
    dw = d @ R_.T
    best = np.full(u.shape, np.inf)
    with np.errstate(divide="ignore", invalid="ignore"):
        t = (GROUND - C[1]) / dw[..., 1]
        best = np.where((dw[..., 1] > 0) & (t > 0), np.minimum(best, t), best)
        oc = C - SPHERE[0]
        a, b, c = (dw * dw).sum(-1), 2 * (dw @ oc), oc @ oc - SPHERE[1] ** 2
        disc = b * b - 4 * a * c
        ts = (-b - np.sqrt(np.maximum(disc, 0))) / (2 * a)
        best = np.where((disc >= 0) & (ts > 0), np.minimum(best, ts), best)
        t0, t1 = (BOX[0] - C) / dw, (BOX[1] - C) / dw
        tn, tf = np.minimum(t0, t1).max(-1), np.maximum(t0, t1).min(-1)
        best = np.where((tn <= tf) & (tn > 0), np.minimum(best, tn), best)
    return np.where(np.isfinite(best), best, 0).astype(F32)


GRID = dict(origin=(-3.0, -0.625, 5.0), vs=0.05, dims=(120, 48, 160))
MIN_WEIGHT = 2.5                # points seen by at least three of the six frames: single-view crossings behind the
                                # silhouettes of the box and the sphere (up to 3.5 voxels off at min_weight 0.5) drop out


def fuse(depths, poses, win=WIN, weight=None):
    s = R.new_state(GRID["dims"], colour=False)
    T = np.linalg.inv(poses)[:, :3].reshape(len(poses), 12).astype(F32)
    trunc = 3 * GRID["vs"]
    for b in range(len(depths)):
        R.integrate(s, GRID["origin"], GRID["vs"], depths[b:b + 1], T[b:b + 1], INTR, win[0], win[1],
                    weight=None if weight is None else weight[b:b + 1], trunc=trunc)
    return s


@pytest.fixture(scope="module")
def clean():
    poses = trajectory()
    depths = np.stack([render(p) for p in poses])
    s = fuse(depths, poses)
    return poses, depths, s, R.surface(s, GRID["origin"], GRID["vs"], MIN_WEIGHT, True, False)


# measured on this scene (MIN_WEIGHT 2.5, 9,973 points): |sdf| 0.0011 m on average; at most 0.0208 m (0.42 voxel) off the
# box's edges, 0.0313 m (0.63 voxel) at its front vertical edge, where the crossings between the inside of the box
# (negative, within trunc of its front face) and the free space seen past the edge fall beside the side face.  Normals
# off the edges: 1.6 deg at the median, 16.3 deg at the 95th percentile (grazing views of the ground)
def test_fused_surface_lies_on_the_analytic_scene(clean):
    _, _, s, (xyz, nrm, _) = clean
    vs = GRID["vs"]
    assert len(xyz) > 8000
    dist = np.abs(scene_sdf(xyz.astype(np.float64)))
    print("surface: %d points, |sdf| max %.4f m (%.3f voxel), mean %.5f m" % (len(xyz), dist.max(), dist.max() / vs,
                                                                            dist.mean()))
    c, h = (BOX[0] + BOX[1]) / 2, (BOX[1] - BOX[0]) / 2
    q = np.abs(xyz - c) - h
    edge = ((q > -3 * vs).sum(1) >= 2) & (q.max(1) < 3 * vs)    # within trunc of two faces of the box
    print("off the box's edges: %d points, |sdf| max %.4f m (%.3f voxel)" % ((~edge).sum(), dist[~edge].max(),
                                                                           dist[~edge].max() / vs))
    assert dist[~edge].max() < 0.5 * vs and dist.max() < 0.75 * vs
    ang = np.degrees(np.arccos(np.clip((nrm * scene_normal(xyz.astype(np.float64))).sum(-1), -1, 1)))
    a = ang[~edge]
    print("normals off the box's edges: median %.2f deg, 95th / 99th percentile %.2f / %.2f deg, max %.2f deg"
          % (np.median(a), np.percentile(a, 95), np.percentile(a, 99), a.max()))
    assert np.median(a) < 4 and np.percentile(a, 95) < 20
    assert (np.linalg.norm(nrm, axis=1) > 0.999).mean() > 0.99


def test_the_observed_ground_is_covered_without_holes(clean):
    """Every column of voxels on the ground in front of the objects, seen by every frame, holds a crossing: y-axis
    crossings of the ground plane, one per (i, k)."""
    _, _, _, (xyz, _, _) = clean
    o, vs = GRID["origin"], GRID["vs"]
    on = np.abs(xyz[:, 1] - GROUND) < 0.5 * vs
    ii = np.rint((xyz[on, 0] - o[0]) / vs).astype(int)
    kk = np.rint((xyz[on, 2] - o[2]) / vs).astype(int)
    cover = np.zeros((GRID["dims"][2], GRID["dims"][0]), bool)
    cover[kk, ii] = True
    xs = np.arange(GRID["dims"][0]) * vs + o[0]
    zs = np.arange(GRID["dims"][2]) * vs + o[2]
    want = (np.abs(xs)[None, :] <= 1.0) & (zs[:, None] >= 7.5) & (zs[:, None] <= 8.7)
    assert want.sum() > 800
    holes = want & ~cover
    longest = 0
    for row in list(holes) + list(holes.T):
        run = 0
        for h in row:
            run = run + 1 if h else 0
            longest = max(longest, run)
    print("ground coverage: %d of %d cells, longest hole %d voxels" % ((want & cover).sum(), want.sum(), longest))
    assert longest <= 2


# measured: one noisy frame's points 0.0355 m rms from the surface, the fused surface 0.0071 m
def test_fusion_averages_the_noise_of_single_frames(clean):
    poses, depths, _, _ = clean
    rng = np.random.default_rng(0)
    noisy = depths.copy()
    for b in range(0, len(noisy), 2):
        noisy[b] = (noisy[b] * (1 + rng.uniform(-0.02, 0.02, noisy[b].shape))).astype(F32)
    fx, fy, cx, cy = INTR
    u0, v0, w, h = WIN
    u, v = np.meshgrid(np.arange(w) + u0, np.arange(h) + v0)
    z = noisy[0].astype(np.float64)
    m = z > 0
    pc = np.stack([(u - cx) / fx * z, (v - cy) / fy * z, z], -1)[m]
    single = np.sqrt(np.mean(scene_sdf(pc @ poses[0][:3, :3].T + poses[0][:3, 3]) ** 2))
    s = fuse(noisy, poses)
    xyz, _, _ = R.surface(s, GRID["origin"], GRID["vs"], MIN_WEIGHT, False, False)
    fused = np.sqrt(np.mean(scene_sdf(xyz.astype(np.float64)) ** 2))
    print("noise +-2%% on frames 0, 2, 4: single-frame rms %.4f m, fused rms %.4f m" % (single, fused))
    assert fused < 0.5 * single


# ---- culling, frame split ----------------------------------------------------------------------------------------
def _random_case(rng, B, H, W):
    depth = rng.uniform(0.3, 9.0, (B, H, W)).astype(F32)
    depth.reshape(-1)[: 3] = [0.0, np.nan, np.inf]
    weight = rng.uniform(-0.2, 1.2, (B, H, W)).astype(F32)
    weight.reshape(-1)[-2:] = [np.nan, 0.0]
    rgb = rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8)
    return depth, weight, rgb


def _random_pose(rng, where):
    """A camera inside the grid, outside it looking at it, or outside it looking away."""
    c = rng.uniform(0.5, 3.0, 3) if where == "inside" else rng.uniform(-6, -3, 3)
    target = np.array([1.5, 1.5, 1.5]) + rng.normal(0, 0.5, 3)
    if where == "away":
        target = 2 * c - target
    return look_at(c, target)


@pytest.mark.parametrize("max_depth", [2.5, 6.0, math.inf])
def test_the_culling_box_equals_the_whole_grid(max_depth):
    rng = np.random.default_rng(int(max_depth) if math.isfinite(max_depth) else 99)
    dims, origin, vs = (23, 19, 17), (0.0, 0.1, -0.2), 0.2
    intr, H, W, u0, v0 = (30.0, 28.0, 14.0, 9.0), 13, 17, 3, -2
    touched = culled = 0
    for where in ("inside", "outside", "away"):
        for _ in range(3):
            B = int(rng.integers(1, 4))
            poses = np.stack([_random_pose(rng, where) for _ in range(B)])
            depth, weight, rgb = _random_case(rng, B, H, W)
            T = np.linalg.inv(poses)[:, :3].reshape(B, 12).astype(F32)
            start = R.new_state(dims)
            start[:, 4:9] = rng.uniform(-1, 1, start[:, 4:9].shape)              # a used volume
            start[1] = np.abs(start[1])
            kw = dict(weight=weight, rgb=rgb, trunc=0.5, max_weight=3.0, max_depth=max_depth)
            whole = R.integrate(start.copy(), origin, vs, depth, T, intr, u0, v0, **kw)
            if math.isfinite(max_depth):
                box = fu.frustum_box(dims, origin, vs, intr, (u0, v0, H, W), poses, max_depth, 0.5)
            else:
                box = (0, 0, 0) + dims
            boxed = start.copy() if box is None else R.integrate(start.copy(), origin, vs, depth, T, intr, u0, v0,
                                                                 box=box, **kw)
            assert np.array_equal(boxed, whole), (where, box)
            touched += int((whole != start).any(0).sum())
            culled += math.prod(dims) - (0 if box is None else box[3] * box[4] * box[5])
    assert touched > 0
    if math.isfinite(max_depth):
        assert culled > 0
    print("max_depth %s: %d voxels updated, %d culled" % (max_depth, touched, culled))


def _patch_integrate(monkeypatch, calls=None):
    def kernel(vol, box, depth, weight, rgb, intr, u0, v0, T, max_depth):
        if calls is not None:
            calls.append((box, depth.shape[0]))
        R.integrate(vol.state.numpy(), vol.origin, vol.voxel_size, depth.numpy(), T, intr, u0, v0,
                    weight=None if weight is None else weight.numpy(), rgb=None if rgb is None else rgb.numpy(),
                    trunc=vol.trunc, max_weight=vol.max_weight, max_depth=max_depth, box=box)
    monkeypatch.setattr(fu, "_integrate_kernel", kernel)


def _patch_extract(monkeypatch):
    def kernel(vol, min_weight, normals, colours):
        xyz, n, c = R.surface(vol.state.numpy(), vol.origin, vol.voxel_size, min_weight, normals, colours)
        return fu.SurfacePoints(torch.from_numpy(xyz), None if n is None else torch.from_numpy(n),
                                None if c is None else torch.from_numpy(c))
    monkeypatch.setattr(fu, "_extract_kernel", kernel)


@pytest.mark.parametrize("max_depth", [None, 7.0])
def test_twenty_frames_are_two_calls_equal_to_one_pass(monkeypatch, max_depth):
    calls = []
    _patch_integrate(monkeypatch, calls)
    rng = np.random.default_rng(3)
    dims, origin, vs = (21, 18, 19), (0.0, 0.0, 0.0), 0.2
    calib = geo.StereoCalib(30.0, 28.0, 10.0, 8.0, 0.5)
    B, H, W = 20, 11, 15
    poses = np.stack([_random_pose(rng, "inside" if b % 3 else "outside") for b in range(B)])
    depth, weight, rgb = _random_case(rng, B, H, W)
    vol = fu.TSDFVolume(origin, vs, dims, trunc=0.4, device="cpu", max_weight=5.0)
    vol.integrate(torch.from_numpy(depth)[:, None], calib, poses, weight=torch.from_numpy(weight),
                  rgb=torch.from_numpy(rgb), window=(4, 2, H, W, 5), max_depth=max_depth)
    assert [c[1] for c in calls] == [16, 4]
    if max_depth is None:
        assert all(c[0] == (0, 0, 0) + dims for c in calls)
    T = np.linalg.inv(poses)[:, :3].reshape(B, 12).astype(F32)
    want = R.integrate(R.new_state(dims), origin, vs, depth, T, (30.0, 28.0, 10.0, 8.0), 2, 5, weight=weight, rgb=rgb,
                       trunc=F32(0.4), max_weight=5.0, max_depth=np.inf if max_depth is None else max_depth)
    assert np.array_equal(vol.state.numpy(), want)
    one_by_one = R.new_state(dims)
    for b in range(B):
        R.integrate(one_by_one, origin, vs, depth[b:b + 1], T[b:b + 1], (30.0, 28.0, 10.0, 8.0), 2, 5,
                    weight=weight[b:b + 1], rgb=rgb[b:b + 1], trunc=F32(0.4), max_weight=5.0,
                    max_depth=np.inf if max_depth is None else max_depth)
    assert np.array_equal(one_by_one, want) and (want[1] > 0).sum() > 100


def test_integrate_rejects_bad_arguments_on_the_host():
    vol = fu.TSDFVolume((0, 0, 0), 0.1, (4, 5, 6), device="cpu")
    assert vol.state.shape == (5, 6, 5, 4) and vol.nbytes == 5 * 120 * 4 and vol.trunc == pytest.approx(0.3)
    c = geo.StereoCalib(10.0, 10.0, 2.0, 2.0, 0.5)
    d = torch.ones(1, 4, 4)
    rgb = torch.zeros(1, 4, 4, 3, dtype=torch.uint8)
    with pytest.raises(ValueError, match="colour"):
        vol.integrate(d, c, np.eye(4))
    with pytest.raises(ValueError, match="window"):
        vol.integrate(d, c, np.eye(4), rgb=rgb, window=(0, 0, 4, 5, 0))
    with pytest.raises(ValueError, match="cam_to_world"):
        vol.integrate(d, c, np.eye(4)[None].repeat(2, 0), rgb=rgb)
    with pytest.raises(ValueError, match="rgb"):
        vol.integrate(d, c, np.eye(4), rgb=rgb[..., :2])
    with pytest.raises(ValueError, match="colour"):
        fu.TSDFVolume((0, 0, 0), 0.1, (4, 5, 6), colour=False, device="cpu").integrate(d, c, np.eye(4), rgb=rgb)
    with pytest.raises(ValueError):
        fu.TSDFVolume((0, 0, 0), 0.0, (4, 5, 6), device="cpu")
    with pytest.raises(ValueError):
        fu.TSDFVolume((0, 0, 0), 0.1, (2048, 1024, 1024), device="meta")
    with pytest.raises(_lib.DcaError):                  # no CPU path
        vol.integrate(d, c, np.eye(4), rgb=rgb)
    with pytest.raises(_lib.DcaError):
        vol.extract()


# ---- poses, PLY ----------------------------------------------------------------------------------------------------
def test_kitti_poses_with_the_calibration_give_the_colour_camera(tmp_path):
    """A world point through a camera-0 pose and P2 (the KITTI convention) lands where the returned camera-2 pose and
    K put it."""
    s = RP.kitti_scene()
    RP.write_kitti_calib(tmp_path / "calib.txt", s)
    rng = np.random.default_rng(4)
    poses0 = np.stack([look_at(rng.normal(0, 5, 3), rng.normal(0, 5, 3) + np.array([0, 0, 20.0])) for _ in range(5)])
    with open(tmp_path / "poses.txt", "w") as f:
        for p in poses0:
            f.write(" ".join("%.12e" % v for v in p[:3].ravel()) + "\n")
    raw = fu.read_kitti_poses(str(tmp_path / "poses.txt"))
    np.testing.assert_allclose(raw, poses0, rtol=0, atol=1e-11)
    cam2 = fu.read_kitti_poses(str(tmp_path / "poses.txt"), str(tmp_path / "calib.txt"))
    assert cam2.shape == (5, 4, 4) and cam2.dtype == np.float64
    for p0, p2 in zip(poses0, cam2):
        for _ in range(10):
            xw = p0 @ np.array([*rng.uniform(-5, 5, 2), rng.uniform(3, 50), 1.0])        # in front of camera 0
            q = s["P2"] @ (np.linalg.inv(p0) @ xw)
            xc = (np.linalg.inv(p2) @ xw)[:3]
            np.testing.assert_allclose([s["fx"] * xc[0] / xc[2] + s["cx"], s["fy"] * xc[1] / xc[2] + s["cy"]],
                                       q[:2] / q[2], rtol=0, atol=1e-7)
            assert xc[2] == pytest.approx(q[2], rel=1e-12)


def test_ply_with_normals_reads_back(tmp_path):
    rng = np.random.default_rng(2)
    xyz = rng.normal(0, 3, (31, 3)).astype(F32)
    nrm = rng.normal(0, 1, (31, 3)).astype(F32)
    rgb = rng.integers(0, 256, (31, 3), dtype=np.uint8)
    geo.save_ply(str(tmp_path / "n.ply"), xyz, rgb, normal=nrm)
    v, props = _read_ply(str(tmp_path / "n.ply"))
    assert [p[0] for p in props] == ["x", "y", "z", "nx", "ny", "nz", "red", "green", "blue"]
    assert np.array_equal(np.stack([v["nx"], v["ny"], v["nz"]], -1), nrm)
    assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], -1), xyz)
    assert np.array_equal(np.stack([v["red"], v["green"], v["blue"]], -1), rgb)
    geo.save_ply(str(tmp_path / "a.ply"), xyz, rgb)
    geo.save_ply(str(tmp_path / "b.ply"), xyz, rgb, normal=None)
    assert open(tmp_path / "a.ply", "rb").read() == open(tmp_path / "b.ply", "rb").read()


# ---- the C entry points without a device -------------------------------------------------------------------------
def test_entry_points_reject_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    t = np.zeros((16, 12), np.float32)
    ok = [p, 5, 4, 5, 6, 0.0, 0.0, 0.0, 0.1, 0, 0, 0, 4, 5, 6, p, 0, 8, 64, 1, 8, 8, p, 3, 24, 192,
          10.0, 10.0, 4.0, 4.0, 0, 0, t.ctypes.data, 0.3, math.inf, math.inf, None]

    def call(**kw):
        args = list(ok)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_tsdf_integrate(*args)

    nan = float("nan")
    for i in (0, 15, 32):
        assert call(**{f"a{i}": None}) == -1, i
    assert call(a1=3) == call(a2=0) == call(a3=-1) == call(a4=0) == -1
    assert call(a5=nan) == call(a8=0.0) == call(a8=nan) == -1
    assert call(a9=-1) == call(a12=0) == call(a9=1) == call(a13=6) == call(a11=1, a14=6) == -1     # box off the grid
    assert call(a19=0) == call(a19=17) == call(a20=0) == call(a21=0) == -1                     # B, H, W
    assert call(a17=7) == call(a18=63) == -1                                                   # pitches
    assert call(a22=None) == call(a1=2) == call(a23=2) == call(a24=23) == call(a25=191) == -1  # colour vs planes
    assert call(a26=nan) == call(a29=nan) == call(a33=0.0) == call(a33=nan) == call(a34=0.0) == call(a35=nan) == -1
    assert call(a2=2048, a3=1024, a4=1024, a12=2048, a13=1024, a14=1024) == -3                  # N = 2^31
    assert call(a30=1 << 24) == -3
    ws = [p, 5, 4, 5, 6, 0.5, p, p, None]

    def ccall(**kw):
        args = list(ws)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_tsdf_count_surface(*args)

    assert ccall(a0=None) == ccall(a6=None) == ccall(a7=None) == ccall(a1=4) == ccall(a4=0) == ccall(a5=nan) == -1
    assert ccall(a2=2048, a3=1024, a4=1024) == -3
    ex = [p, 5, 4, 5, 6, 0.0, 0.0, 0.0, 0.1, 0.5, p, 10, p, p, p, None]

    def ecall(**kw):
        args = list(ex)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_tsdf_extract_surface(*args)

    assert ecall(a0=None) == ecall(a10=None) == ecall(a12=None) == ecall(a11=-1) == ecall(a1=2) == -1
    assert ecall(a8=-0.1) == ecall(a9=nan) == ecall(a6=nan) == ecall(a3=0) == -1
    assert ecall(a2=2048, a3=1024, a4=1024) == -3


# ---- files in, one volume out, with the kernels replaced by their restatements ------------------------------------
@pytest.mark.parametrize("filters", [False, True])
def test_fuse_files_equals_a_serial_loop(tmp_path, monkeypatch, filters):
    monkeypatch.setattr(geo, "_reproject_kernel", _restated_kernel)
    _patch_integrate(monkeypatch)
    _patch_extract(monkeypatch)
    sizes = [(37, 53), (48, 64), (60, 70), (20, 64), (37, 53)]
    model = _FakeStereoFilters().eval()
    calib = geo.StereoCalib(50.0, 52.0, 30.0, 20.0, 0.5)
    rng = np.random.default_rng(6)
    poses = np.stack([look_at(rng.normal(0, 0.3, 3), np.array([0.0, 0.0, 10.0]) + rng.normal(0, 0.5, 3))
                      for _ in sizes])
    kw = dict(min_confidence=0.4, lr_check=True) if filters else {}
    grid = dict(origin=(-1.5, -1.0, 0.2), voxel_size=0.1, dims=(30, 20, 40), trunc=0.3, device="cpu")
    items = []
    ref = fu.TSDFVolume(**grid)
    for i, (h, w) in enumerate(sizes):
        rgb = _rgb(10 + i, h, w)
        Image.fromarray(rgb).save(tmp_path / f"l{i}.png")
        Image.fromarray(_rgb(50 + i, h, w)).save(tmp_path / f"r{i}.png")
        items.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png")))
        left, right, (y0, x0, hh, ww, vo) = _frame(io.load_pair(*items[-1]), "fit", 48, 64)
        with torch.no_grad():
            out = model(left, right, confidence=True, lr_check=filters)
        pc = geo.reproject(out[0], calib, confidence=out[2].peak if filters else None, min_confidence=0.4,
                           label=out[3].label if filters else None, window=(y0, x0, hh, ww, vo), max_depth=4.0)
        ref.integrate(pc.depth, calib, poses[i], weight=out[2].peak[:, 0, y0:y0 + hh, x0:x0 + ww],
                      rgb=torch.from_numpy(np.ascontiguousarray(rgb[vo:vo + hh, x0:x0 + ww])),
                      window=(y0, x0, hh, ww, vo), max_depth=4.0)
    vol = fu.TSDFVolume(**grid)
    got = fu.fuse_files(model, items, poses, vol, calib, crop=(48, 64), max_depth=4.0, depth=2, workers=3,
                        ply=str(tmp_path / "s.ply"), min_weight=0.1, **kw)
    assert got is vol and np.array_equal(vol.state.numpy(), ref.state.numpy())
    assert (ref.weight > 0).sum() > 500
    xyz, nrm, col = ref.extract(0.1).numpy()
    v, props = _read_ply(str(tmp_path / "s.ply"))
    assert len(xyz) > 0 and [p[0] for p in props] == ["x", "y", "z", "nx", "ny", "nz", "red", "green", "blue"]
    assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], -1), xyz)
    assert np.array_equal(np.stack([v["nx"], v["ny"], v["nz"]], -1), nrm)
    assert np.array_equal(np.stack([v["red"], v["green"], v["blue"]], -1), col)
    unit = fu.fuse_files(model, items[:2], poses[:2], fu.TSDFVolume(**grid), calib, crop=(48, 64), max_depth=4.0,
                         weight=None, **kw)
    first = fu.fuse_files(model, items[:2], poses[:2], fu.TSDFVolume(**grid), calib, crop=(48, 64), max_depth=4.0,
                          **kw)
    assert not np.array_equal(unit.weight.numpy(), first.weight.numpy())


def test_an_infinite_or_overflowing_max_depth_fuses_the_whole_grid(monkeypatch):
    """max_depth = inf (reproject's own "no limit") behaves as None, and a finite max_depth whose window corners
    overflow float64 falls back to the whole grid instead of a cast of NaN / inf to a voxel index."""
    dims, origin, vs = (21, 18, 19), (0.0, 0.0, 0.0), 0.2
    intr = (30.0, 28.0, 10.0, 8.0)
    pose = look_at(np.array([-1.0, 1.5, -2.0]), np.array([2.0, 1.8, 2.0]))[None]
    for md in (math.inf, 1e308, 1e300):
        assert fu.frustum_box(dims, origin, vs, intr, (2, 5, 11, 15), pose, md, 0.4) == (0, 0, 0) + dims, md
    calls = []
    _patch_integrate(monkeypatch, calls)
    rng = np.random.default_rng(8)
    calib = geo.StereoCalib(*intr, 0.5)
    depth, weight, rgb = (torch.from_numpy(a) for a in _random_case(rng, 3, 11, 15))
    poses = np.stack([_random_pose(rng, "inside") for _ in range(3)])
    vols = {}
    for md in (None, math.inf):
        vols[md] = fu.TSDFVolume(origin, vs, dims, trunc=0.4, device="cpu")
        vols[md].integrate(depth, calib, poses, weight=weight, rgb=rgb, window=(4, 2, 11, 15, 5), max_depth=md)
    assert [c[0] for c in calls] == [(0, 0, 0) + dims] * 2
    assert torch.equal(vols[None].state, vols[math.inf].state) and int((vols[None].weight > 0).sum()) > 100
    with pytest.raises(ValueError, match="max_depth"):
        vols[None].integrate(depth, calib, poses, weight=weight, rgb=rgb, max_depth=float("nan"))


def test_integrate_refuses_a_depth_map_on_another_device():
    vol = fu.TSDFVolume((0, 0, 0), 0.1, (4, 5, 6), colour=False, device="meta")
    with pytest.raises(ValueError, match="device|meta|cpu"):
        vol.integrate(torch.ones(1, 4, 4), geo.StereoCalib(10.0, 10.0, 2.0, 2.0, 0.5), np.eye(4))


def test_fuse_pipeline_allocates_no_point_cloud_read_back():
    model = _FakeStereoFilters().eval()
    vol = fu.TSDFVolume((0, 0, 0), 0.1, (4, 5, 6), device="cpu")
    pipe = fu.FusePipeline(model, geo.StereoCalib(50.0, 52.0, 30.0, 20.0, 0.5), vol, crop_height=48, crop_width=64)
    assert all(o is None for o in pipe.slot_out) and not hasattr(pipe, "rgb_out")
