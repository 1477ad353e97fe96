"""GPU: the moving-object kernels (csrc/motion.cu) bit-exact against their restatement (tests/_motion_restatement.py)
at KITTI size, for one image and for four with a different transform each, pitched depth maps, holes and every radius;
CUDA-graph capture; and fuse_files / track_files with motion= on the real forward against a serial loop."""
import importlib

import numpy as np
import pytest
import torch
from PIL import Image

import _motion_restatement as R
from test_motion_host import CALIB, INTR, _moving_box, pose, render

pytestmark = pytest.mark.gpu

mo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.motion")
fu = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.fusion")
tk = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.tracking")
geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")

F32 = np.float32


def _case(B, seed):
    """B (prev, cur, cur_to_prev float64) at 375 x 1242: moving boxes, depth noise, holes (0 and NaN) and a transform
    per image perturbed around 1 m forward."""
    rng = np.random.default_rng(seed)
    prevs, curs, As = [], [], []
    for b in range(B):
        start = np.array([rng.uniform(-3, 3), 0.0, rng.uniform(7, 14)])
        step = np.array([rng.uniform(-1.5, 1.5), 0.0, rng.uniform(-2.5, 2.5)])
        prev, cur, _ = _moving_box(start, step)
        for z in (prev, cur):
            z *= (1 + rng.normal(0, 0.003, z.shape)).astype(F32)
            z[rng.random(z.shape) < 0.02] = 0
            z[rng.random(z.shape) < 0.01] = np.nan
        p1 = pose(1)
        p1[:3, 3] += rng.normal(0, 0.01, 3)
        prevs.append(prev)
        curs.append(cur)
        As.append(np.linalg.solve(pose(0), p1))
    return np.stack(prevs), np.stack(curs), np.stack(As)


def _check(m, cur, prev, A, u0, v0, **kw):
    lk = {k: kw[k] for k in ("tau", "tau_rel", "radius") if k in kw}
    ck = {k: kw[k] for k in ("gate", "min_pixels") if k in kw}
    fB = CALIB.focal_baseline
    Af = A[:, :3].reshape(len(A), 12).astype(F32)
    lab, res = R.labels(cur, prev, INTR, fB, CALIB.doffs, u0, v0, Af, **lk)
    want = R.components(cur, lab, res, INTR, fB, CALIB.doffs, u0, v0, **ck)
    assert np.array_equal(m.label.cpu().numpy(), lab)
    assert np.array_equal(m.residual.cpu().numpy(), res, equal_nan=True)
    assert np.array_equal(m.instance.cpu().numpy(), want["instance"])
    o = m.objects
    assert np.array_equal(o.count.cpu().numpy(), want["count"]) and np.array_equal(o.dropped.cpu().numpy(),
                                                                                  want["dropped"])
    assert np.array_equal(o.ints.cpu().numpy(), want["ints"])
    assert np.array_equal(o.extent.cpu().numpy(), want["extent"], equal_nan=True)
    assert np.array_equal(o.res_sum.cpu().numpy(), want["res_sum"])
    return lab, want


@pytest.mark.parametrize("B,radius,seed", [(1, 1, 0), (4, 1, 1), (4, 0, 2), (4, 2, 3), (2, 4, 4)])
def test_kernels_equal_the_restatement_at_kitti_size(B, radius, seed):
    prev, cur, A = _case(B, seed)
    kw = dict(radius=radius, min_pixels=50 if seed % 2 else 100, gate=1.0 if seed != 3 else 0.5)
    m = mo.motion(torch.from_numpy(cur).cuda(), torch.from_numpy(prev).cuda(), CALIB, A, **kw)
    lab, want = _check(m, cur, prev, A, 0, 0, **kw)
    moving = (lab == R.APPEARED) | (lab == R.BEHIND)
    print("B=%d r=%d: %d moving pixels, objects %s" % (B, radius, moving.sum(), want["count"].tolist()))
    assert want["count"].sum() >= B and (lab == R.STATIC).sum() > lab.size // 2


def test_a_pitched_window_and_many_small_objects():
    """A window of a larger map (pitched, u0 / v0 offsets), and more components than the table holds: min_pixels = 1 on
    noisy depth, so `dropped` counts the rest."""
    prev, cur, A = _case(3, 7)
    big_p = np.zeros((3, 400, 1300), F32)
    big_c = np.zeros((3, 400, 1300), F32)
    big_p[:, 10:385, 20:1262] = prev
    big_c[:, 10:385, 20:1262] = cur
    rng = np.random.default_rng(8)
    cur2 = cur * (1 + rng.normal(0, 0.05, cur.shape)).astype(F32)
    big_c[:, 10:385, 20:1262] = cur2
    dp, dc = torch.from_numpy(big_p).cuda(), torch.from_numpy(big_c).cuda()
    win = (0, 0, 375, 1242, 0)
    m = mo.motion(dc[:, 10:385, 20:1262], dp[:, 10:385, 20:1262], CALIB, A, window=win, min_pixels=1, radius=0)
    _, want = _check(m, cur2, prev, A, 0, 0, min_pixels=1, radius=0)
    assert (want["dropped"] > 0).all()
    u = (5, 100, 80, 200, 30)
    m = mo.motion(dc[:, 10:90, 100:300], dp[:, 10:90, 100:300], CALIB, A, window=u)
    _check(m, cur2[:, :80, 80:280], prev[:, :80, 80:280], A, 100, 30)


def test_graph_capture_equals_eager():
    prev, cur, A = _case(4, 9)
    dp, dc = torch.from_numpy(prev).cuda(), torch.from_numpy(cur).cuda()
    eager = mo.motion(dc, dp, CALIB, A)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        mo.motion(dc, dp, CALIB, A)                               # warm-up on the side stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        got = mo.motion(dc, dp, CALIB, A)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager[:3], got[:3]):
        assert torch.equal(a.nan_to_num(), b.nan_to_num()) if a.is_floating_point() else torch.equal(a, b)
    for a, b in zip(eager.objects, got.objects):
        assert torch.equal(a.nan_to_num(), b.nan_to_num()) if a.is_floating_point() else torch.equal(a, b)
    assert int(eager.objects.count.sum()) >= 4


def _pairs(tmp_path):
    rng = np.random.default_rng(0)
    items = []
    base = rng.integers(0, 256, (64, 150, 3), dtype=np.uint8)
    for i in range(4):
        left = np.ascontiguousarray(base[:, 2 * i:2 * i + 128])
        right = np.ascontiguousarray(base[:, 2 * i + 4:2 * i + 132])
        left[20:40, 30 + 6 * i:60 + 6 * i] = 255 - 40 * i                 # a patch that moves between the pairs
        Image.fromarray(left).save(tmp_path / f"l{i}.png")
        Image.fromarray(right).save(tmp_path / f"r{i}.png")
        items.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png")))
    return items


def _serial(net, items, calib, poses, ref, motion_kw, track_kw=None):
    """The serial loop: forward, reproject, (tracking,) motion against the last frame integrated, masked integration."""
    last, trk, out_poses, oks, masked = None, None, [], [], 0
    win = (0, 0, 64, 128, 0)
    for i, it in enumerate(items):
        pair = io.load_pair(*it)
        left = torch.from_numpy(pair[None, 0:3]).cuda()
        right = torch.from_numpy(pair[None, 3:6]).cuda()
        with torch.no_grad():
            out = net(left, right, confidence=True)
        pc = geo.reproject(out[0], calib, window=win, max_depth=45.0)
        peak = out[2].peak[:, 0]
        rgb = torch.from_numpy(np.asarray(Image.open(it[0]).convert("RGB")).copy()).cuda()
        pose, ok = poses[i] if poses is not None else np.eye(4), True
        if track_kw is not None:
            if i == 0:
                trk = tk.Tracker(ref, calib, (64, 128), win, max_depth=45.0, **track_kw)
            else:
                r = trk.track(pc.depth, weight=peak)
                pose, ok = r.cam_to_world, r.ok
        out_poses.append(pose)
        oks.append(ok)
        if not ok:
            continue
        w = peak
        if last is not None:
            m = mo.motion(pc.depth, last[0], calib, np.linalg.solve(last[1], pose), window=win, **motion_kw)
            w = torch.where(m.instance == 0, peak, torch.zeros((), device=peak.device))
            masked += int((m.instance > 0).sum())
        ref.integrate(pc.depth, calib, pose, weight=w, rgb=rgb[None], window=win, max_depth=45.0)
        last = (pc.depth, pose)
    return out_poses, oks, masked


def test_fuse_and_track_files_with_motion_equal_a_serial_loop(tmp_path):
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    calib = geo.StereoCalib(100.0, 100.0, 64.0, 32.0, 0.5)
    items = _pairs(tmp_path)
    grid = dict(origin=(-20.0, -10.0, 0.0), voxel_size=0.5, dims=(80, 40, 100), trunc=1.5)
    motion_kw = dict(min_pixels=5, tau=1.0)
    poses = np.stack([np.eye(4)] * 4)
    for i in range(4):
        poses[i, 0, 3] = 0.05 * i
    vol = fu.TSDFVolume(**grid)
    fu.fuse_files(net, items, poses, vol, calib, crop=(64, 128), max_depth=45.0, motion=motion_kw)
    ref = fu.TSDFVolume(**grid)
    _, _, masked = _serial(net, items, calib, poses, ref, motion_kw)
    print("fuse_files(motion=): %d pixels masked" % masked)
    assert torch.equal(vol.state, ref.state) and int((ref.weight > 0).sum()) > 100
    plain = fu.fuse_files(net, items, poses, fu.TSDFVolume(**grid), calib, crop=(64, 128), max_depth=45.0)
    assert masked == 0 or not torch.equal(plain.state, vol.state)
    kw = dict(levels=((2, 3, 4.0), (1, 3, 2.0)), min_inliers=50)
    vol = fu.TSDFVolume(**grid)
    traj = tk.track_files(net, items, vol, calib, crop=(64, 128), max_depth=45.0, motion=motion_kw, **kw)
    ref = fu.TSDFVolume(**grid)
    poses_s, oks, masked = _serial(net, items, calib, None, ref, motion_kw, kw)
    print("track_files(motion=): ok %s, %d pixels masked" % (traj.ok.tolist(), masked))
    assert traj.ok.tolist() == oks and np.array_equal(traj.poses, np.stack(poses_s))
    assert torch.equal(vol.state, ref.state)
