"""GPU: dca_reproject bit-exact against its float32 restatement (tests/_reproject_restatement.py) at odd shapes, at KITTI
size and on a strided 1536x2048 window, with and without each filter and T, at the edge cases of the definition;
reproject and a meter update with a calibration without a host sync; the argument codes; the forward followed by
reproject; reproject_files against a serial loop; dca_depth_metrics against its restatement, and evaluate_files(calib=...)
against a serial loop."""
import importlib
import math

import numpy as np
import pytest
import torch

import _reproject_restatement as R

pytestmark = pytest.mark.gpu

geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
ev = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.evaluation")

CALIB = dict(fx=721.5377, fy=721.5377, cx=609.5593, cy=172.854, baseline=0.5327)


def _calib(velo=False, doffs=0.0):
    s = R.kitti_scene()
    T = None
    if velo:
        M = s["Rv"].T @ s["R0_rect"].T
        T = np.hstack([M, (-M @ np.array([s["t2"][0], s["t2"][1], 0.0]) - s["Rv"].T @ s["tv"])[:, None]])
    return geo.StereoCalib(doffs=doffs, rect_to_velo=T, **CALIB)


def _maps(B, H, W, seed):
    """Disparities over (0, 200) px with the edge cases on the first row, a peak map and LR labels."""
    rng = np.random.default_rng(seed)
    d = rng.uniform(0.05, 200, (B, H, W)).astype(np.float32)
    d.reshape(-1)[:7] = [np.nan, np.inf, -np.inf, 0.0, -1.0, -0.0, 3.0]
    peak = rng.uniform(0, 1, (B, H, W)).astype(np.float32)
    peak.reshape(-1)[-1] = np.nan
    label = rng.choice(np.array([0, 0, 0, 1, 2, 3], np.uint8), (B, H, W))
    return d, peak, label


def _check(pc, want):
    xyz, index, count, depth = want
    got_count = pc.count.cpu().numpy()
    assert np.array_equal(got_count, count)
    assert np.array_equal(pc.depth.cpu().numpy(), depth)
    for b in range(len(count)):
        n = int(count[b])
        assert np.array_equal(pc.index[b, :n].cpu().numpy(), index[b])
        assert np.array_equal(pc.xyz[b, :n].cpu().numpy(), xyz[b], equal_nan=True)


@pytest.mark.parametrize("B,H,W", [(1, 7, 5), (2, 13, 97), (1, 384, 1248)])
@pytest.mark.parametrize("filters", [False, True])
@pytest.mark.parametrize("velo", [False, True])
def test_kernel_equals_the_restatement_exactly(B, H, W, filters, velo):
    d, peak, label = _maps(B, H, W, seed=H * W + filters)
    c = _calib(velo, doffs=0.0 if velo else 1.5)
    _, _, Z = R.keep_and_points(d, None, None, 0, 0, c.Q(), None, 0, -np.inf, np.inf)
    fin = np.sort(Z[np.isfinite(Z) & (Z > 0)])
    lo, hi = fin[len(fin) // 8], fin[-len(fin) // 8 - 1]           # Z exactly at both bounds on some pixel
    kw = dict(min_peak=0.25 if filters else 0.0, min_depth=lo, max_depth=hi)
    want = R.reproject(d, peak if filters else None, label if filters else None, 0, 0, c.Q(), c.rect_to_velo if velo
                       else None, **kw)
    if not filters:                                                # the bounds are inclusive
        assert (want[3][Z == lo] == lo).all() and (want[3][Z == hi] == hi).all()
    td = torch.from_numpy(d).cuda()
    pc = geo.reproject(td[:, None], c, confidence=torch.from_numpy(peak).cuda() if filters else None,
                       min_confidence=0.25, label=torch.from_numpy(label).cuda() if filters else None,
                       frame="velodyne" if velo else "camera", min_depth=float(lo), max_depth=float(hi))
    _check(pc, want)
    pc2 = geo.reproject(td, c, confidence=torch.from_numpy(peak).cuda() if filters else None, min_confidence=0.25,
                        label=torch.from_numpy(label).cuda() if filters else None,
                        frame="velodyne" if velo else "camera", min_depth=float(lo), max_depth=float(hi))
    assert torch.equal(pc.count, pc2.count) and torch.equal(pc.depth, pc2.depth)         # two calls, same outputs
    for b in range(B):
        n = int(pc.count[b])
        assert torch.equal(pc.xyz[b, :n], pc2.xyz[b, :n]) and torch.equal(pc.index[b, :n], pc2.index[b, :n])
    print("reproject %s filters=%d velo=%d: kept %s of %d" % ((B, H, W), filters, velo, want[2].tolist(), H * W))


def test_bounds_are_inclusive_and_all_or_none_kept():
    c = _calib(doffs=0.0)
    d = np.full((2, 33, 65), 40.0, np.float32)
    d[1] = np.nan
    d[0, 5, 7] = 80.0
    _, _, Z = R.keep_and_points(d, None, None, 0, 0, c.Q(), None, 0, 0, np.inf)
    lo, hi = float(Z[0, 5, 7]), float(Z[0, 0, 0])
    pc = geo.reproject(torch.from_numpy(d).cuda(), c, min_depth=lo, max_depth=hi)
    assert pc.count.tolist() == [33 * 65, 0]                          # all kept (two exactly on a bound), none kept
    _check(pc, R.reproject(d, Q=c.Q(), min_depth=lo, max_depth=hi))
    pc = geo.reproject(torch.from_numpy(d).cuda(), c, min_depth=np.nextafter(np.float32(lo), np.float32(1e9)),
                       max_depth=np.nextafter(np.float32(hi), np.float32(0)))
    assert pc.count.tolist() == [0, 0] and not bool(pc.depth.any())


def test_strided_window_with_an_origin():
    """A 1536x2048 window at (y0, x0) = (37, 101) of a [2, 1, 1700, 2300] map (pitch != W), image origin v = 200."""
    B, Hn, Wn = 2, 1700, 2300
    d, peak, label = _maps(B, Hn, Wn, seed=7)
    c = _calib(velo=True, doffs=0.0)
    win = (37, 101, 1536, 2048, 200)
    y0, x0, h, w, vo = win
    for filters in (False, True):
        cut = lambda a: np.ascontiguousarray(a[:, y0:y0 + h, x0:x0 + w])
        want = R.reproject(cut(d), cut(peak) if filters else None, cut(label) if filters else None, x0, vo, c.Q(),
                           c.rect_to_velo, 0.5 if filters else 0.0, 1.0, 100.0)
        pc = geo.reproject(torch.from_numpy(d).cuda()[:, None], c, frame="velodyne", window=win, min_depth=1.0,
                           max_depth=100.0, confidence=torch.from_numpy(peak).cuda()[:, None] if filters else None,
                           min_confidence=0.5, label=torch.from_numpy(label).cuda()[:, None] if filters else None)
        _check(pc, want)
        assert pc.depth.shape == (B, h, w) and 0 < int(pc.count.min()) < h * w


def test_reproject_and_a_meter_update_with_a_calibration_do_not_synchronise():
    c = _calib()
    d, peak, label = (torch.from_numpy(a).cuda() for a in _maps(1, 64, 128, seed=3))
    gt = (torch.rand(1, 64, 128, generator=torch.Generator().manual_seed(0)) * 100).cuda()
    meter = ev.DisparityMeter(192, capacity=1)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            pc = geo.reproject(d, c, confidence=peak, min_confidence=0.3, label=label, window=(2, 3, 60, 120, 5),
                               min_depth=1.0, max_depth=80.0)
            meter.update(d, gt, calib=c)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert int(pc.count[0]) > 0 and meter.depth_rows().shape == (3, ev.DEPTH_COUNT)


def test_kernel_argument_codes():
    from dcanet_b200 import _lib
    lib = _lib.load()
    s = torch.cuda.current_stream().cuda_stream
    H, W = 3, 5
    d = torch.full((1, H, W), 10.0, device="cuda")
    xyz, idx = torch.empty(1, H * W, 3, device="cuda"), torch.empty(1, H * W, dtype=torch.int32, device="cuda")
    cnt, ws = torch.empty(1, dtype=torch.int64, device="cuda"), torch.empty(1, 1, dtype=torch.int32, device="cuda")
    dep = torch.empty(1, H, W, device="cuda")
    q = _calib().Q()
    a = [d.data_ptr(), None, None, W, H * W, 1, H, W, 0, 0, q.ctypes.data, None, 0.0, 0.0, math.inf, dep.data_ptr(),
         xyz.data_ptr(), idx.data_ptr(), cnt.data_ptr(), ws.data_ptr(), s]
    assert lib.dca_reproject(*a) == 0
    torch.cuda.synchronize()
    assert int(cnt[0]) == H * W and idx[0].tolist() == list(range(H * W))
    for i, v in ((0, None), (10, None), (16, None), (19, None), (3, W - 1), (4, H * W - 1), (5, 0), (6, 0),
                 (12, float("nan")), (14, -1.0)):
        b = list(a)
        b[i] = v
        assert lib.dca_reproject(*b) == -1, i


# ---- the forward, then reproject -------------------------------------------------------------------------------
def _images(B, H, W, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    left = torch.randn(B, 3, H, W, device="cuda", generator=g)
    return left, torch.roll(left, -4, 3) + 0.1 * torch.randn(B, 3, H, W, device="cuda", generator=g)


def test_forward_then_reproject_equals_the_restatement_of_the_outputs():
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    left, right = _images(1, 64, 128, seed=0)
    c = geo.StereoCalib(100.0, 100.0, 64.0, 32.0, 0.5)
    with torch.no_grad():
        pred, pv, conf, lr = net(left, right, confidence=True, lr_check=True)
    pc = geo.reproject(pred, c, confidence=conf.peak, min_confidence=0.1, label=lr.label, min_depth=0.5,
                       max_depth=200.0)
    want = R.reproject(pred[:, 0].cpu().numpy(), conf.peak[:, 0].cpu().numpy(), lr.label[:, 0].cpu().numpy(), 0, 0,
                       c.Q(), None, 0.1, 0.5, 200.0)
    _check(pc, want)
    print("forward + reproject 64x128: %d of %d pixels kept" % (int(want[2][0]), 64 * 128))


def _pngs(tmp_path, sizes):
    from PIL import Image
    rng = np.random.default_rng(0)
    items = []
    for i, (h, w) in enumerate(sizes):
        base = rng.integers(0, 256, (h, w + 8, 3), dtype=np.uint8)
        Image.fromarray(base[:, :w]).save(tmp_path / f"l{i}.png")          # disparity 8 px
        Image.fromarray(base[:, 8:]).save(tmp_path / f"r{i}.png")
        items.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png")))
    return items


def test_reproject_files_equals_a_serial_loop(tmp_path):
    import dcanet_b200 as d
    import workloads
    from PIL import Image
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    pairs = _pngs(tmp_path, [(64, 128), (50, 100), (64, 128), (40, 90)])
    calibs = [geo.StereoCalib(100.0 + i, 100.0, 60.0, 30.0, 0.5) for i in range(len(pairs))]
    items = [(l, r, str(tmp_path / f"p{i}.ply"), str(tmp_path / f"d{i}.png")) for i, (l, r) in enumerate(pairs)]
    fitems = [(l, r, str(tmp_path / f"fp{i}.ply"), str(tmp_path / f"fd{i}.png")) for i, (l, r) in enumerate(pairs)]
    got = geo.reproject_files(net, items, calibs, crop=(64, 128), depth=2, workers=2, max_depth=500.0)
    filt = geo.reproject_files(net, fitems, calibs, crop=(64, 128), depth=2, min_confidence=0.05, lr_check=True,
                               max_depth=500.0)

    def files_hold(item, xyz, rgb, depth):
        v = np.fromfile(item[2], dtype=[("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("red", "u1"), ("green", "u1"),
                                        ("blue", "u1")], offset=open(item[2], "rb").read().index(b"end_header\n") + 11)
        assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], -1), xyz)
        assert np.array_equal(np.stack([v["red"], v["green"], v["blue"]], -1), rgb)
        assert np.array_equal(np.asarray(Image.open(item[3])), geo.save_depth_png(str(tmp_path / "x.png"), depth))

    for i, ((l, r, ply, png), c) in enumerate(zip(items, calibs)):
        rgb = np.asarray(Image.open(l))
        disp = d.kitti_io.predict_files(net, l, r, crop_height=64, crop_width=128)
        xyz, index, _, depth = R.reproject(disp[None], Q=c.Q(), max_depth=500.0)
        assert np.array_equal(got[i][0], xyz[0]) and np.array_equal(got[i][1], rgb.reshape(-1, 3)[index[0]]), i
        files_hold(items[i], xyz[0], got[i][1], depth[0])
        h, w = disp.shape
        left, right, _, _ = d.kitti_io.fit_to_crop(d.kitti_io.load_pair(l, r), 64, 128)
        with torch.no_grad():
            pred, _, conf, lr = net(left.cuda(), right.cuda(), confidence=True, lr_check=True)
        cut = lambda t: t[:, 0, 64 - h:, :w].cpu().numpy()
        fx, fi, _, fd = R.reproject(cut(pred), cut(conf.peak), cut(lr.label), Q=c.Q(), min_peak=0.05, max_depth=500.0)
        assert np.array_equal(filt[i][0], fx[0]) and np.array_equal(filt[i][1], rgb.reshape(-1, 3)[fi[0]]), i
        files_hold(fitems[i], fx[0], filt[i][1], fd[0])
        assert len(filt[i][0]) < len(got[i][0])
    print("reproject_files: points per pair %s, filtered %s" % ([len(g[0]) for g in got], [len(f[0]) for f in filt]))


# ---- depth evaluation ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,H,W", [(1, 7, 5), (2, 13, 97), (1, 384, 1248)])
def test_depth_metrics_equal_the_restatement(B, H, W):
    """Every counter equal, except DCA_DEPTH_LOG_SQ: logf (CUDA, <= 1 ulp) and numpy's float32 log may differ.  With Z in
    [1e-3, 80], |ln Z| < 8, so each log differs by <= 2 ulp(8) = 2^-20 between the two, lg = ln Zp - ln Zg by
    < 2^-18 after its own rounding (|lg| < 16), lg^2 by < 2 |lg| 2^-18 + lg^2 2^-23 + 2^-36, i.e. by
    < 8 |lg| + lg^2 / 8 + 1 units of 2^-20, plus 1 for the rounding to an integer."""
    rng = np.random.default_rng(W)
    gt = rng.uniform(-1, 220, (B, H, W)).astype(np.float32)
    gt.reshape(-1)[:4] = [0.0, np.nan, np.inf, 1e-3]
    pred = (gt * rng.uniform(0.6, 1.5, gt.shape)).astype(np.float32)
    pred.reshape(-1)[-4:] = [np.nan, np.inf, -3.0, 0.0]
    c = _calib(doffs=0.25)
    rows = torch.zeros(B, ev.DEPTH_COUNT, dtype=torch.int64, device="cuda")
    ev._depth_metrics(torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda(), rows, 192.0, c.focal_baseline,
                      c.doffs, 1e-3, 80.0)
    want, lg = R.depth_metrics(pred, gt, 192.0, c.focal_baseline, c.doffs, 1e-3, 80.0)
    got = rows.cpu().numpy()
    log_col = ev.DEPTH_LOG_SQ
    others = [k for k in range(ev.DEPTH_COUNT) if k != log_col]
    assert np.array_equal(got[:, others], want[:, others])
    lg = np.abs(lg.astype(np.float64))
    bound = (8 * lg + lg ** 2 / 8 + 2).reshape(B, -1).sum(1)
    diff = np.abs(got[:, log_col] - want[:, log_col])
    assert (diff <= bound).all(), (diff, bound)
    print("depth metrics %s: valid %s, log-sum difference %s (bound %s)" % ((B, H, W), want[:, 0].tolist(),
                                                                            diff.tolist(), bound.astype(int).tolist()))


def test_evaluate_files_with_a_calibration_equals_a_serial_loop(tmp_path):
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    pairs = _pngs(tmp_path, [(64, 128), (50, 100), (64, 128)])
    calibs = [geo.StereoCalib(400.0 + 50 * i, 400.0, 60.0, 30.0, 0.54) for i in range(len(pairs))]
    quads, ref = [], ev.DisparityMeter(48, min_depth=1e-3, max_depth=80.0)
    for i, (l, r) in enumerate(pairs):
        h, w = (64, 128) if i != 1 else (50, 100)
        gt = np.full((h, w), 8.0, np.float32)
        gt[: h // 4] = 0
        d.kitti_io.save_disparity_png(str(tmp_path / f"g{i}.png"), gt)
        quads.append((l, r, str(tmp_path / f"g{i}.png"), None))
        gt = torch.from_numpy(d.kitti_io.fit_gt_to_crop(ev.read_kitti_disparity(quads[-1][2]), 64, 128))[None].cuda()
        left, right, _, _ = d.kitti_io.fit_to_crop(d.kitti_io.load_pair(l, r), 64, 128)
        with torch.no_grad():
            pred, pv = net(left.cuda(), right.cuda())
        ref.update(pred, gt, pv, calib=calibs[i])
    summary, rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2, calib=calibs)
    plain, plain_rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2)
    assert np.array_equal(rows, ref.rows()) and np.array_equal(rows, plain_rows)
    assert summary == ref.summary() and {k: v for k, v in summary.items() if k != "depth"} == plain
    dep = summary["depth"]
    assert dep["n_valid"] == summary["n_valid"] and 0.0 <= dep["a1"] <= dep["a3"] <= 1.0
    print("evaluate_files depth: abs_rel %.4f rmse %.3f m a1 %.3f" % (dep["abs_rel"], dep["rmse"], dep["a1"]))
