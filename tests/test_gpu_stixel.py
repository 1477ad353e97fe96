"""GPU: ground_profile, stixels and render (include/dca_b200.h section 15) equal the numpy restatement bit for bit, from
single pixels to B = 8 KITTI windows, pitched maps with a window, with and without confidence and labels, NaN / +-inf /
negative disparities, empty columns, a zero profile and the row limit; no host sync after the first call, CUDA-graph
replay, the real forward's output, evaluate_files(stixels=) against a serial loop, and the entry points' error codes."""
import numpy as np
import pytest
import torch

import _stixel_restatement as R

pytestmark = pytest.mark.gpu


def _dev():
    import dcanet_b200 as d
    return d


def _random_maps(B, H, W, seed):
    rng = np.random.default_rng(seed)
    disp = rng.uniform(0, 60, (B, H, W)).astype(np.float32)
    disp[rng.random((B, H, W)) < 0.1] = np.nan
    disp[rng.random((B, H, W)) < 0.03] = np.inf
    disp[rng.random((B, H, W)) < 0.03] = -np.inf
    disp[rng.random((B, H, W)) < 0.05] = -2.0
    if W > 3:
        disp[:, :, 1:3] = np.nan                     # an empty column at width 1 or 2
    peak = rng.random((B, H, W)).astype(np.float32)
    label = rng.integers(0, 4, (B, H, W)).astype(np.uint8)
    label[rng.random((B, H, W)) < 0.6] = 0
    return disp, peak, label


def _scene(B, seed):
    return np.stack([R.driving_scene(seed + b)[0] for b in range(B)])


def _embed(a, pad, fill):
    """a [B,h,w] -> a map [B,h+2p,w+3p] holding a at (p, 2p), as a device tensor, and its window."""
    B, h, w = a.shape
    big = np.full((B, h + 2 * pad, w + 3 * pad), fill, a.dtype)
    big[:, pad:pad + h, 2 * pad:2 * pad + w] = a
    return torch.from_numpy(big).cuda(), (pad, 2 * pad, h, w, 7)


def _check(disp, peak, label, profile, width, min_peak=0.3, pitched=False, max_disp=192, **priors):
    d = _dev()
    B, H, W = disp.shape
    if pitched:
        cd, window = _embed(disp, 3, np.float32(5))
        cp = _embed(peak, 3, np.float32(1))[0] if peak is not None else None
        cl = _embed(label, 3, np.uint8(0))[0] if label is not None else None
    else:
        cd, window = torch.from_numpy(disp).cuda(), None
        cp = torch.from_numpy(peak).cuda() if peak is not None else None
        cl = torch.from_numpy(label).cuda() if label is not None else None
    kw = dict(confidence=cp, min_confidence=min_peak, label=cl, max_disp=max_disp, window=window)
    gp = d.ground_profile(cd, min_inliers=50, **kw)
    wp, wl, wi, wo = R.ground_profile(disp, peak, label, min_peak if peak is not None else 0.0, max_disp, 50)
    assert np.array_equal(gp.disp.cpu().numpy(), wp)
    assert np.array_equal(gp.line.cpu().numpy(), wl)
    assert np.array_equal(gp.inliers.cpu().numpy(), wi) and np.array_equal(gp.ok.cpu().numpy(), wo)
    prof = gp.disp if profile is None else torch.from_numpy(profile).cuda()
    pnp = prof.cpu().numpy()
    st = d.stixels(cd, prof, width=width, **kw, **priors)
    q = lambda v: int(np.rint(256 * v))
    rs_pr = dict(R.DEFAULTS)
    for k, v in priors.items():
        rs_pr[{"sigma_ground": "s_ground", "sigma_object": "s_object", "sigma_sky": "s_sky"}.get(k, k)] = \
            q(v) if k.startswith(("sigma", "eps")) else v
    want = R.stixels(disp, pnp, peak, label, min_peak if peak is not None else 0.0, width, max_disp, **rs_pr)
    count = st.count.cpu().numpy()
    assert np.array_equal(count, want["count"])
    assert np.array_equal(st.free_space.cpu().numpy(), want["free_space"])
    valid = np.arange(H)[None, None] < count[..., None]
    for got, key in ((st.bottom, "bottom"), (st.top, "top"), (st.cls, "cls"), (st.disp, "disp")):
        g = got.cpu().numpy()
        assert np.array_equal(g[valid], want[key][valid].astype(g.dtype)), key
    out, cls = st.render(prof)
    wd, wc = R.render(want, pnp, W, width)
    assert np.array_equal(out.cpu().numpy(), wd) and np.array_equal(cls.cpu().numpy(), wc)
    return gp, st, want


@pytest.mark.parametrize("B,H,W", [(1, 1, 1), (1, 1, 37), (1, 29, 1), (1, 7, 5), (2, 64, 65)])
@pytest.mark.parametrize("width", [1, 5, 7, 16])
@pytest.mark.parametrize("filters,pitched", [(False, False), (True, True)])
def test_small_shapes_equal_the_restatement(B, H, W, width, filters, pitched):
    disp, peak, label = _random_maps(B, H, W, seed=B * 1000 + H * 10 + W)
    rng = np.random.default_rng(width)
    profile = np.where(rng.random((B, H)) < 0.6, rng.uniform(0, 70, (B, H)), 0).astype(np.float32)
    profile[:, ::5] = np.nan
    _check(disp, peak if filters else None, label if filters else None, profile, width, pitched=pitched)


def test_zero_profile_and_the_ground_profile_of_small_maps():
    disp, peak, label = _random_maps(2, 64, 65, seed=3)
    gp, st, _ = _check(disp, None, None, np.zeros((2, 64), np.float32), 5)
    assert (st.cls.cpu().numpy()[np.arange(64)[None, None] < st.count.cpu().numpy()[..., None]] != 0).all()
    _check(disp, peak, label, None, 7, pitched=True, p_gravity=3000, p_order=0, eps_order=0.5, sigma_sky=0.5, tau=2)


@pytest.mark.parametrize("B,width,filters,pitched", [(1, 5, False, False), (1, 16, True, True), (8, 5, False, True)])
def test_kitti_windows_equal_the_restatement(B, width, filters, pitched):
    disp = _scene(B, seed=10)
    _, peak, label = _random_maps(B, 375, 1242, seed=5)
    gp, st, want = _check(disp, peak if filters else None, label if filters else None, None, width, min_peak=0.05,
                          pitched=pitched)
    assert gp.ok.all()
    print("KITTI B=%d width=%d: %.2f segments per column" % (B, width, float(st.count.float().mean())))


def test_row_limit():
    d = _dev()
    rng = np.random.default_rng(1)
    disp = rng.uniform(0, 30, (1, d.stixel.MAX_ROWS, 3)).astype(np.float32)
    prof = np.linspace(40, 0, d.stixel.MAX_ROWS, dtype=np.float32)[None]
    _check(disp, None, None, prof, 2)
    # above the limit the entry point refuses the shape
    from dcanet_b200 import _lib
    H = d.stixel.MAX_ROWS + 1
    x = torch.zeros(1, H, 3, device="cuda")
    p = torch.zeros(1, H, device="cuda")
    o = [torch.zeros(1, H, device="cuda", dtype=t) for t in (torch.int32, torch.int16, torch.int16, torch.uint8,
                                                             torch.float32, torch.int32)]
    ws = torch.empty(d.stixel.stixel_workspace_bytes(1, H, 3, 2, 16), dtype=torch.uint8, device="cuda")
    rc = _lib.load().dca_stixels(x.data_ptr(), None, None, 3, 3 * H, 1, H, 3, 0.0, p.data_ptr(), 2, 16, 256, 256, 256,
                                 3, 100, 0, 0, 0, 0, *[t.data_ptr() for t in o], ws.data_ptr(),
                                 torch.cuda.current_stream().cuda_stream)
    assert rc == -3


def test_repeatable_no_host_sync_and_graph_replay():
    d = _dev()
    disp = torch.from_numpy(_scene(2, seed=20)).cuda()
    run = lambda: (lambda g: (g, d.stixels(disp, g)))(d.ground_profile(disp))
    g0, s0 = run()
    r0 = s0.render(g0)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        again = []
        for _ in range(2):
            g, s = run()
            again.append((g, s, s.render(g)))
    finally:
        torch.cuda.set_sync_debug_mode("default")
    for g, s, r in again:
        assert torch.equal(g.disp, g0.disp) and torch.equal(g.line, g0.line)
        assert torch.equal(s.count, s0.count) and torch.equal(s.free_space, s0.free_space)
        assert torch.equal(r[0], r0[0]) and torch.equal(r[1], r0[1])
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        run()
    torch.cuda.current_stream().wait_stream(stream)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gc, sc = run()
        rc = sc.render(gc)
    new = _scene(2, seed=30)
    disp.copy_(torch.from_numpy(new))
    graph.replay()
    torch.cuda.synchronize()
    wp = R.ground_profile(new)[0]
    assert np.array_equal(gc.disp.cpu().numpy(), wp)
    want = R.stixels(new, wp)
    assert np.array_equal(sc.count.cpu().numpy(), want["count"])
    assert np.array_equal(rc[0].cpu().numpy(), R.render(want, wp, new.shape[2], 5)[0])


def _net(maxdisp):
    import dcanet_b200 as d
    import workloads
    return workloads.init_bench_weights_(d.GwcNet(maxdisp), 0).cuda().eval()


def test_forward_output_flows_through_the_stixels():
    d = _dev()
    net = _net(192)
    gen = torch.Generator(device="cuda").manual_seed(1)
    left = torch.randn(1, 3, 384, 1248, device="cuda", generator=gen)
    right = torch.roll(left, -4, 3) + 0.1 * torch.randn(1, 3, 384, 1248, device="cuda", generator=gen)
    with torch.no_grad():
        pred, pv, conf, lr = net(left, right, confidence=True, lr_check=True)
    window = (9, 0, 375, 1242, 0)
    g = d.ground_profile(lr.filled, confidence=conf.peak, min_confidence=0.1, label=lr.label, window=window)
    st = d.stixels(lr.filled, g, confidence=conf.peak, min_confidence=0.1, label=lr.label, window=window)
    assert tuple(g.disp.shape) == (1, 375) and tuple(st.bottom.shape) == (1, 249, 375)
    count = st.count.cpu().numpy()
    assert (count >= 1).all() and (count <= 375).all()
    bottom, top = st.bottom.cpu().numpy(), st.top.cpu().numpy()
    for k in range(249):
        n = count[0, k]
        assert bottom[0, k, 0] == 374 and top[0, k, n - 1] == 0
        assert (top[0, k, :n - 1] == bottom[0, k, 1:n] + 1).all()
    cut = lambda t: t[:, 0, 9:384, :1242].cpu().numpy()
    wp = R.ground_profile(cut(lr.filled), cut(conf.peak), cut(lr.label), 0.1)[0]
    assert np.array_equal(g.disp.cpu().numpy(), wp)
    want = R.stixels(cut(lr.filled), wp, cut(conf.peak), cut(lr.label), 0.1)
    assert np.array_equal(count, want["count"])
    print("forward + stixels: ok %s, %.2f segments per column" % (bool(g.ok[0]), count.mean()))


def test_metric_of_an_object_segment():
    d = _dev()
    disp = torch.from_numpy(_scene(1, seed=0)).cuda()
    calib = d.StereoCalib(**{k: v for k, v in R.KITTI.items()})
    st = d.stixels(disp, d.ground_profile(disp))
    m = st.metric(calib)
    k = 30                                            # a column of the 8 m box
    cls, count = st.cls[0, k].cpu().numpy(), int(st.count[0, k])
    i = [j for j in range(count) if cls[j] == 1][0]
    z = float(m.z[0, k, i])
    assert abs(z - 8.0) < 0.1
    assert abs(float(m.x[0, k, i]) - (152 - R.KITTI["cx"]) * z / R.KITTI["fx"]) < 1e-3
    assert float(m.y_bottom[0, k, i]) > float(m.y_top[0, k, i])
    assert torch.isnan(m.z[0, k, count:]).all()


def test_kernel_argument_codes():
    from dcanet_b200 import _lib
    d = _dev()
    lib = _lib.load()
    s = torch.cuda.current_stream().cuda_stream
    B, H, W = 1, 6, 7
    x = torch.full((B, H, W), 3.0, device="cuda")
    prof = torch.zeros(B, H, device="cuda")
    line = torch.empty(B, 2, dtype=torch.float64, device="cuda")
    inl = torch.empty(B, dtype=torch.int32, device="cuda")
    ok = torch.empty(B, dtype=torch.uint8, device="cuda")
    ws = torch.empty(d.stixel.ground_workspace_bytes(B, H, 16), dtype=torch.uint8, device="cuda")
    a = [x.data_ptr(), None, None, W, H * W, B, H, W, 0.0, 16, 1, prof.data_ptr(), line.data_ptr(), inl.data_ptr(),
         ok.data_ptr(), ws.data_ptr(), s]
    assert lib.dca_ground_profile(*a) == 0
    for i, v in ((0, None), (11, None), (12, None), (13, None), (14, None), (15, None), (3, W - 1), (4, H * W - 1),
                 (5, 0), (5, 65536), (6, 0), (7, 0), (8, float("nan")), (9, 0), (9, 1025), (10, 0)):
        b = list(a)
        b[i] = v
        assert lib.dca_ground_profile(*b) == -1, i
    o = [torch.zeros(B, 2, H, device="cuda", dtype=t) for t in (torch.int32, torch.int16, torch.int16, torch.uint8,
                                                                 torch.float32, torch.int32)]
    sws = torch.empty(d.stixel.stixel_workspace_bytes(B, H, W, 4, 16), dtype=torch.uint8, device="cuda")
    a = [x.data_ptr(), None, None, W, H * W, B, H, W, 0.0, prof.data_ptr(), 4, 16, 256, 256, 256, 3, 100, 0, 0, 0, 0] \
        + [t.data_ptr() for t in o] + [sws.data_ptr(), s]
    assert lib.dca_stixels(*a) == 0
    for i, v in ((0, None), (9, None), (21, None), (26, None), (27, None), (3, W - 1), (5, 0), (8, float("nan")),
                 (10, 0), (10, 17), (11, 0), (11, 1025), (12, 0), (13, 16385), (14, -1), (15, 0), (15, 9), (16, -1),
                 (17, (1 << 20) + 1), (18, -1), (19, -1), (20, -1)):
        b = list(a)
        b[i] = v
        assert lib.dca_stixels(*b) == -1, i
    out = torch.empty(B, H, W, device="cuda")
    oc = torch.empty(B, H, W, dtype=torch.uint8, device="cuda")
    a = [o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr(), o[4].data_ptr(), prof.data_ptr(), B, H, W,
         4, 2, out.data_ptr(), oc.data_ptr(), s]
    assert lib.dca_stixel_render(*a) == 0
    for i, v in ((0, None), (5, None), (11, None), (6, 0), (9, 0), (9, 17), (10, 3)):
        b = list(a)
        b[i] = v
        assert lib.dca_stixel_render(*b) == -1, i
    b = list(a)
    b[7] = 769
    assert lib.dca_stixel_render(*b) == -3
    torch.cuda.synchronize()


# ---- evaluation -------------------------------------------------------------------------------------------------
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


@pytest.mark.parametrize("flags", [dict(), dict(confidence=True, lr_check=True)])
def test_evaluate_files_with_stixels_equals_a_serial_loop(tmp_path, flags):
    import dcanet_b200 as d
    ev = d.evaluation
    net = _net(48)
    pairs = _pngs(tmp_path, [(64, 128), (50, 100), (64, 128)])
    params = dict(width=4, p_seg=4096, min_inliers=20)
    quads, ref, segs = [], ev.DisparityMeter(48), 0
    for i, (l, r) in enumerate(pairs):
        h, w = (64, 128) if i != 1 else (50, 100)
        gt = np.full((h, w), 8.0, np.float32)
        gt[: h // 4] = 0
        d.kitti_io.save_disparity_png(str(tmp_path / f"g{i}.png"), gt)
        quads.append((l, r, str(tmp_path / f"g{i}.png"), None))
        gt = torch.from_numpy(ev.read_kitti_disparity(quads[-1][2]))[None].cuda()
        left, right, _, _ = d.kitti_io.fit_to_crop(d.kitti_io.load_pair(l, r), 64, 128)
        window = (64 - h, 0, h, w, 0)
        with torch.no_grad():
            out = net(left.cuda(), right.cuda(), **flags)
        if flags:
            pred, _, conf, lr = out
            src, kw = lr.filled, dict(confidence=conf.peak, label=lr.label)
        else:
            src, kw = out[0], {}
        g = d.ground_profile(src, window=window, max_disp=48, min_inliers=20, **kw)
        st = d.stixels(src, g, window=window, max_disp=48, width=4, p_seg=4096, **kw)
        ref.update(st.render(g)[0][:, None], gt)
        segs += int(st.count.sum())
    summary, rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2, stixels=params, **flags)
    plain, plain_rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2, **flags)
    assert summary["stixels"] == ref.summary()
    assert summary["stixels_per_image"] == segs / 3
    assert np.array_equal(rows, plain_rows)
    assert {k: v for k, v in summary.items() if k not in ("stixels", "stixels_per_image")} == plain
    assert "stixels" not in plain
    with pytest.raises(ValueError):
        d.evaluate_files(net, quads, crop=(64, 128), stixels=dict(sigma=1.0))
    print("evaluate_files stixels %s: epe %.4f (pred %.4f), %.1f segments per image"
          % (flags, summary["stixels"]["epe"], summary["epe"], summary["stixels_per_image"]))
