"""GPU: dca_wls_filter bit-exact against its float32 restatement (tests/_wls_restatement.py) at degenerate, odd and
KITTI shapes (lines without separators, with a one-element last segment, with many segments), with RGB / RGBA and pitched inputs, with and without peak and label, T = 1..3, non-finite disparities and
pixels below min_support; the real forward's outputs fed through wls_filter; determinism, no host sync and CUDA-graph
replay; the entry point's codes on the device; evaluate_files(wls=...) against a serial loop."""
import importlib

import numpy as np
import pytest
import torch

import _wls_restatement as R

pytestmark = pytest.mark.gpu

wls = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.wls")


def _inputs(B, H, W, seed, C=3):
    rng = np.random.default_rng(seed)
    g, d, _, pk = R.scene(H, W, B, seed=seed, confident=0.6, blocks=(min(H, 6), min(W, 10)))
    if C == 4:
        g = np.concatenate([g, rng.integers(0, 256, (B, H, W, 1), dtype=np.uint8)], 3)
    flat = d.reshape(-1)
    k = flat.size
    flat[rng.integers(0, k, max(1, k // 97))] = np.nan
    flat[rng.integers(0, k, max(1, k // 131))] = np.inf
    flat[rng.integers(0, k, max(1, k // 173))] = -np.inf
    p = pk.reshape(-1)
    p[rng.integers(0, k, max(1, k // 89))] = np.nan
    p[rng.integers(0, k, max(1, k // 61))] = 1.7
    p[rng.integers(0, k, max(1, k // 67))] = -0.4
    if H >= 12 and W >= 12:                      # a block without confident pixels behind strong colour edges
        g[0, 2:10, 2:10, :3] = 0
        g[0, 3:9, 3:9, :3] = 255
        pk[0, 3:9, 3:9] = 0.0
    label = rng.integers(0, 4, (B, H, W)).astype(np.uint8)
    label[rng.random((B, H, W)) < 0.6] = 0
    return g, d, pk, label


CASES = [(3, False, False, False, 1), (4, True, True, True, 3), (3, True, True, False, 2)]


@pytest.mark.parametrize("B,H,W", [(1, 1, 1), (1, 1, 37), (1, 29, 1), (1, 7, 5), (1, 13, 97), (1, 64, 65),
                                   (1, 129, 64), (1, 375, 1242), (2, 375, 1242)])
@pytest.mark.parametrize("C,pitched,with_peak,with_label,T", CASES)
def test_kernel_equals_the_restatement_exactly(B, H, W, C, pitched, with_peak, with_label, T):
    g, d, pk, label = _inputs(B, H, W, seed=H * 7 + W + T, C=C)
    want = R.wls(d, g, pk if with_peak else None, label if with_label else None, T=T)
    if pitched:                                  # maps inside a larger frame, the guide a view of a wider image
        y0, x0 = 3, 5
        frame = lambda a, fill: np.pad(a, ((0, 0), (y0, 4), (x0, 7)), constant_values=fill)
        dd, pp, ll = frame(d, 1e30), frame(pk, 1.0), frame(label, 0)
        big = np.zeros((B, H + 2, W + 9, C), np.uint8)
        big[:, 1:H + 1, 2:W + 2] = g
        gt = torch.from_numpy(big).cuda()[:, 1:H + 1, 2:W + 2]
        window = (y0, x0, H, W, 0)
    else:
        dd, pp, ll, gt, window = d, pk, label, torch.from_numpy(g).cuda(), None
    ref = wls.wls_filter(torch.from_numpy(dd).cuda()[:, None], gt,
                         confidence=torch.from_numpy(pp).cuda() if with_peak else None,
                         label=torch.from_numpy(ll).cuda() if with_label else None, num_iter=T, window=window)
    assert ref.disp.shape == ref.support.shape == (B, 1, H, W)
    got_d, got_s = ref.disp[:, 0].cpu().numpy(), ref.support[:, 0].cpu().numpy()
    assert np.array_equal(got_s, want[1]), np.abs(got_s - want[1]).max()
    assert np.array_equal(got_d, want[0], equal_nan=True), np.nanmax(np.abs(got_d - want[0]))
    if H * W > 1000:
        low = want[1] < 1e-3
        print("wls %s C=%d T=%d: %d pixels below min_support" % ((B, H, W), C, T, int(low.sum())))


def test_a_colour_jump_decouples_on_the_device():
    g, d, _, pk = R.scene(24, 60, seed=9, confident=0.6, blocks=(1, 1))
    g[0, :, :25] = 0
    g[0, :, 25:] = 255
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    whole = wls.wls_filter(cu(d), cu(g), confidence=cu(pk))
    left = wls.wls_filter(cu(d[:, :, :25]), cu(g[:, :, :25]), confidence=cu(pk[:, :, :25]))
    assert torch.equal(whole.disp[:, :, :25], left.disp) and torch.equal(whole.support[:, :, :25], left.support)


def _net(maxdisp):
    import dcanet_b200 as d
    import workloads
    return workloads.init_bench_weights_(d.GwcNet(maxdisp), 0).cuda().eval()


@pytest.mark.parametrize("maxdisp,H,W,window", [(48, 64, 128, (5, 0, 59, 120, 0)),
                                                (192, 384, 1248, (9, 0, 375, 1242, 0))])
def test_forward_outputs_through_wls_filter_equal_the_restatement(maxdisp, H, W, window):
    net = _net(maxdisp)
    gen = torch.Generator(device="cuda").manual_seed(1)
    left = torch.randn(1, 3, H, W, device="cuda", generator=gen)
    right = torch.roll(left, -4, 3) + 0.1 * torch.randn(1, 3, H, W, device="cuda", generator=gen)
    y0, x0, h, w, _ = window
    rgb = torch.randint(0, 256, (1, h, w, 3), dtype=torch.uint8, device="cuda", generator=gen)
    with torch.no_grad():
        pred, pv, conf, lr = net(left, right, confidence=True, lr_check=True)
    ref = wls.wls_filter(lr.filled, rgb, confidence=conf.peak, label=lr.label, window=window)
    cut = lambda t: t[:, 0, y0:y0 + h, x0:x0 + w].cpu().numpy()
    want = R.wls(cut(lr.filled), rgb.cpu().numpy(), cut(conf.peak), cut(lr.label))
    assert np.array_equal(ref.disp[:, 0].cpu().numpy(), want[0]) and np.array_equal(ref.support[:, 0].cpu().numpy(),
                                                                                     want[1])
    plain = wls.wls_filter(pred, rgb, window=window)
    assert np.array_equal(plain.disp[:, 0].cpu().numpy(), R.wls(cut(pred), rgb.cpu().numpy())[0])
    print("forward + wls %dx%d: support < 1e-3 at %d of %d pixels" % (H, W, int((want[1] < 1e-3).sum()), h * w))


def test_repeatable_no_host_sync_and_graph_replay():
    g, d, pk, label = _inputs(2, 96, 160, seed=4, C=4)
    cu = lambda a: torch.from_numpy(a).cuda()
    d_, g_, p_, l_ = cu(d), cu(g), cu(pk), cu(label)
    first = wls.wls_filter(d_, g_, confidence=p_, label=l_, sigma=2.5)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        again = [wls.wls_filter(d_, g_, confidence=p_, label=l_, sigma=2.5) for _ in range(2)]
    finally:
        torch.cuda.set_sync_debug_mode("default")
    for r in again:
        assert torch.equal(r.support, first.support) and torch.equal(r.disp.nan_to_num(7.0), first.disp.nan_to_num(7.0))
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        wls.wls_filter(d_, g_, confidence=p_, label=l_, sigma=2.5)            # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(graph):
        cap = wls.wls_filter(d_, g_, confidence=p_, label=l_, sigma=2.5)
    d_.copy_(torch.flip(d_, [2]))
    graph.replay()
    torch.cuda.synchronize()
    want = R.wls(d[:, :, ::-1], g, pk, label, sigma=2.5)
    assert np.array_equal(cap.support.cpu().numpy(), want[1])
    assert np.array_equal(cap.disp.cpu().numpy(), want[0], equal_nan=True)


def test_kernel_argument_codes():
    from dcanet_b200 import _lib
    lib = _lib.load()
    s = torch.cuda.current_stream().cuda_stream
    B, H, W = 1, 3, 5
    d = torch.full((B, H, W), 10.0, device="cuda")
    g = torch.zeros(B, H, W, 3, dtype=torch.uint8, device="cuda")
    lut = wls._device_lut(d.device, 1.5)
    ref, sup = torch.empty(B, H, W, device="cuda"), torch.empty(B, H, W, device="cuda")
    ws = torch.empty(5 * B * H * W, device="cuda")
    a = [d.data_ptr(), None, None, W, H * W, B, H, W, g.data_ptr(), 3, 3 * W, 3 * W * H, lut.data_ptr(), 8000.0, 3,
         1e-3, ref.data_ptr(), sup.data_ptr(), ws.data_ptr(), s]
    assert lib.dca_wls_filter(*a) == 0
    torch.cuda.synchronize()
    want = R.wls(d.cpu().numpy(), g.cpu().numpy())           # support ~1 up to the fp32 rounding of the solves
    assert np.array_equal(ref.cpu().numpy(), want[0]) and np.array_equal(sup.cpu().numpy(), want[1])
    assert torch.allclose(ref, d, atol=1e-4) and torch.allclose(sup, torch.ones_like(sup), atol=1e-3)
    for i, v in ((0, None), (8, None), (12, None), (16, None), (17, None), (18, None), (3, W - 1), (4, H * W - 1),
                 (5, 0), (9, 2), (10, 3 * W - 1), (14, 0), (14, 9), (13, float("nan")), (13, -1.0),
                 (15, float("nan")), (15, -1.0)):
        b = list(a)
        b[i] = v
        assert lib.dca_wls_filter(*b) == -1, i


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
def test_evaluate_files_with_wls_equals_a_serial_loop(tmp_path, flags):
    import dcanet_b200 as d
    from PIL import Image
    ev = d.evaluation
    net = _net(48)
    pairs = _pngs(tmp_path, [(64, 128), (50, 100), (64, 128)])
    params = dict(lam=2000.0, num_iter=2)
    quads, ref = [], ev.DisparityMeter(48)
    for i, (l, r) in enumerate(pairs):
        h, w = (64, 128) if i != 1 else (50, 100)
        gt = np.full((h, w), 8.0, np.float32)
        gt[: h // 4] = 0
        d.kitti_io.save_disparity_png(str(tmp_path / f"g{i}.png"), gt)
        quads.append((l, r, str(tmp_path / f"g{i}.png"), None))
        gt = torch.from_numpy(ev.read_kitti_disparity(quads[-1][2]))[None].cuda()
        left, right, _, _ = d.kitti_io.fit_to_crop(d.kitti_io.load_pair(l, r), 64, 128)
        rgb = torch.from_numpy(np.asarray(Image.open(l))[:, :, :3].copy()).cuda()
        window = (64 - h, 0, h, w, 0)
        with torch.no_grad():
            out = net(left.cuda(), right.cuda(), **flags)
        if flags:
            pred, _, conf, lr = out
            refined = d.wls_filter(lr.filled, rgb, confidence=conf.peak, label=lr.label, window=window, **params)
        else:
            refined = d.wls_filter(out[0], rgb, window=window, **params)
        ref.update(refined.disp, gt)
    summary, rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2, wls=params, **flags)
    plain, plain_rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2, **flags)
    assert summary["wls"] == ref.summary()
    assert np.array_equal(rows, plain_rows) and {k: v for k, v in summary.items() if k != "wls"} == plain
    assert "wls" not in plain
    print("evaluate_files wls %s: epe %.4f (pred %.4f)" % (flags, summary["wls"]["epe"], summary["epe"]))
