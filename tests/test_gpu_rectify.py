"""GPU: dca_rectify and dca_standardise_frame bit-exact against their float32 restatement (tests/_rectify_restatement.py)
at odd shapes, at KITTI raw size, from RGB and RGBA sources with strided pitches, on maps with NaN, out-of-image, integer
and last-row / last-column coordinates; the standardised input within 1 ulp of kitti_io.load_pair for fit (smaller and
larger images) and pad16; rectify without a host sync; rectify_files and reproject_files(rectifier=) against serial
loops; the argument codes on the device."""
import importlib

import numpy as np
import pytest
import torch

import _rectify_restatement as Rs
import _reproject_restatement as R
from test_rectify_host import _kitti_rectifier, _raw_pngs, _small_rectifier, _ulp_close

pytestmark = pytest.mark.gpu

rect = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.rectify")
geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")


def _edge_maps(H, W, Hs, Ws, seed):
    """float32 [2, H, W, 2]: coordinates over (-2, Ws + 1) x (-2, Hs + 1) with NaN, inf, exact integers, the last column
    and row, just inside and just outside the borders."""
    rng = np.random.default_rng(seed)
    m = np.empty((2, H, W, 2), np.float32)
    m[..., 0] = rng.uniform(-2.0, Ws + 1.0, (2, H, W))
    m[..., 1] = rng.uniform(-2.0, Hs + 1.0, (2, H, W))
    f = np.float32
    xs = [np.nan, np.inf, -np.inf, -1.0, np.nextafter(f(-1), f(0)), 0.0, Ws - 1.0, Ws - 0.5, np.nextafter(f(Ws), f(0)),
          float(Ws), 3.0, 2.5, 1e30, -1e30]
    ys = [2.0, 1.0, 0.0, Hs - 1.0, 0.5, np.nan, Hs - 1.0, np.nextafter(f(Hs), f(0)), float(Hs), -1.0, 3.0, 0.0, 1.0, 0.25]
    flat = m.reshape(2, -1, 2)
    n = min(len(xs), flat.shape[1])
    flat[:, :n, 0], flat[:, :n, 1] = np.array(xs[:n], f), np.array(ys[:n], f)
    ints = rng.integers(0, flat.shape[1], flat.shape[1] // 5)
    flat[:, ints] = np.round(flat[:, ints])                            # exact integers (a whole source pixel)
    return m


def _raw(B, Hs, Ws, C, seed, pad=0):
    """uint8 [B, Hs, Ws, C] views into a wider buffer (row pitch (Ws + pad) C) on the device, and the host copies."""
    rng = np.random.default_rng(seed)
    full = rng.integers(0, 256, (2, B, Hs, Ws + pad, C), dtype=np.uint8)
    dev = torch.from_numpy(full).cuda()
    return dev[0, :, :, :Ws], dev[1, :, :, :Ws], full[0, :, :, :Ws], full[1, :, :, :Ws]


@pytest.mark.parametrize("B,Hs,Ws,H,W,C,pad", [(1, 11, 9, 5, 7, 3, 0), (2, 20, 100, 13, 97, 4, 5),
                                               (2, 20, 100, 13, 97, 3, 3), (1, 512, 1392, 375, 1242, 3, 0)])
def test_kernels_equal_the_restatement_exactly(B, Hs, Ws, H, W, C, pad):
    maps = _edge_maps(H, W, Hs, Ws, seed=H * W + C)
    dl, dr, hl, hr = _raw(B, Hs, Ws, C, seed=W, pad=pad)
    rgb, moments = rect._rectify_kernel(dl, dr, torch.from_numpy(maps).cuda(), H, W)
    want_rgb, want_m = Rs.remap(hl, hr, maps)
    assert np.array_equal(rgb.cpu().numpy(), want_rgb)
    assert np.array_equal(moments.cpu().numpy(), want_m)
    assert (want_rgb == 0).any() and (want_rgb > 0).mean() > 0.3
    for mode, crop in (("fit", (8, 8)), ("fit", (max(1, H // 2), max(1, W // 2))), ("pad16", None)):
        frame, _ = Rs.framing(H, W, mode, *(crop or (0, 0)))
        l, r = rect._standardise_kernel(rgb, moments, frame)
        wl, wr = Rs.standardise_frame(want_rgb, want_m, frame)
        assert np.array_equal(l.cpu().numpy(), wl, equal_nan=True) and np.array_equal(r.cpu().numpy(), wr,
                                                                                       equal_nan=True)
    print("rectify %s: bit-exact, %.3f of the pixels zero" % ((B, Hs, Ws, H, W, C, pad), (want_rgb == 0).mean()))


def test_kitti_raw_rectification_and_the_standardised_input():
    """The KITTI raw rig, 1392x512 -> 1242x375, B = 2: bit-exact against the restatement, and the network input within 1
    ulp of load_pair + fit_to_crop / pad_to_multiple on the rectified images (fit to the smaller 384x1248 crop and to a
    larger image's 256x1024 centre crop)."""
    r = _kitti_rectifier()
    dl, dr, hl, hr = _raw(2, 512, 1392, 3, seed=1)
    for mode, crop in (("fit", (384, 1248)), ("fit", (256, 1024)), ("pad16", (384, 1248))):
        x = rect.rectify(dl, dr, r, mode, crop)
        want_rgb, want_m = Rs.remap(hl, hr, r.maps)
        assert np.array_equal(x.rgb.cpu().numpy(), want_rgb)
        frame, window = Rs.framing(375, 1242, mode, *crop)
        wl, wr = Rs.standardise_frame(want_rgb, want_m, frame)
        assert np.array_equal(x.left.cpu().numpy(), wl) and np.array_equal(x.right.cpu().numpy(), wr)
        assert x.window == window
        for b in range(2):
            pair = io.load_pair(want_rgb[b, 0], want_rgb[b, 1])
            if mode == "fit":
                ll, rr, _, _ = io.fit_to_crop(pair, *crop)
            else:
                p, _, _ = io.pad_to_multiple(torch.from_numpy(pair)[None], 16)
                ll, rr = p[:, 0:3], p[:, 3:6]
            assert _ulp_close(x.left[b:b + 1].cpu().numpy(), ll.numpy())
            assert _ulp_close(x.right[b:b + 1].cpu().numpy(), rr.numpy())


def test_rectify_does_not_synchronise_once_the_maps_are_cached():
    r = _small_rectifier()
    dl, dr, _, _ = _raw(2, 40, 56, 4, seed=2, pad=3)
    rect.rectify(dl, dr, r)                                             # uploads the maps
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for mode in ("fit", "pad16", "fit"):
            x = rect.rectify(dl, dr, r, mode, (48, 64))
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert x.left.shape == (2, 3, 48, 64) and torch.isfinite(x.left).all()


def test_entry_point_argument_codes():
    from dcanet_b200 import _lib
    lib = _lib.load()
    s = torch.cuda.current_stream().cuda_stream
    dl, dr, _, _ = _raw(1, 6, 8, 3, seed=3)
    maps = torch.zeros(2, 4, 5, 2, device="cuda")
    rgb = torch.empty(1, 2, 4, 5, 3, dtype=torch.uint8, device="cuda")
    mom = torch.zeros(1, 2, 3, 2, dtype=torch.int64, device="cuda")
    a = [dl.data_ptr(), dr.data_ptr(), 3, 24, 144, 1, 6, 8, maps.data_ptr(), 4, 5, rgb.data_ptr(), mom.data_ptr(), s]
    assert lib.dca_rectify(*a) == 0
    torch.cuda.synchronize()
    want = int(dl[0, 0, 0, 0]), int(dl[0, 0, 0, 0]) ** 2                 # every pixel samples the raw pixel (0, 0)
    assert mom[0, 0, 0].tolist() == [20 * want[0], 20 * want[1]]
    for i, v in ((0, None), (8, None), (12, None), (2, 2), (3, 23), (4, 143), (5, 0), (9, 0), (5, 65536)):
        b = list(a)
        b[i] = v
        assert lib.dca_rectify(*b) == -1, i
    left, right = torch.empty(1, 3, 6, 5, device="cuda"), torch.empty(1, 3, 6, 5, device="cuda")
    f = [rgb.data_ptr(), mom.data_ptr(), 1, 4, 5, left.data_ptr(), right.data_ptr(), 6, 5, 2, 0, 4, 5, s]
    assert lib.dca_standardise_frame(*f) == 0
    torch.cuda.synchronize()
    assert (left[:, :, :2] == 0).all() and (right[:, :, :2] == 0).all()
    for i, v in ((0, None), (6, None), (9, 3), (10, 1), (12, 6), (7, 0)):
        b = list(f)
        b[i] = v
        assert lib.dca_standardise_frame(*b) == -1, i


# ---- pipelines against serial loops ----------------------------------------------------------------------------
def _net():
    import dcanet_b200 as d
    import workloads
    return workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()


def test_rectify_files_equals_a_serial_loop(tmp_path):
    from PIL import Image
    net = _net()
    r = _small_rectifier(raw=(140, 72), rect_size=(128, 60))
    pairs = _raw_pngs(tmp_path, r, 4, rgba_at=(1,))
    triples = [(l, rr, str(tmp_path / f"o{i}.png")) for i, (l, rr) in enumerate(pairs)]
    got = rect.rectify_files(net, triples, r, 64, 128, depth=2, workers=2)
    for i, (l, rr, png) in enumerate(triples):
        a = torch.from_numpy(np.asarray(Image.open(l))[None]).cuda()
        b = torch.from_numpy(np.asarray(Image.open(rr))[None]).cuda()
        x = rect.rectify(a, b, r, "fit", (64, 128))
        with torch.no_grad():
            pred, _ = net(x.left, x.right)
        want = io.crop_prediction(pred[0, 0].cpu().numpy(), 60, 128, 64, 128)
        assert np.array_equal(got[i], want), i
        assert np.array_equal(np.asarray(Image.open(png)), io.save_disparity_png(str(tmp_path / "x.png"), want))
    print("rectify_files: %d pairs, mean disparity %s" % (len(got), [round(float(g.mean()), 3) for g in got]))


@pytest.mark.parametrize("mode", ["fit", "pad16"])
def test_reproject_files_with_a_rectifier_equals_a_serial_loop(tmp_path, mode):
    from PIL import Image
    net = _net()
    r = _small_rectifier(raw=(140, 72), rect_size=(128, 60))
    pairs = _raw_pngs(tmp_path, r, 3)
    items = [(l, rr, str(tmp_path / f"p{i}.ply"), str(tmp_path / f"d{i}.png")) for i, (l, rr) in enumerate(pairs)]
    got = geo.reproject_files(net, items, mode=mode, crop=(64, 128), min_confidence=0.05, lr_check=True,
                              max_depth=500.0, depth=2, rectifier=r)
    c = r.calib
    for i, (l, rr, ply, png) in enumerate(items):
        a = torch.from_numpy(np.asarray(Image.open(l))[None]).cuda()
        b = torch.from_numpy(np.asarray(Image.open(rr))[None]).cuda()
        x = rect.rectify(a, b, r, mode, (64, 128))
        with torch.no_grad():
            pred, _, conf, lr = net(x.left, x.right, confidence=True, lr_check=True)
        pc = geo.reproject(pred, c, confidence=conf.peak, min_confidence=0.05, label=lr.label, max_depth=500.0,
                           window=x.window)
        y0, x0, h, w, vo = x.window
        n = int(pc.count[0])
        xyz, idx = pc.xyz[0, :n].cpu().numpy(), pc.index[0, :n].cpu().numpy()
        col = x.rgb[0, 0, vo:vo + h, x0:x0 + w].cpu().numpy().reshape(-1, 3)[idx]
        assert n > 0 and np.array_equal(got[i][0], xyz) and np.array_equal(got[i][1], col), i
        assert np.array_equal(np.asarray(Image.open(png)),
                              geo.save_depth_png(str(tmp_path / "x.png"), pc.depth[0].cpu().numpy()))
        # the restatement of the reprojection agrees on the same disparity
        cut = lambda t: t[:, 0, y0:y0 + h, x0:x0 + w].cpu().numpy()
        rx, ri, _, _ = R.reproject(cut(pred), cut(conf.peak), cut(lr.label), x0, vo, c.Q(), None, 0.05, 0.0, 500.0)
        assert np.array_equal(rx[0], xyz) and np.array_equal(ri[0], idx)
    print("reproject_files(rectifier=) %s: points per pair %s" % (mode, [len(g[0]) for g in got]))
