"""GPU: dca_lr_consistency bit-exact against its float32 restatement (tests/_lr_restatement.py) in both layouts, the
synthetic two-camera scene, the argument checks; model(l, r, lr_check=True) against the forwards it stands for; the
meter updates of the check without a host sync, and evaluate_files(lr_check=True) against a serial loop."""
import importlib

import numpy as np
import pytest
import torch

import _lr_restatement as R

pytestmark = pytest.mark.gpu

ev = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.evaluation")


def _engine():
    import dcanet_b200 as d
    return d.engine


def _pair(B, H, W, seed):
    """Disparities on a 1/8 px grid (integer and exact xr are frequent) around a per-row level, with about a quarter
    of the pixels consistent at tau = 1, and the edge cases of the definition on the first rows."""
    rng = np.random.default_rng(seed)
    lvl = rng.uniform(-2, min(W - 1, 60), (B, H, 1))
    dl = (np.round((lvl + rng.normal(0, 3, (B, H, W))) * 8) / 8).astype(np.float32)
    dr = (np.round((lvl + rng.normal(0, 1.5, (B, H, W))) * 8) / 8).astype(np.float32)
    x = np.arange(W, dtype=np.float32)
    rows = [("xr = 0", lambda: (x, None)), ("xr = x up to W-1", lambda: (np.zeros(W, np.float32), None)),
            ("negative d", lambda: (-np.abs(dl[0, 2]) - 0.5, None)),
            ("no consistent pixel", lambda: (None, np.full(W, 1e4, np.float32))),
            ("fractional xr", lambda: (rng.uniform(0, W - 1, W).astype(np.float32), None))]
    for y, (_, f) in enumerate(rows[:H]):
        a, b = f()
        if a is not None:
            dl[0, y] = a
        if b is not None:
            dr[0, y] = b
    dl[0, -1, : min(W, 4)] = [np.nan, np.inf, -np.inf, 3.0][: min(W, 4)]
    dr[-1, -1, W // 2:] = np.nan
    dr[0, -1, -1] = np.inf
    return dl, dr


@pytest.mark.parametrize("B,H,W", [(1, 7, 5), (2, 13, 97), (1, 384, 1248), (2, 3, 4096)])
@pytest.mark.parametrize("mirrored", [False, True])
@pytest.mark.parametrize("tau", [1.0, 0.0])
def test_kernel_equals_the_restatement_exactly(B, H, W, mirrored, tau):
    E = _engine()
    dl, dr = _pair(B, H, W, seed=W + H + int(mirrored))
    want_label, want_filled = R.lr_check(dl, dr, tau)
    src = np.ascontiguousarray(dr[..., ::-1]) if mirrored else dr
    label, filled, right = E.lr_consistency(torch.from_numpy(dl).cuda(), torch.from_numpy(src).cuda(), tau,
                                            mirrored=mirrored, want_right=True)
    assert label.dtype == torch.uint8 and label.shape == filled.shape == right.shape == (B, H, W)
    assert np.array_equal(label.cpu().numpy(), want_label)
    assert np.array_equal(filled.cpu().numpy(), want_filled, equal_nan=True)
    assert np.array_equal(right.cpu().numpy(), dr, equal_nan=True)
    counts = np.bincount(want_label.ravel(), minlength=4)
    print("lr kernel %s mirrored=%d tau=%g: labels %s" % ((B, H, W), mirrored, tau, counts.tolist()))
    if W > 8 and H > 5 and tau > 0:
        assert (counts > 0).all()
    label2, filled2, none = E.lr_consistency(torch.from_numpy(dl).cuda()[:, None], torch.from_numpy(src).cuda()[:, None],
                                             tau, mirrored=mirrored)
    assert none is None and label2.shape == (B, 1, H, W)
    assert torch.equal(label2[:, 0], label) and torch.equal(filled2[:, 0].nan_to_num(), filled.nan_to_num())


@pytest.mark.parametrize("mirrored", [False, True])
def test_kernel_on_the_synthetic_scene(mirrored):
    import dcanet_b200 as d
    dl, dr, want = (a[None] for a in R.scene(4, 1248, 400, 520, 6, 40))          # [1, H, W]
    src = np.ascontiguousarray(dr[..., ::-1]) if mirrored else dr
    label, filled, _ = d.engine.lr_consistency(torch.from_numpy(dl).cuda(), torch.from_numpy(src).cuda(),
                                               mirrored=mirrored)
    assert np.array_equal(label.cpu().numpy(), want)
    f = filled.cpu().numpy()
    assert (f[..., 400 - 34:400] == 6).all() and (f[..., :6] == 6).all() and np.array_equal(f[want == 0], dl[want == 0])
    dr_t = torch.from_numpy(dr).cuda()
    lr = d.lr_consistency(torch.from_numpy(dl).cuda(), dr_t)
    assert isinstance(lr, d.LRCheck) and np.array_equal(lr.label.cpu().numpy(), want)
    assert lr.disp_right is dr_t and torch.equal(lr.filled, filled)


def test_kernel_argument_codes():
    from dcanet_b200 import _lib
    lib = _lib.load()
    s = torch.cuda.current_stream().cuda_stream
    W = 4097
    dl, dr = torch.zeros(1, 2, W, device="cuda"), torch.zeros(1, 2, W, device="cuda")
    lab, fil = torch.empty(1, 2, W, dtype=torch.uint8, device="cuda"), torch.empty(1, 2, W, device="cuda")
    a = [dl.data_ptr(), dr.data_ptr(), 0, lab.data_ptr(), fil.data_ptr(), 0]
    assert lib.dca_lr_consistency(*a, 1, 2, W, 1.0, s) == -3                 # DCA_ERR_UNSUPPORTED above DCA_LR_MAX_W
    assert lib.dca_lr_consistency(*a, 1, 2, W - 1, 1.0, s) == 0
    assert lib.dca_lr_consistency(*a, 1, 2, W - 1, float("nan"), s) == -1
    assert lib.dca_lr_consistency(*a, 1, 2, W - 1, -0.5, s) == -1
    assert lib.dca_lr_consistency(*a, 65536, 1, 1, 1.0, s) == -1
    assert lib.dca_lr_consistency(*a, 1, 0, 4, 1.0, s) == -1
    assert lib.dca_lr_consistency(a[0], a[1], 0, None, a[4], 0, 1, 2, 4, 1.0, s) == -1
    assert lib.dca_lr_consistency(a[0], None, 0, a[3], a[4], 0, 1, 2, 4, 1.0, s) == -1
    torch.cuda.synchronize()
    n = 2 * (W - 1)                                   # the 2 x 4096 launch wrote the first n elements
    assert bool((lab.flatten()[:n] == 0).all()) and bool((fil.flatten()[:n] == 0).all())   # zero disparity: consistent


# ---- the forward ----------------------------------------------------------------------------------------------
def _images(B, H, W, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    left = torch.randn(B, 3, H, W, device="cuda", generator=g)
    return left, torch.roll(left, -4, 3) + 0.1 * torch.randn(B, 3, H, W, device="cuda", generator=g)


@pytest.mark.parametrize("maxdisp,B,H,W", [(48, 2, 64, 128), (192, 1, 384, 1248)])
def test_lr_forward_left_outputs_are_those_of_the_plain_forward(maxdisp, B, H, W):
    """pred / prob_volume bit-identical to model(l, r), disp_right to flip(model(flip(r), flip(l))), and label / filled
    to the function-level check of those two; with confidence=True as well, the Confidence of the left view."""
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(maxdisp), 0).cuda().eval()
    left, right = _images(B, H, W, seed=maxdisp)
    with torch.no_grad():
        pred, pv = net(left, right)
        pred_r, _ = net(right.flip(-1), left.flip(-1))
        pred2, pv2, lr = net(left, right, lr_check=True)
        pred3, pv3, conf3, lr3 = net(left, right, confidence=True, lr_check=True, lr_threshold=2.0)
        _, _, conf = net(left, right, confidence=True)
    assert torch.equal(pred2, pred) and torch.equal(pv2, pv) and torch.equal(pred3, pred) and torch.equal(pv3, pv)
    assert torch.equal(lr.disp_right, pred_r.flip(-1)) and torch.equal(lr3.disp_right, lr.disp_right)
    assert torch.equal(conf3.peak, conf.peak) and torch.equal(conf3.std, conf.std)
    ref = d.lr_consistency(pred, pred_r.flip(-1))
    assert torch.equal(lr.label, ref.label) and torch.equal(lr.filled, ref.filled)
    ref2 = d.lr_consistency(pred, pred_r.flip(-1), 2.0)
    assert torch.equal(lr3.label, ref2.label) and torch.equal(lr3.filled, ref2.filled)
    assert lr.label.shape == lr.filled.shape == lr.disp_right.shape == pred.shape == (B, 1, H, W)
    counts = torch.bincount(lr.label.flatten().long(), minlength=4).tolist()
    print("lr forward %dx%d maxdisp %d: labels %s" % (H, W, maxdisp, counts))


def test_lr_forward_variants_squeeze():
    import dcanet_b200 as d
    import workloads
    left, right = _images(1, 64, 128, seed=0)
    for n, squeeze in ((0, True), (1, True), (2, True), (4, False)):
        mod = getattr(d, f"gwcnet_dca{n}_g")
        m = workloads.init_bench_weights_(mod.GwcNet(48), 0).cuda().eval()
        with torch.no_grad():
            pred, pv = m(left, right)
            pred2, pv2, lr = m(left, right, lr_check=True)
        shape = (1, 64, 128) if squeeze else (1, 1, 64, 128)
        assert pred2.shape == lr.label.shape == lr.filled.shape == lr.disp_right.shape == shape, n
        assert torch.equal(pred, pred2) and torch.equal(pv, pv2), n


# ---- evaluation -----------------------------------------------------------------------------------------------
def test_meter_updates_of_the_lr_check_do_not_synchronise():
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    left, right = _images(1, 64, 128, seed=1)
    gt = (torch.rand(1, 64, 128, generator=torch.Generator().manual_seed(0)) * 40).cuda()
    cons, fill = ev.DisparityMeter(48, capacity=2), ev.DisparityMeter(48, capacity=2)
    with torch.no_grad():
        for _ in range(3):
            pred, pv, lr = net(left, right, lr_check=True)
            torch.cuda.set_sync_debug_mode("error")
            try:
                cons.update(pred, torch.where(lr.label.reshape(gt.shape) == 0, gt, 0.0))
                fill.update(lr.filled, gt)
            finally:
                torch.cuda.set_sync_debug_mode("default")
    assert 0 <= cons.summary()["n_valid"] <= fill.summary()["n_valid"] == 3 * 64 * 128


def test_evaluate_files_with_lr_check_equals_a_serial_loop(tmp_path):
    import dcanet_b200 as d
    import workloads
    from PIL import Image
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    rng = np.random.default_rng(0)
    quads, ref, cons, fill = [], ev.DisparityMeter(48), ev.DisparityMeter(48), ev.DisparityMeter(48)
    for i, (h, w) in enumerate([(64, 128), (50, 100), (64, 128)]):
        base = rng.integers(0, 256, (h, w + 8, 3), dtype=np.uint8)
        Image.fromarray(base[:, :w]).save(tmp_path / f"l{i}.png")          # disparity 8 px
        Image.fromarray(base[:, 8:]).save(tmp_path / f"r{i}.png")
        gt = np.full((h, w), 8.0, np.float32)
        gt[: h // 4] = 0
        d.kitti_io.save_disparity_png(str(tmp_path / f"g{i}.png"), gt)
        quads.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"), str(tmp_path / f"g{i}.png"), None))
        gt = torch.from_numpy(d.kitti_io.fit_gt_to_crop(ev.read_kitti_disparity(quads[-1][2]), 64, 128))[None].cuda()
        left, right, _, _ = d.kitti_io.fit_to_crop(d.kitti_io.load_pair(quads[-1][0], quads[-1][1]), 64, 128)
        with torch.no_grad():
            pred, pv, conf, lr = net(left.cuda(), right.cuda(), confidence=True, lr_check=True)
        ref.update(pred, gt, pv, conf.peak)
        cons.update(pred, torch.where(lr.label.reshape(gt.shape) == 0, gt, 0.0))
        fill.update(lr.filled, gt)
    summary, rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2, confidence=True, lr_check=True)
    plain, plain_rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2, confidence=True)
    assert np.array_equal(rows, ref.rows()) and np.array_equal(rows, plain_rows)
    assert {k: v for k, v in summary.items() if not k.startswith("lr_")} == ref.summary() == plain
    assert summary["lr_consistent"] == cons.summary() and summary["lr_filled"] == fill.summary()
    assert 0.0 <= summary["lr_density"] <= 1.0
    print("evaluate_files lr: density %.3f, epe %.3f, consistent epe %.3f, filled epe %.3f px"
          % (summary["lr_density"], summary["epe"], summary["lr_consistent"]["epe"], summary["lr_filled"]["epe"]))
