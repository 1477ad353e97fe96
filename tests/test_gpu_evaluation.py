"""GPU: dca_disparity_metrics / dca_class_confusion against their CPU restatements (exact), the metrics of our forward on
the reference-generated fixture, evaluate_files against a serial loop, and DisparityMeter.update without host syncs."""
import importlib

import numpy as np
import pytest
import torch

import _eval_restatement as O

pytestmark = pytest.mark.gpu

ev = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.evaluation")


def _metric_inputs(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    gt = torch.rand(B, H, W, generator=g) * 220 - 10                   # negatives and values >= 192
    pred = gt + torch.randn(B, H, W, generator=g) * 3
    gf, pf = gt.view(-1), pred.view(-1)
    gf[:6] = torch.tensor([0.0, -1.0, 192.0, 500.0, float("inf"), float("nan")])
    up = lambda x: float(np.nextafter(np.float32(x), np.float32(np.inf)))
    # (gt, pred): errors exactly on 1 / 2 / 3 px and on the 5 % boundary of D1, and one ulp above them
    cases = [(10.0, 11.0), (10.0, 12.0), (10.0, 13.0), (10.0, 7.0), (80.0, 84.0), (60.0, 63.0), (100.0, 105.0),
             (10.0, up(11.0)), (10.0, up(12.0)), (10.0, up(13.0)), (80.0, up(84.0)), (100.0, up(105.0)),
             (10.0, float("nan")), (10.0, float("inf")), (10.0, float("-inf")), (150.0, float("nan"))]
    for i, (a, b) in enumerate(cases):
        gf[W + 3 + i], pf[W + 3 + i] = a, b
    pf[(B - 1) * H * W + 7] = float("nan")                            # a NaN prediction in the last image
    return pred, gt


@pytest.mark.parametrize("B,H,W", [(3, 40, 72), (3, 40, 37), (1, 7, 5), (2, 64, 128)])
@pytest.mark.parametrize("max_valid", [192.0, 0.0])
def test_disparity_metrics_match_the_restatement_exactly(B, H, W, max_valid):
    """Every counter, the fixed-point SUM_ABS included, equals the fp32 restatement; a second call adds into the same
    rows (vector path W % 4 == 0 and scalar path)."""
    pred, gt = _metric_inputs(B, H, W, seed=W)
    ref = O.disparity_metric_counts(pred, gt, max_valid)
    assert ref[:, ev.PRED_NONFINITE].sum() > 0 and ref[:, ev.D1].sum() > 0
    rows = torch.zeros((B, ev.METRIC_COUNT), dtype=torch.int64, device="cuda")
    p, g = pred.cuda(), gt.cuda()
    ev._disparity_metrics(p, g, rows, max_valid)
    assert np.array_equal(rows.cpu().numpy(), ref)
    ev._disparity_metrics(p, g, rows, max_valid)
    assert np.array_equal(rows.cpu().numpy(), 2 * ref)


def _class_inputs(B, D8, H8, W8, seed):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(B, D8, H8, W8, generator=g) * 3
    logits[0, 3, 1, 2] = logits[0, 1, 1, 2] = 40.0                   # an exact tie: the first index wins
    gt = torch.rand(B, 8 * H8, 8 * W8, generator=g) * (8 * D8 + 24) - 4
    s = gt[:, ::8, ::8]
    s[0, 0, :6] = torch.tensor([0.0, -2.0, float("inf"), float("nan"), 4.0, 3.999])   # invalid ones; class 1 vs 0
    return logits, gt


@pytest.mark.parametrize("D8", [6, 24, 30, 48])
def test_class_confusion_matches_restatement_and_class_stats(D8):
    import dcanet_b200 as d
    B, H8, W8, mv = 2, 5, 37, 8.0 * D8
    logits, gt = _class_inputs(B, D8, H8, W8, seed=D8)
    conf = torch.zeros((D8, D8), dtype=torch.int64, device="cuda")
    lc, gc = logits.cuda(), gt.cuda()
    ev._class_confusion(lc, gc, conf, mv)
    got = conf.cpu().numpy()
    assert np.array_equal(got, O.class_confusion(logits, gt, D8, mv))
    # predicted classes bit-identical to dca_class_stats' class map: the confusion built from that map is the same
    cls = d.engine.class_stats(lc)[0].cpu().long()
    g8 = gt[:, ::8, ::8]
    valid = torch.from_numpy(O.gt_valid_mask(g8, mv))
    gcls = torch.clamp(torch.floor(g8[valid] * 0.125 + 0.5), max=D8 - 1).long()
    want = torch.bincount(gcls * D8 + cls[valid], minlength=D8 * D8).view(D8, D8).numpy()
    assert np.array_equal(got, want)
    ev._class_confusion(lc, gc, conf, mv)
    assert np.array_equal(conf.cpu().numpy(), 2 * want)


def test_class_confusion_refuses_more_than_64_classes():
    from dcanet_b200 import _lib
    conf = torch.zeros((65, 65), dtype=torch.int64, device="cuda")
    with pytest.raises(_lib.DcaError, match="UNSUPPORTED"):
        ev._class_confusion(torch.zeros(1, 65, 2, 2, device="cuda"), torch.ones(1, 16, 16, device="cuda"), conf, 0.0)


def _fixture_net():
    import dcanet_b200 as d
    from _util import load_e2e
    z, sd, maxdisp = load_e2e()
    net = d.GwcNet(maxdisp)
    own = net.state_dict()
    own.update(sd)
    net.load_state_dict(own)
    net = net.cuda().eval()
    cu = lambda k: torch.from_numpy(z[k]).cuda()
    with torch.no_grad():
        pred4, pv2 = net.hot_path(cu("gwc_l"), cu("gwc_r"), cu("cat_l"), cu("cat_r"), cu("g"))
    return z, maxdisp, pred4, pv2


def test_forward_scored_against_the_reference_output():
    """The parity contract restated as metrics on the reference-generated 64x128 fixture: with the reference's pred4 as
    ground truth our forward has EPE <= 0.01 px and no pixel above 1 px; with a GT placed at (8i, 8j) as
    8 * k_ref + 0.25 (k_ref = argmax of the reference's prob_volume2) our class map is purely diagonal."""
    z, maxdisp, pred4, pv2 = _fixture_net()
    m = ev.DisparityMeter(maxdisp, max_valid=0)
    gt = torch.from_numpy(z["pred4"]).cuda().view(pred4.shape[0], pred4.shape[-2], pred4.shape[-1])
    m.update(pred4, gt, None)
    s = m.summary()
    assert s["n_valid"] > 0.9 * gt.numel() and s["n_pred_nonfinite"] == 0
    assert s["epe"] <= 0.01 and s["bad1"] == 0.0, s
    k_ref = torch.from_numpy(z["prob_volume2"]).argmax(dim=1)            # [B,H8,W8]
    gt8 = torch.zeros_like(gt)
    gt8[:, ::8, ::8] = (8 * k_ref + 0.25).float().cuda()
    m2 = ev.DisparityMeter(maxdisp, max_valid=0)
    m2.update(pred4, gt8, pv2)
    cm = m2.confusion()
    assert cm.sum() == k_ref.numel() and np.array_equal(np.diag(np.diag(cm)), cm), cm
    assert m2.summary()["pixel_accuracy"] == 1.0


@pytest.mark.parametrize("mode", ["fit", "pad16"])
def test_evaluate_files_equals_serial_forward_and_meter(tmp_path, mode):
    """evaluate_files (loader threads, pinned image + GT slots, copy / compute streams) with the real model: rows and
    confusion bit-identical to a serial loop of forward + DisparityMeter.update; more pairs than slots, padded and exact
    sizes, KITTI PNG and PFM ground truth."""
    import dcanet_b200 as d
    import workloads
    from PIL import Image
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    rng = np.random.default_rng(0)
    quads = []
    ref = ev.DisparityMeter(48)
    for i, (h, w) in enumerate([(64, 128), (50, 100), (64, 128), (60, 128), (64, 90)]):
        for side in "lr":
            Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).save(tmp_path / f"{side}{i}.png")
        gt = rng.uniform(0, 60, (h, w)).astype(np.float32)
        gt[: h // 4] = 0
        if i % 2:
            d.kitti_io.save_disparity_png(str(tmp_path / f"g{i}.png"), gt)
            gpath = str(tmp_path / f"g{i}.png")
        else:
            gpath = str(tmp_path / f"g{i}.pfm")
            with open(gpath, "wb") as f:
                f.write(b"Pf\n%d %d\n-1.0\n" % (w, h) + np.ascontiguousarray(gt[::-1]).astype("<f4").tobytes())
        quads.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"), gpath,
                      str(tmp_path / f"p{i}.png") if i % 2 == 0 else None))
        gt = ev.read_pfm(gpath) if gpath.endswith(".pfm") else ev.read_kitti_disparity(gpath)
        pair = d.kitti_io.load_pair(quads[-1][0], quads[-1][1])
        if mode == "fit":
            left, right, _, _ = d.kitti_io.fit_to_crop(pair, 64, 128)
            gt = d.kitti_io.fit_gt_to_crop(gt, 64, 128)
        else:
            x, top, _ = d.kitti_io.pad_to_multiple(torch.from_numpy(pair)[None], 16)
            left, right = x[:, 0:3], x[:, 3:6]
            gt = d.kitti_io.pad_gt_to_multiple(gt, 16)[0]
        with torch.no_grad():
            pred, pv = net(left.cuda(), right.cuda())
        ref.update(pred, torch.from_numpy(gt)[None].cuda(), pv)
        if quads[-1][3]:
            disp = pred.reshape(gt.shape).cpu().numpy()
            disp = d.kitti_io.crop_prediction(disp, h, w, 64, 128) if mode == "fit" else disp[top:top + h, :w]
            d.kitti_io.save_disparity_png(str(tmp_path / f"q{i}.png"), disp)
    summary, rows = d.evaluate_files(net, quads, mode=mode, crop=(64, 128), depth=2, workers=2)
    assert np.array_equal(rows, ref.rows())
    assert summary == ref.summary() and summary["n_class_pixels"] > 0
    for i, q in enumerate(quads):
        if q[3]:
            assert np.array_equal(np.asarray(Image.open(q[3])), np.asarray(Image.open(tmp_path / f"q{i}.png"))), i


def test_meter_update_does_not_synchronise():
    """meter.update between forwards: no host sync (torch's sync debug mode raises on one), the row table growing
    included."""
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    f = [t.cuda() for t in workloads.feature_maps(1, 1, 16, 32)]
    gt = (torch.rand(1, 64, 128, generator=torch.Generator().manual_seed(0)) * 40).cuda()
    m = ev.DisparityMeter(48, capacity=2)
    with torch.no_grad():
        net.hot_path(*f)
        for _ in range(5):
            pred4, pv = net.hot_path(*f)
            torch.cuda.set_sync_debug_mode("error")
            try:
                m.update(pred4, gt, pv)
            finally:
                torch.cuda.set_sync_debug_mode("default")
    rows = m.rows()
    assert rows.shape == (5, ev.METRIC_COUNT) and (rows == rows[0]).all() and rows[0, ev.VALID] > 0
    assert m.confusion().sum() > 0
