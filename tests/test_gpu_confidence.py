"""GPU: dca_softmax_confidence_upsample against its fp64 restatement, the confidence of the forward against the reference
fixture and the live oracle, graphed = eager, the stage-count variants, dca_confidence_histograms integer-exact, and the
meter / evaluate_files with a confidence map."""
import importlib

import numpy as np
import pytest
import torch

import _confidence_restatement as C

pytestmark = pytest.mark.gpu

ev = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.evaluation")
FIX_PEAK, FIX_STD = 2e-3, 0.05       # forward vs the reference's head logits: |d peak|, |d std| px


def _engine():
    import dcanet_b200 as d
    return d.engine


def _logits_mask(B, D, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    lg = torch.randn(B, D, H, W, generator=g) * 3
    lg[0, :, 0, 0] = 1.5                                     # flat row: p = 1/D
    lg[0, :, H - 1, W - 1] = 0.0
    lg[0, D // 3, H - 1, W - 1] = 60.0                       # one-hot row: peak 1, std ~ 0
    mask = torch.randn(B, H, W, 144, generator=g) * 2
    return lg, mask


@pytest.mark.parametrize("B,D,H,W", [(1, 12, 7, 5), (2, 48, 40, 37), (1, 96, 16, 32)])
def test_kernel_matches_the_fp64_restatement(B, D, H, W):
    E = _engine()
    lg, mask = _logits_mask(B, D, H, W, seed=D + H)
    conf, pq, sq = E.softmax_confidence_upsample(lg.cuda(), mask.cuda(), quarter=True)
    rpq, rsq, rpeak, rstd = C.confidence(lg, mask)
    dq = (pq.cpu().double()[:, 0] - rpq).abs().max(), (sq.cpu().double()[:, 0] - rsq).abs().max()
    df = (conf.peak.cpu().double() - rpeak).abs().max(), (conf.std.cpu().double() - rstd).abs().max()
    print("confidence kernel %s: 1/4 res |d peak| %.2e |d std| %.2e; full res |d peak| %.2e |d std| %.2e px"
          % ((B, D, H, W), dq[0], dq[1], df[0], df[1]))
    assert dq[0] <= 1e-6 and df[0] <= 1e-6
    assert 4 * dq[1] <= 1e-4 and df[1] <= 1e-4                # std in full-res px
    assert float(conf.peak.min()) >= 0.0 and float(conf.peak.max()) <= 1.0
    assert float(pq.min()) >= 1.0 / D - 1e-7 and float(pq.max()) <= 1.0
    assert abs(float(pq[0, 0, 0, 0]) - 1.0 / D) < 1e-7 and float(pq[0, 0, H - 1, W - 1]) == 1.0
    assert float(sq[0, 0, H - 1, W - 1]) < 1e-6
    conf2, n1, n2 = E.softmax_confidence_upsample(lg.cuda(), mask.cuda(), quarter=False)   # NULL 1/4-res outputs
    assert n1 is None and n2 is None
    assert torch.equal(conf2.peak, conf.peak) and torch.equal(conf2.std, conf.std)


def test_kernel_rejects_bad_arguments():
    from dcanet_b200 import _lib
    lib = _lib.load()
    lg, mask = torch.zeros(1, 4, 2, 2, device="cuda"), torch.zeros(1, 2, 2, 144, device="cuda")
    pk, sd = torch.empty(1, 1, 8, 8, device="cuda"), torch.empty(1, 1, 8, 8, device="cuda")
    a = (lg.data_ptr(), mask.data_ptr(), 0, 0, pk.data_ptr())
    s = torch.cuda.current_stream().cuda_stream
    assert lib.dca_softmax_confidence_upsample(*a, 0, 1, 4, 2, 2, s) == -1
    assert lib.dca_softmax_confidence_upsample(*a, sd.data_ptr(), 1, 4, 0, 2, s) == -1
    assert lib.dca_softmax_confidence_upsample(*a, sd.data_ptr(), 70000, 4, 1, 1, s) == -1
    assert lib.dca_softmax_confidence_upsample(*a, sd.data_ptr(), 1, 4, 2, 2, s) == 0
    torch.cuda.synchronize()
    assert 0.0 < float(pk.min()) <= float(pk.max()) <= 0.25 and float(sd.max()) > 0     # p = 1/4, zero padding


def _load_into(model, sd):
    own = model.state_dict()
    own.update(sd)
    model.load_state_dict(own)
    return model


def test_forward_confidence_against_the_reference_fixture():
    """peak / std of hot_path(confidence=True) against the restatement from the fixture's reference classif3 logits and
    the oracle's prop-net mask on the fixture's guidance features; pred4 / prob_volume2 bit-identical to the plain forward."""
    import dcanet_b200 as d
    from _util import load_e2e
    z, sd, maxdisp = load_e2e()
    net = _load_into(d.GwcNet(maxdisp), sd).cuda().eval()
    cu = lambda k: torch.from_numpy(z[k]).cuda()
    feats = [cu(k) for k in ("gwc_l", "gwc_r", "cat_l", "cat_r", "g")]
    with torch.no_grad():
        pred4, pv = net.hot_path(*feats)
        pred4c, pvc, conf = net.hot_path(*feats, confidence=True)
        mask = C.prop_mask(sd, torch.from_numpy(z["g"]))
    assert torch.equal(pred4, pred4c) and torch.equal(pv, pvc)
    _, _, rpeak, rstd = C.confidence(torch.from_numpy(z["classif3_logits"]), mask)
    dp = float((conf.peak.cpu().double() - rpeak).abs().max())
    ds = float((conf.std.cpu().double() - rstd).abs().max())
    print("fixture 64x128: max |d peak| %.2e, max |d std| %.2e px" % (dp, ds))
    assert dp <= FIX_PEAK and ds <= FIX_STD


def test_forward_confidence_kitti_full_size_against_the_oracle():
    """KITTI 384x1248, maxdisp 192, seed 2 of test_gpu_e2e: the same comparison against the live oracle's head logits."""
    import dcanet_b200 as d
    from oracle import dcanet_oracle as Or
    feats = Or.synth_features(2, 1, 96, 312, shift=3)
    sd = Or.calibrate_state_dict(Or.synth_state_dict(2), feats, 192)
    col = {}
    with torch.no_grad():
        Or.hot_path(sd, *feats, maxdisp=192, collect=col)
        mask = C.prop_mask(sd, feats[4])
    net = _load_into(d.GwcNet(192), sd).cuda().eval()
    with torch.no_grad():
        pred4, pv, conf = net.hot_path(*[f.cuda() for f in feats], confidence=True)
    assert conf.peak.shape == conf.std.shape == (1, 1, 384, 1248)
    _, _, rpeak, rstd = C.confidence(col["classif3_logits"], mask)
    dp = float((conf.peak.cpu().double() - rpeak).abs().max())
    ds = float((conf.std.cpu().double() - rstd).abs().max())
    print("KITTI full size: max |d peak| %.2e, max |d std| %.2e px" % (dp, ds))
    assert dp <= FIX_PEAK and ds <= FIX_STD


def test_graphed_confidence_is_bit_identical_and_variants_squeeze():
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(96), 0).cuda().eval()
    f = [t.cuda() for t in workloads.feature_maps(1, 1, 32, 64)]
    with torch.no_grad():
        e = net.hot_path(*f, confidence=True)
        g = net.hot_path_graphed(*f, confidence=True)
        p = net.hot_path_graphed(*f)
        g2 = net.hot_path_graphed(*f, confidence=True)
    assert len(p) == 2 and len(net.graphed().graphs) == 2 and net.graphed().replays == 3
    for x in (g, g2):
        assert torch.equal(x[0], e[0]) and torch.equal(x[1], e[1])
        assert torch.equal(x[2].peak, e[2].peak) and torch.equal(x[2].std, e[2].std)
    assert torch.equal(p[0], e[0]) and torch.equal(p[1], e[1])
    left = torch.randn(1, 3, 64, 128, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    right = torch.roll(left, -4, 3)
    for n, squeeze in ((0, True), (1, True), (2, True), (4, False)):
        mod = getattr(d, f"gwcnet_dca{n}_g")
        m = workloads.init_bench_weights_(mod.GwcNet(48), 0).cuda().eval()
        with torch.no_grad():
            pred, pv = m(left, right)
            pred_c, pv_c, conf = m(left, right, confidence=True)
        shape = (1, 64, 128) if squeeze else (1, 1, 64, 128)
        assert pred.shape == pred_c.shape == conf.peak.shape == conf.std.shape == shape, n
        assert torch.equal(pred, pred_c) and torch.equal(pv, pv_c), n
        assert bool(torch.isfinite(conf.std).all()) and 0.0 <= float(conf.peak.min()) <= float(conf.peak.max()) <= 1.0


def _hist_inputs(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    gt = torch.rand(B, H, W, generator=g) * 100 - 5
    pred = gt + torch.randn(B, H, W, generator=g) * 8
    peak = torch.rand(B, H, W, generator=g) * 1.2 - 0.1
    pf, gf, cf = pred.view(-1), gt.view(-1), peak.view(-1)
    cases = [  # (gt, pred, peak): error / confidence bin edges, E >= 64, non-finite predictions and peaks
        (10.0, 10.0 + 1 / 32, 0.5), (10.0, 10.0 + 2 / 32, 1.0), (10.0, 74.0, 255 / 256), (10.0, 80.0, 1 / 256),
        (10.0, 10.0 - 64.0, 0.0), (10.0, 500.0, 2.0), (10.0, float("nan"), 0.5), (10.0, float("inf"), 0.5),
        (10.0, 11.0, float("nan")), (10.0, 12.0, float("inf")), (10.0, 13.0, float("-inf")), (10.0, 14.0, -0.25)]
    for i, (a, b, c) in enumerate(cases):
        gf[W + i], pf[W + i], cf[W + i] = a, b, c
    return pred, gt, peak


@pytest.mark.parametrize("B,H,W", [(2, 40, 72), (1, 7, 5), (1, 384, 1248)])
@pytest.mark.parametrize("max_valid", [96.0, 0.0])
def test_confidence_histograms_match_the_restatement_exactly(B, H, W, max_valid):
    pred, gt, peak = _hist_inputs(B, H, W, seed=H + W)
    rc, re = C.confidence_histograms(pred, gt, peak, max_valid)
    ch = torch.zeros((ev.CONF_BINS, 2), dtype=torch.int64, device="cuda")
    eh = torch.zeros((ev.ERR_BINS, 2), dtype=torch.int64, device="cuda")
    p, g, c = pred.cuda(), gt.cuda(), peak.cuda()
    ev._confidence_histograms(p, g, c, ch, eh, max_valid)
    assert np.array_equal(ch.cpu().numpy(), rc) and np.array_equal(eh.cpu().numpy(), re)
    assert re[-1, 0] > 0 and rc[0, 0] > 0 and rc[-1, 0] > 0
    rows = torch.zeros((B, ev.METRIC_COUNT), dtype=torch.int64, device="cuda")
    ev._disparity_metrics(p, g, rows, max_valid)
    r = rows.cpu().numpy()
    for h in (rc, re):
        assert h[:, 1].sum() == r[:, ev.SUM_ABS].sum() and h[:, 0].sum() == (r[:, ev.VALID] - r[:, ev.PRED_NONFINITE]).sum()
    ev._confidence_histograms(p, g, c, ch, eh, max_valid)
    assert np.array_equal(ch.cpu().numpy(), 2 * rc) and np.array_equal(eh.cpu().numpy(), 2 * re)


def test_meter_update_with_confidence_does_not_synchronise():
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    f = [t.cuda() for t in workloads.feature_maps(1, 1, 16, 32)]
    gt = (torch.rand(1, 64, 128, generator=torch.Generator().manual_seed(0)) * 40).cuda()
    m = ev.DisparityMeter(48, capacity=2)
    with torch.no_grad():
        net.hot_path(*f, confidence=True)
        for _ in range(4):
            pred4, pv, conf = net.hot_path(*f, confidence=True)
            torch.cuda.set_sync_debug_mode("error")
            try:
                m.update(pred4, gt, pv, conf.peak)
            finally:
                torch.cuda.set_sync_debug_mode("default")
    ch, eh = m.sparsification_histograms()
    rows = m.rows()
    assert ch[:, 0].sum() == eh[:, 0].sum() == (rows[:, ev.VALID] - rows[:, ev.PRED_NONFINITE]).sum() > 0
    s = m.summary()
    assert s["sparsification_epe"][0] == s["epe_pooled"] and np.isfinite(s["ause_epe"])


def test_evaluate_files_with_confidence_equals_a_serial_loop(tmp_path):
    import dcanet_b200 as d
    import workloads
    from PIL import Image
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    rng = np.random.default_rng(0)
    quads, ref = [], ev.DisparityMeter(48)
    for i, (h, w) in enumerate([(64, 128), (50, 100), (64, 128)]):
        for side in "lr":
            Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).save(tmp_path / f"{side}{i}.png")
        gt = rng.uniform(0, 60, (h, w)).astype(np.float32)
        gt[: h // 4] = 0
        d.kitti_io.save_disparity_png(str(tmp_path / f"g{i}.png"), gt)
        quads.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"), str(tmp_path / f"g{i}.png"), None))
        gt = d.kitti_io.fit_gt_to_crop(ev.read_kitti_disparity(quads[-1][2]), 64, 128)
        left, right, _, _ = d.kitti_io.fit_to_crop(d.kitti_io.load_pair(quads[-1][0], quads[-1][1]), 64, 128)
        with torch.no_grad():
            pred, pv, conf = net(left.cuda(), right.cuda(), confidence=True)
        ref.update(pred, torch.from_numpy(gt)[None].cuda(), pv, conf.peak)
    summary, rows = d.evaluate_files(net, quads, crop=(64, 128), depth=2, workers=2, confidence=True)
    assert np.array_equal(rows, ref.rows())
    assert summary == ref.summary() and len(summary["sparsification_epe"]) == 20
    print("evaluate_files: epe %.3f, auc %.3f, ause %.3f px" % (summary["epe"], summary["auc_epe"], summary["ause_epe"]))
