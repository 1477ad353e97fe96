"""CPU: the confidence forward's launch sequence (dry run, tests/_dryrun.py), the graph key, the sparsification summary
against sort-based curves, and evaluate_files(confidence=True) with the kernels replaced by their restatements
(tests/_confidence_restatement.py)."""
import importlib
import os

import numpy as np
import pytest
import torch
from PIL import Image

import _confidence_restatement as C
import _dryrun
import _eval_restatement as O
from test_evaluation_host import _FakeStereoLogits, _gt_file, _patch_kernels
from test_kitti_io import _rgb

ev = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.evaluation")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")

FEAT_C = (320, 320, 12, 12, 64)


# ---- launch sequence ---------------------------------------------------------------------------------------
def _trace(net, H4, W4, **kw):
    """Full dry-run rows (pointers kept) of one hot_path call, and its outputs."""
    feats = [torch.zeros(1, c, H4, W4) for c in FEAT_C]
    with _dryrun.recording() as trace:
        net.packed()
        n0 = len(trace.full)
        with torch.no_grad():
            out = net.hot_path(*feats, **kw)
        return list(trace.full[n0:]), out


def _norm(row):
    return tuple("P" if isinstance(a, int) and a >= (1 << 20) else a for a in row)


def _check_one_extra_launch(base, conf, H4, W4, D4, keep=False):
    """conf = base + one dca_softmax_confidence_upsample right after dca_convex_upsample, reading the mask of that
    upsampling and the logits the head produced; the only other change is the logits output of the fused tail."""
    names = [r[0] for r in conf]
    i = names.index("dca_softmax_confidence_upsample")
    assert names[i - 1] == "dca_convex_upsample" and names.count("dca_softmax_confidence_upsample") == 1
    extra, rest = conf[i], conf[:i] + conf[i + 1:]
    assert len(rest) == len(base)
    changed = [(a, b) for a, b in zip(base, rest) if _norm(a) != _norm(b)]
    for a, b in changed:
        assert a[0] == b[0] == "dca_tap_gather_softmax_regress" and a[3] == 0 and b[3] >= (1 << 20)
        assert _norm(a[:3] + a[4:]) == _norm(b[:3] + b[4:])
    tails = [r for r in rest if r[0] in ("dca_tap_gather_softmax_regress", "dca_softmax_regress")]
    assert len(tails) == 1
    logits = tails[0][3] if tails[0][0] == "dca_tap_gather_softmax_regress" else tails[0][1]
    assert extra[1] == logits and extra[2] == conf[i - 1][1]           # same logits, same mask
    assert extra[7:11] == (1, D4, H4, W4)
    assert (extra[3] != 0) == keep and (extra[4] != 0) == keep        # 1/4-res maps only for `keep`
    return changed


def test_confidence_forward_adds_one_launch_to_the_default_sequence():
    """KITTI 384x1248 / maxdisp 192: the default sequence (pinned by test_host_sequence), the tail kernel now writing its
    logits, and one dca_softmax_confidence_upsample after dca_convex_upsample."""
    import dcanet_b200 as d
    net = d.GwcNet(192).eval()
    base, (pred4, pv) = _trace(net, 96, 312)
    conf, (pred4c, pvc, c) = _trace(net, 96, 312, confidence=True)
    assert len(_check_one_extra_launch(base, conf, 96, 312, 48)) == 1
    assert isinstance(c, d.Confidence) and c.peak.shape == c.std.shape == pred4c.shape == (1, 1, 384, 1248)
    assert pvc.shape == pv.shape
    keep = {}
    kept, _ = _trace(net, 96, 312, confidence=True, keep=keep)
    _check_one_extra_launch(_trace(net, 96, 312, keep={})[0], kept, 96, 312, 48, keep=True)
    assert keep["peak_quarter"].shape == keep["std_quarter"].shape == (1, 1, 96, 312)


def test_confidence_forward_no_cva_variant_and_cuda_core_tail():
    """The 0-stage variant already returns the head's logits: nothing but the extra launch changes.  Without the fused
    tail (CUDA-core head + dca_softmax_regress) the new kernel reads the logits dca_softmax_regress read."""
    import dcanet_b200 as d
    net = d.gwcnet_dca0_g.GwcNet(48).eval()
    base, _ = _trace(net, 16, 32)
    conf, (pred, pv, c) = _trace(net, 16, 32, confidence=True)
    assert _check_one_extra_launch(base, conf, 16, 32, 12) == []
    assert c.peak.shape == pred.shape == (1, 1, 64, 128)
    E = d.engine
    saved = E.Options.fuse_tail
    E.Options.fuse_tail = False
    try:
        net = d.GwcNet(48).eval()
        base, _ = _trace(net, 16, 32)
        conf, _ = _trace(net, 16, 32, confidence=True)
    finally:
        E.Options.fuse_tail = saved
    assert "dca_softmax_regress" in [r[0] for r in base]
    assert _check_one_extra_launch(base, conf, 16, 32, 12) == []


def test_graphed_forward_keys_on_the_confidence_flag(monkeypatch):
    """With and without confidence are two graphs of the same buffers; replays return copies, the Confidence included."""
    import dcanet_b200 as d
    E = d.engine
    gh = E.GraphedHotPath(None)
    captured = []

    class _Graph:
        def replay(self):
            pass

    def capture(ins, confidence=False):
        captured.append(confidence)
        out = (torch.zeros(1, 1, 8, 8), torch.zeros(1, 6, 1, 1))
        return _Graph(), out + ((E.Confidence(torch.ones(1, 1, 8, 8), torch.ones(1, 1, 8, 8)),) if confidence else ())

    monkeypatch.setattr(gh, "_capture", capture)
    monkeypatch.setattr(E, "_require_cuda", lambda *a: None)
    ins = [torch.zeros(1, c, 2, 2) for c in FEAT_C]
    a = gh(*ins, confidence=True)
    b = gh(*ins)
    a2 = gh(*ins, confidence=True)
    assert captured == [True, False] and len(gh.graphs) == 2 and gh.replays == 3
    assert len(b) == 2 and len(a) == 3 and isinstance(a[2], E.Confidence)
    static = next(v for k, v in gh.graphs.items() if k[-1] is True)[1][2]
    assert a[2].peak is not static.peak and a2[2].std is not static.std and torch.equal(a[2].peak, static.peak)


# ---- sparsification summary ----------------------------------------------------------------------------------
def _pixels(sizes, seed):
    """Groups of pixels; group k has one confidence (its own conf bin) and one error value (its own error bin, one group
    at E >= 64 px).  Returns pred, gt, peak fp32 [1, N] and the per-pixel fixed-point error in px."""
    rng = np.random.default_rng(seed)
    n = len(sizes)
    cbins = rng.choice(256, n, replace=False)
    ebins = rng.choice(2048, n, replace=False)
    err = (ebins + rng.uniform(0.1, 0.9, n)) / 32
    err[rng.integers(n)] = 100.0
    peak = (cbins + rng.uniform(0.1, 0.9, n)) / 256
    rep = lambda v: np.repeat(v, sizes).astype(np.float32)
    gt = np.full(sum(sizes), 10.0, np.float32)
    pred = gt + rep(err)
    fix = np.rint(np.abs(pred - gt) * np.float32(2.0 ** 20)).astype(np.float64)
    return pred[None], gt[None], rep(peak)[None], fix * 2.0 ** -20


def _summary(pred, gt, peak):
    ch, eh = C.confidence_histograms(pred, gt, peak, 0.0)
    rows = O.disparity_metric_counts(pred[:, None], gt[:, None], 0.0)
    return ev.summarize(rows.astype(np.uint64), None, ch.astype(np.uint64), eh.astype(np.uint64)), rows, ch, eh


@pytest.mark.parametrize("sizes_seed", [0, 1])
def test_sparsification_curves_equal_sorting_the_pixels(sizes_seed):
    """One error value per bin, N a multiple of 20: the binned curves (boundary bins taken in part) equal sorting the
    pixels by confidence / by error; seed 0 puts every density on a bin boundary (20 equal groups)."""
    rng = np.random.default_rng(10 + sizes_seed)
    sizes = [7] * 20 if sizes_seed == 0 else list(rng.integers(1, 30, 37))
    sizes[-1] += (-sum(sizes)) % 20
    pred, gt, peak, err = _pixels(sizes, sizes_seed)
    s, _, _, _ = _summary(pred, gt, peak)
    curve, oracle = C.sparsification_bruteforce(err, peak[0], ev.SPARSIFICATION_DENSITY)
    assert s["sparsification_density"] == ev.SPARSIFICATION_DENSITY and len(curve) == 20
    np.testing.assert_allclose(s["sparsification_epe"], curve, rtol=1e-12)
    np.testing.assert_allclose(s["sparsification_epe_ideal"], oracle, rtol=1e-12)
    x = 1.0 - np.asarray(ev.SPARSIFICATION_DENSITY)
    trap = lambda y: float(np.sum((np.asarray(y[1:]) + np.asarray(y[:-1])) / 2 * np.diff(x)))
    assert s["auc_epe"] == pytest.approx(trap(curve), rel=1e-12)
    assert s["ause_epe"] == pytest.approx(trap(curve) - trap(oracle), rel=1e-9)
    assert s["ause_epe"] > 0


def test_sparsification_at_full_density_is_epe_pooled_and_tables_add():
    """Both curves at q = 1 equal epe_pooled exactly (same integer sums); two meters' tables summed give the pooled
    result; without both tables there are no sparsification keys."""
    rng = np.random.default_rng(3)
    B, N = 2, 4000
    gt = rng.uniform(-5, 120, (B, N)).astype(np.float32)
    pred = (gt + rng.standard_normal((B, N)) * 4).astype(np.float32)
    peak = rng.uniform(-0.1, 1.1, (B, N)).astype(np.float32)
    pred[0, :3] = [np.nan, np.inf, 5.0]
    peak[0, 3:6] = [np.nan, np.inf, -1.0]
    gt[1, :2] = [np.nan, 0.0]
    ch, eh = C.confidence_histograms(pred, gt, peak, 96.0)
    rows = O.disparity_metric_counts(pred[:, None], gt[:, None], 96.0)
    s = ev.summarize(rows.astype(np.uint64), None, ch.astype(np.uint64), eh.astype(np.uint64))
    assert s["sparsification_epe"][0] == s["epe_pooled"] and s["sparsification_epe_ideal"][0] == s["epe_pooled"]
    assert ch[:, 0].sum() == eh[:, 0].sum() == rows[:, ev.VALID].sum() - rows[:, ev.PRED_NONFINITE].sum()
    assert ch[:, 1].sum() == eh[:, 1].sum() == rows[:, ev.SUM_ABS].sum()
    parts = [C.confidence_histograms(pred[b:b + 1], gt[b:b + 1], peak[b:b + 1], 96.0) for b in range(B)]
    s2 = ev.summarize(rows.astype(np.uint64), None, (parts[0][0] + parts[1][0]).astype(np.uint64),
                      (parts[0][1] + parts[1][1]).astype(np.uint64))
    assert s2 == s
    plain = ev.summarize(rows.astype(np.uint64))
    assert not any(k.startswith(("sparsification", "auc", "ause")) for k in plain)
    assert ev.summarize(rows.astype(np.uint64), None, ch.astype(np.uint64)) == plain
    assert {k: v for k, v in s.items() if k in plain} == plain


# ---- evaluate_files(confidence=True) on the CPU ----------------------------------------------------------------
class _FakeStereoConfidence(_FakeStereoLogits):
    """_FakeStereoLogits with GwcNet's confidence output: peak = a fixed function of the disparity."""

    def forward(self, left, right, disp_true=None, confidence=False):
        import dcanet_b200 as d
        disp, lg = super().forward(left, right)
        if not confidence:
            return disp, lg
        peak = torch.sigmoid(torch.sin(disp * 3.0))
        return disp, lg, d.Confidence(peak, 1.0 - peak)


def test_evaluate_files_with_confidence_equals_a_serial_loop(tmp_path, monkeypatch):
    _patch_kernels(monkeypatch)
    monkeypatch.setattr(ev, "_confidence_histograms", lambda p, g, c, ch, eh, mv: [
        t.add_(torch.from_numpy(h)) for t, h in zip((ch, eh), C.confidence_histograms(p, g, c, mv))])
    sizes = [(37, 53), (48, 64), (60, 70), (20, 64)]
    model = _FakeStereoConfidence().eval()
    quads, rows, ch, eh, cm = [], [], 0, 0, np.zeros((6, 6), np.int64)
    for i, (h, w) in enumerate(sizes):
        Image.fromarray(_rgb(10 + i, h, w)).save(tmp_path / f"l{i}.png")
        Image.fromarray(_rgb(50 + i, h, w)).save(tmp_path / f"r{i}.png")
        quads.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"), _gt_file(tmp_path, i, h, w), None))
        gt = ev.read_pfm(quads[-1][2]) if quads[-1][2].endswith(".pfm") else ev.read_kitti_disparity(quads[-1][2])
        left, right, _, _ = io.fit_to_crop(io.load_pair(quads[-1][0], quads[-1][1]), 48, 64)
        gt = io.fit_gt_to_crop(gt, 48, 64)[None]
        with torch.no_grad():
            pred, lg, conf = model(left, right, confidence=True)
        rows.append(O.disparity_metric_counts(pred, gt, 48)[0])
        cm += O.class_confusion(lg, gt, 6, 48)
        a, b = C.confidence_histograms(pred, gt, conf.peak, 48)
        ch, eh = ch + a, eh + b
    summary, got = ev.evaluate_files(model, quads, crop=(48, 64), depth=2, workers=2, maxdisp=48, confidence=True)
    assert np.array_equal(got.astype(np.int64), np.stack(rows))
    assert summary == ev.summarize(np.stack(rows).astype(np.uint64), cm, ch.astype(np.uint64), eh.astype(np.uint64))
    assert len(summary["sparsification_epe"]) == 20 and "ause_epe" in summary
    plain, _ = ev.evaluate_files(model, quads, crop=(48, 64), depth=2, workers=2, maxdisp=48)
    assert "ause_epe" not in plain


def test_meter_validates_the_confidence_map():
    m = ev.DisparityMeter(48, device="cpu")
    pred, gt = torch.zeros(1, 1, 8, 8), torch.ones(1, 8, 8)
    with pytest.raises(ValueError, match="confidence"):
        m.update(pred, gt, None, torch.zeros(1, 1, 8, 4))
    with pytest.raises(ValueError, match="confidence"):
        m.update(pred, gt, None, torch.zeros(1, 1, 8, 8, dtype=torch.float16))
    assert m.sparsification_histograms() is None


def test_confidence_entry_points_reject_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    assert lib.dca_softmax_confidence_upsample(None, p, 0, 0, p, p, 1, 12, 4, 4, None) == -1
    assert lib.dca_softmax_confidence_upsample(p, None, 0, 0, p, p, 1, 12, 4, 4, None) == -1
    assert lib.dca_softmax_confidence_upsample(p, p, 0, 0, None, p, 1, 12, 4, 4, None) == -1
    assert lib.dca_softmax_confidence_upsample(p, p, 0, 0, p, None, 1, 12, 4, 4, None) == -1
    assert lib.dca_softmax_confidence_upsample(p, p, 0, 0, p, p, 1, 0, 4, 4, None) == -1
    assert lib.dca_softmax_confidence_upsample(p, p, 0, 0, p, p, 1, 12, 4, -1, None) == -1
    assert lib.dca_confidence_histograms(p, p, None, p, p, 1, 4, 4, 0.0, None) == -1
    assert lib.dca_confidence_histograms(p, p, p, p, None, 1, 4, 4, 0.0, None) == -1
    assert lib.dca_confidence_histograms(p, p, p, p, p, 0, 4, 4, 0.0, None) == -1
    assert lib.dca_confidence_histograms(p, p, p, p, p, 1, 4, 4, float("nan"), None) == -1


def test_meter_refuses_to_mix_updates_with_and_without_confidence(monkeypatch):
    """The sparsification tables must cover the pixels of the counter rows: a meter takes a confidence map with every
    update or with none, and says so before launching anything."""
    _patch_kernels(monkeypatch)
    monkeypatch.setattr(ev, "_confidence_histograms", lambda p, g, c, ch, eh, mv: [
        t.add_(torch.from_numpy(h)) for t, h in zip((ch, eh), C.confidence_histograms(p, g, c, mv))])
    pred, gt, peak = torch.rand(1, 1, 8, 8) * 9, torch.rand(1, 8, 8) * 9 + 0.5, torch.rand(1, 1, 8, 8)
    m = ev.DisparityMeter(48, device="cpu")
    m.update(pred, gt, None, peak)
    with pytest.raises(ValueError, match="every update"):
        m.update(pred, gt)
    m.update(pred, gt, None, peak)
    assert len(m) == 2 and m.summary()["sparsification_epe"][0] == m.summary()["epe_pooled"]
    m = ev.DisparityMeter(48, device="cpu")
    m.update(pred, gt)
    with pytest.raises(ValueError, match="every update"):
        m.update(pred, gt, None, peak)
    assert len(m) == 1 and m.sparsification_histograms() is None


def test_prop_mask_restatement_reproduces_the_oracle_upsampling():
    """prop_mask + convex_up (the restatement the GPU tests compare the confidence maps with) give the oracle's own
    convex_upsample of a disparity map: the copy of the oracle's mask lines cannot drift from it unnoticed."""
    from oracle import dcanet_oracle as Or
    feats = Or.synth_features(0, 1, 8, 16, shift=2)
    sd = Or.calibrate_state_dict(Or.synth_state_dict(0), feats, 48)
    disp = torch.rand(1, 1, 8, 16, generator=torch.Generator().manual_seed(0)) * 12
    with torch.no_grad():
        ref = Or.convex_upsample(Or._Ctx(sd), "prop", feats[4], disp).double()
        got = C.convex_up(C.prop_mask(sd, feats[4]), 4.0 * disp[:, 0])       # pred4 = up(4 * pred_quarter)
    assert got.shape == ref.shape == (1, 1, 32, 64)
    assert float((got - ref).abs().max()) < 1e-4 * max(1.0, float(ref.abs().max()))
