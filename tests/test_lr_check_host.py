"""CPU: the left-right consistency check.  Its float32 restatement (tests/_lr_restatement.py) on the two-camera synthetic
scene and against a per-pixel reading of the definition; the launch sequence of net(l, r, lr_check=True) by dry run
(tests/_dryrun.py); evaluate_files(lr_check=True) with the kernels replaced by their restatements; and the entry
point's argument checks, which return before any CUDA call."""
import importlib
import os

import numpy as np
import pytest
import torch
from PIL import Image

import _dryrun
import _eval_restatement as O
import _lr_restatement as R
from test_evaluation_host import _FakeStereoLogits, _gt_file, _patch_kernels
from test_kitti_io import _rgb

ev = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.evaluation")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")


# ---- the restatement ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,a,b,d_b,d_f", [(64, 20, 40, 3, 9), (128, 50, 51 + 30, 0, 30), (97, 12, 96, 5, 11)])
@pytest.mark.parametrize("tau", [1.0, 0.0])
def test_synthetic_scene_labels_and_background_fill(W, a, b, d_b, d_f, tau):
    """Background at d_b, a box over [a, b) at d_f: occluded on the band [a - (d_f - d_b), a) the right camera cannot
    see behind the box, out of view for x < d_b, consistent elsewhere; the band and the out-of-view columns fill with
    the background, d_b."""
    dl, dr, want = R.scene(3, W, a, b, d_b, d_f)
    label, filled = R.lr_check(dl, dr, tau)
    assert np.array_equal(label, want)
    band = slice(a - (d_f - d_b), a)
    assert (label[:, band] == R.OCCLUDED).all() and (label[:, :d_b] == R.OUT_OF_VIEW).all()
    assert (filled[:, band] == d_b).all() and (filled[:, :d_b] == d_b).all()
    assert np.array_equal(filled[want == R.CONSISTENT], dl[want == R.CONSISTENT])


def _definition(dl, dr, tau):
    """The definition read literally, one pixel at a time with numpy float32 scalars."""
    f32 = np.float32
    W = len(dl)
    lab = []
    for x in range(W):
        d = dl[x]
        with np.errstate(invalid="ignore", over="ignore"):
            xr = f32(x) - d
            if not (f32(0) <= xr <= f32(W - 1)):
                lab.append(R.OUT_OF_VIEW)
                continue
            x0 = int(np.floor(xr))
            v = dr[x0] if x0 == W - 1 else dr[x0] + (xr - f32(x0)) * (dr[x0 + 1] - dr[x0])
            lab.append(R.CONSISTENT if abs(d - v) <= tau else R.OCCLUDED if v - d > tau else R.MISMATCH)
    cons = [x for x in range(W) if lab[x] == R.CONSISTENT]
    filled = []
    for x in range(W):
        left = [c for c in cons if c < x]
        right = [c for c in cons if c > x]
        if lab[x] == R.CONSISTENT or not (left or right):
            filled.append(dl[x])
        elif left and right:
            filled.append(min(dl[left[-1]], dl[right[0]]))
        else:
            filled.append(dl[left[-1]] if left else dl[right[0]])
    return np.array(lab, np.uint8), np.array(filled, np.float32)


@pytest.mark.parametrize("tau", [1.0, 0.0, 0.25])
def test_restatement_equals_the_definition_pixel_by_pixel(tau):
    rng = np.random.default_rng(int(tau * 8))
    H, W = 6, 37
    dl = (rng.integers(-16, 40 * 8, (H, W)) / 8).astype(np.float32)        # many integer / exact xr
    dr = (dl + rng.integers(-12, 12, (H, W)) / 8).astype(np.float32)
    dl[0, :3] = [np.nan, np.inf, -np.inf]
    dr[1, 5:9] = np.nan
    dl[2, :] = np.arange(W)                                              # xr = 0 everywhere
    dl[3, :] = 0.0                                                       # xr = x, up to W - 1
    dr[4, :] = 500.0                                                     # no consistent pixel on the row
    dl[5, :] = rng.uniform(0, 36, W).astype(np.float32)                  # fractional xr
    label, filled = R.lr_check(dl, dr, tau)
    for y in range(H):
        lab, fil = _definition(dl[y], dr[y], np.float32(tau))
        assert np.array_equal(label[y], lab), y
        assert np.array_equal(filled[y], fil, equal_nan=True), y
    assert (label[4] != R.CONSISTENT).all() and np.array_equal(filled[4], dl[4])


# ---- launch sequence ---------------------------------------------------------------------------------------
def _forward_trace(net, B, **kw):
    g = torch.Generator().manual_seed(0)
    left, right = torch.randn(B, 3, 64, 128, generator=g), torch.randn(B, 3, 64, 128, generator=g)
    with _dryrun.recording() as trace:
        net.packed()
        n0 = len(trace)
        with torch.no_grad():
            out = net(left, right, **kw)
        return list(trace[n0:]), list(trace.full[n0:]), out


def _check_lr_sequence(net, squeeze, **kw):
    import dcanet_b200 as d
    plain, _, _ = _forward_trace(net, 2, **kw)                # the forward of 2 pairs without the flag
    tr, full, out = _forward_trace(net, 1, lr_check=True, lr_threshold=0.75, **kw)
    assert [t[0] for t in tr].count("dca_lr_consistency") == 1 and tr[-1][0] == "dca_lr_consistency"
    assert tr[:-1] == plain
    up = [r for r in full if r[0] == "dca_convex_upsample"][-1]           # pred4 of the hot path at batch 2
    name, dl, dr, mirrored, label, filled, right, B, H, W, tau, _ = full[-1]
    assert (B, H, W, mirrored, tau) == (1, 64, 128, 1, 0.75)
    assert dl == up[3] and dr == up[3] + 64 * 128 * 4 and right != 0
    lr = out[-1]
    assert isinstance(lr, d.LRCheck)
    shape = (1, 64, 128) if squeeze else (1, 1, 64, 128)
    assert out[0].shape == lr.disp_right.shape == lr.label.shape == lr.filled.shape == shape
    assert lr.label.dtype == torch.uint8 and out[1].shape[0] == 1
    return out


def test_lr_forward_is_the_default_forward_at_twice_the_batch_plus_one_launch():
    """64x128, maxdisp 48: net(l, r, lr_check=True) launches exactly the default forward's sequence for 2 pairs, then
    one dca_lr_consistency over the two halves of that forward's pred4 (right half mirrored) with the given threshold;
    the plain forward of one pair still launches the recorded sequence."""
    import dcanet_b200 as d
    from test_host_sequence import _gold
    net = d.GwcNet(48).eval()
    one, _, (pred, pv) = _forward_trace(net, 1)
    assert one == _gold("kernel_sequence_tiny.json")
    assert pred.shape == (1, 1, 64, 128)
    _check_lr_sequence(net, squeeze=False)
    out = _check_lr_sequence(net, squeeze=False, confidence=True)
    assert len(out) == 4 and isinstance(out[2], d.Confidence) and out[2].peak.shape == (1, 1, 64, 128)


def test_lr_forward_no_cva_variant():
    import dcanet_b200 as d
    net = d.gwcnet_dca0_g.GwcNet(48).eval()
    out = _check_lr_sequence(net, squeeze=True)
    assert len(out) == 3 and out[1].shape == (1, 12, 16, 32)


# ---- evaluate_files(lr_check=True) on the CPU ----------------------------------------------------------------
class _FakeStereoLR(_FakeStereoLogits):
    """_FakeStereoLogits with GwcNet's lr_check output; the right view is a fixed function of the left one."""

    def forward(self, left, right, disp_true=None, confidence=False, lr_check=False, lr_threshold=1.0):
        import dcanet_b200 as d
        disp, lg = super().forward(left, right)
        if not lr_check:
            return disp, lg
        disp_right = disp + torch.sin(disp * 5.0) * 1.5
        label, filled, _ = d.engine.lr_consistency(disp, disp_right, lr_threshold)
        return disp, lg, d.LRCheck(disp_right, label, filled)


def _restated_lr(disp_left, disp_right, tau=1.0, mirrored=False, want_right=False):
    lab, fil = R.lr_check(disp_left.numpy(), disp_right.numpy(), tau)
    return torch.from_numpy(lab), torch.from_numpy(fil), None


@pytest.mark.parametrize("mode", ["fit", "pad16"])
def test_evaluate_files_with_lr_check_equals_a_serial_loop(tmp_path, monkeypatch, mode):
    import dcanet_b200 as d
    _patch_kernels(monkeypatch)
    monkeypatch.setattr(d.engine, "lr_consistency", _restated_lr)
    sizes = [(37, 53), (48, 64), (60, 70), (20, 64)]
    model = _FakeStereoLR().eval()
    quads, rows, cons, fill = [], [], [], []
    for i, (h, w) in enumerate(sizes):
        Image.fromarray(_rgb(10 + i, h, w)).save(tmp_path / f"l{i}.png")
        Image.fromarray(_rgb(50 + i, h, w)).save(tmp_path / f"r{i}.png")
        quads.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"), _gt_file(tmp_path, i, h, w), None))
        gt = ev.read_pfm(quads[-1][2]) if quads[-1][2].endswith(".pfm") else ev.read_kitti_disparity(quads[-1][2])
        pair = io.load_pair(quads[-1][0], quads[-1][1])
        if mode == "fit":
            left, right, _, _ = io.fit_to_crop(pair, 48, 64)
            gt = io.fit_gt_to_crop(gt, 48, 64)
        else:
            x, _, _ = io.pad_to_multiple(torch.from_numpy(pair)[None], 16)
            left, right = x[:, 0:3], x[:, 3:6]
            gt = io.pad_gt_to_multiple(gt, 16)[0]
        gt = gt[None]
        with torch.no_grad():
            pred, _, lr = model(left, right, lr_check=True, lr_threshold=0.5)
        rows.append(O.disparity_metric_counts(pred, gt, 48)[0])
        cons.append(O.disparity_metric_counts(pred, np.where(lr.label.numpy()[:, 0] == 0, gt, 0), 48)[0])
        fill.append(O.disparity_metric_counts(lr.filled, gt, 48)[0])
    kw = dict(mode=mode, crop=(48, 64), depth=2, workers=2, maxdisp=48)
    summary, got = ev.evaluate_files(model, quads, lr_check=True, lr_threshold=0.5, **kw)
    plain, plain_rows = ev.evaluate_files(model, quads, **kw)
    assert np.array_equal(got, plain_rows) and np.array_equal(got.astype(np.int64), np.stack(rows))
    assert {k: v for k, v in summary.items() if not k.startswith("lr_")} == plain
    assert set(summary) - set(plain) == {"lr_consistent", "lr_filled", "lr_density"}
    assert summary["lr_consistent"] == ev.summarize(np.stack(cons).astype(np.uint64))
    assert summary["lr_filled"] == ev.summarize(np.stack(fill).astype(np.uint64))
    assert 0.0 < summary["lr_density"] < 1.0
    assert summary["lr_density"] == summary["lr_consistent"]["n_valid"] / summary["n_valid"]


# ---- the entry point's argument checks ------------------------------------------------------------------------
def test_lr_entry_point_rejects_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    ok = [p, p, 1, p, p, 0, 2, 4, 8, 1.0, None]

    def call(**kw):
        args = list(ok)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_lr_consistency(*args)

    for i in (0, 1, 3, 4):
        assert call(**{f"a{i}": None}) == -1
    assert call(a6=0) == call(a7=0) == call(a8=0) == call(a8=-3) == call(a6=65536) == -1
    assert call(a9=float("nan")) == call(a9=-1e-6) == -1
    assert call(a8=4097) == -3
