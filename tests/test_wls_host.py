"""CPU: the float32 restatement of dca_wls_filter (tests/_wls_restatement.py) against a float64 banded solve, its
invariants (support range, constants, decoupling across a colour jump, non-finite inputs, error reduction), the lambda
schedule and the weight table, wls_filter's argument checks, its C-ABI call (dry run), the entry point's argument codes
without a device, and evaluate_files' check of the wls keys (evaluate_files(wls=...) itself runs in test_gpu_wls.py)."""
import importlib
import math
import os

import numpy as np
import pytest
import torch

import _dryrun
import _wls_restatement as R

wls = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.wls")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")


# ---- the definition against float64 ------------------------------------------------------------------------------
@pytest.mark.parametrize("confident", [0.7, 0.05])
def test_restatement_matches_float64_where_supported(confident):
    g, d, clean, pk = R.scene(96, 312, seed=3, confident=confident)
    ref, sup = R.wls(d, g, pk)
    r64, s64 = R.wls64(d, g, pk)
    m = s64 >= 2e-3
    assert m.mean() > 0.5
    assert np.abs(ref - r64)[m].max() <= 1e-3
    assert np.abs(sup.astype(np.float64) - s64).max() <= 1e-4


def _enclosed_block(H=48, W=64):
    """A block with no confident pixel, enclosed by colour edges whose weights are exactly 0 or tiny."""
    g, d, _, pk = R.scene(H, W, seed=5, confident=0.5, blocks=(1, 1))
    g[:] = 0
    g[0, 16:32, 20:40] = (255, 255, 255)
    pk[0, 16:32, 20:40] = 0.0
    return g, d, pk


def test_pixels_without_support_keep_the_input():
    g, d, pk = _enclosed_block()
    ref, sup = R.wls(d, g, pk)
    low = sup < 0.5e-3
    assert low.sum() == 16 * 20
    assert np.array_equal(ref[low], d[low])
    assert (sup[~low] >= 1e-3).all()


def test_support_in_unit_interval_and_constants_stay():
    g, d, _, pk = R.scene(40, 70, seed=7, confident=0.3)
    _, sup = R.wls(d, g, pk)
    assert sup.min() >= 0.0 and sup.max() <= 1.0
    const = np.full((1, 40, 70), 37.25, np.float32)
    ref, sup = R.wls(const, g)
    assert np.abs(ref - 37.25).max() <= 1e-4 and np.abs(sup - 1.0).max() <= 1e-4


def test_a_colour_jump_whose_weight_underflows_decouples_the_two_sides():
    assert R.lut(1.5)[3 * 255 * 255] == 0.0
    g, d, _, pk = R.scene(24, 60, seed=9, confident=0.6, blocks=(1, 1))
    g[0, :, :25] = (0, 0, 0)
    g[0, :, 25:] = (255, 255, 255)
    whole = R.wls(d, g, pk)
    left = R.wls(d[:, :, :25], g[:, :, :25], pk[:, :, :25])
    right = R.wls(d[:, :, 25:], g[:, :, 25:], pk[:, :, 25:])
    for k in range(2):
        assert np.array_equal(whole[k], np.concatenate([left[k], right[k]], 2))


def test_non_finite_inputs_never_leak():
    g, d, _, pk = R.scene(32, 48, seed=11, confident=0.9)
    d[0, ::5, ::7] = np.nan
    d[0, 3::6, 2::5] = np.inf
    d[0, 1::9, 4::3] = -np.inf
    pk[0, ::4, ::3] = np.nan
    ref, sup = R.wls(d, g, pk)
    ok = sup >= 1e-3
    assert ok.mean() > 0.9 and np.isfinite(ref[ok]).all() and np.isfinite(sup).all()
    label = (np.arange(32 * 48).reshape(1, 32, 48) % 3).astype(np.uint8)
    ref, sup = R.wls(d, g, pk, label)
    assert np.isfinite(ref[sup >= 1e-3]).all()


def test_the_synthetic_scene_error_drops():
    g, d, clean, pk = R.scene(96, 312, seed=13, confident=0.7)
    ref, _ = R.wls(d, g, pk)
    before, after = np.abs(d - clean).mean(), np.abs(ref - clean).mean()
    assert after < 0.5 * before, (before, after)


# ---- schedule, table ---------------------------------------------------------------------------------------------
def test_lambda_schedule_and_weight_table():
    for T in range(1, 9):
        s = wls.lambda_schedule(8000.0, T)
        assert s == R.schedule(8000.0, T) and all(v.dtype == np.float32 for v in s)
        for t, v in enumerate(s, 1):
            assert v == np.float32(8000.0 * 1.5 * 4.0 ** (T - t) / (4.0 ** T - 1))
        assert sum(float(v) for v in s) == pytest.approx(4000.0, rel=1e-6)        # sum of 4^(T-t) = (4^T - 1) / 3
    t = wls.weight_table(1.5)
    assert t.dtype == np.float32 and t.shape == (wls.LUT_SIZE,) and np.array_equal(t, R.lut(1.5))
    assert t[0] == 1.0 and t[1] == np.float32(math.exp(-1 / 1.5)) and t[900] == np.float32(math.exp(-20.0))
    assert (np.diff(t) <= 0).all() and t[-1] == 0.0


# ---- wrapper: arguments and the call -----------------------------------------------------------------------------
def test_wls_filter_rejects_bad_arguments_on_the_host():
    d = torch.zeros(1, 1, 8, 12)
    g = torch.zeros(1, 8, 12, 3, dtype=torch.uint8)
    bad = [dict(disp=torch.zeros(1, 8, 12, dtype=torch.float64)), dict(disp=torch.zeros(8, 12)),
           dict(guide=torch.zeros(1, 8, 12, 3)), dict(guide=torch.zeros(1, 8, 11, 3, dtype=torch.uint8)),
           dict(guide=torch.zeros(1, 8, 12, 2, dtype=torch.uint8)), dict(guide=np.zeros((1, 8, 12, 3), np.uint8)),
           dict(confidence=torch.zeros(1, 8, 11)), dict(label=torch.zeros(1, 8, 12)),
           dict(num_iter=0), dict(num_iter=9), dict(num_iter=2.0), dict(lam=float("nan")), dict(lam=-1.0),
           dict(lam=float("inf")), dict(sigma=0.0), dict(sigma=float("nan")), dict(min_support=-1e-3),
           dict(min_support=float("nan")), dict(window=(0, 0, 9, 12, 0)), dict(window=(1, 2, 8, 12, 0))]
    for kw in bad:
        args = dict(disp=d, guide=g)
        args.update(kw)
        with pytest.raises(ValueError):
            wls.wls_filter(args.pop("disp"), args.pop("guide"), **args)
    with pytest.raises(ValueError):                                  # a [h,w,C] guide stands for B = 1 only
        wls.wls_filter(torch.zeros(2, 8, 12), g[0])
    with pytest.raises(_lib.DcaError, match="CUDA"):                 # no CPU path
        wls.wls_filter(d, g)


def test_wls_filter_is_one_entry_point_call():
    big = torch.zeros(3, 1, 40, 70)
    pk = torch.zeros(3, 1, 40, 70)
    lab = torch.zeros(3, 1, 40, 70, dtype=torch.uint8)
    rgb = torch.zeros(3, 2, 50, 80, 4, dtype=torch.uint8)                   # a strided RGBA view of view 0
    guide = rgb[:, 0, 5:35, 10:70]
    with _dryrun.recording() as trace:
        r = wls.wls_filter(big, guide, confidence=pk, label=lab, lam=100.0, num_iter=2, min_support=0.5,
                           window=(4, 6, 30, 60, 1))
    assert [t[0] for t in trace] == ["dca_wls_filter"]
    f = trace.full[0]
    assert f[1] == big.data_ptr() + (4 * 70 + 6) * 4 and f[2] == pk.data_ptr() + (4 * 70 + 6) * 4
    assert f[3] == lab.data_ptr() + 4 * 70 + 6
    assert f[4:9] == (70, 40 * 70, 3, 30, 60)
    assert f[9] == guide.data_ptr() and f[10:13] == (4, 80 * 4, 2 * 50 * 80 * 4)
    assert f[14:17] == (100.0, 2, 0.5)
    assert r.disp.shape == r.support.shape == (3, 1, 30, 60)
    assert f[17] == r.disp.data_ptr() and f[18] == r.support.data_ptr()
    with _dryrun.recording() as trace:
        wls.wls_filter(torch.zeros(1, 30, 60), torch.zeros(30, 60, 3, dtype=torch.uint8))
    f = trace.full[0]
    assert f[2] == 0 and f[3] == 0 and f[4:9] == (60, 30 * 60, 1, 30, 60) and f[10:13] == (3, 180, 30 * 180)
    assert f[14:17] == (8000.0, 3, 1e-3)
    with _dryrun.recording() as trace:                                       # mixed layouts: all made contiguous
        wls.wls_filter(big[:, 0, :, :60], torch.zeros(3, 40, 60, 3, dtype=torch.uint8), confidence=torch.zeros(3, 40, 60))
    f = trace.full[0]
    assert f[4:6] == (60, 40 * 60)


def test_entry_point_rejects_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    ok = [p, None, None, 10, 70, 2, 7, 10, p, 3, 30, 210, p, 8000.0, 3, 1e-3, p, p, p, None]

    def call(**kw):
        args = list(ok)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_wls_filter(*args)

    for i in (0, 8, 12, 16, 17, 18):
        assert call(**{f"a{i}": None}) == -1, i
    for i in (5, 6, 7):
        assert call(**{f"a{i}": 0}) == -1 and call(**{f"a{i}": -2}) == -1, i
    assert call(a5=65536) == call(a9=2) == call(a9=5) == -1
    assert call(a3=9) == call(a4=69) == call(a10=29) == call(a11=209) == call(a9=4, a10=39) == -1
    assert call(a14=0) == call(a14=9) == -1
    assert call(a13=float("nan")) == call(a13=-1.0) == call(a13=float("inf")) == -1
    assert call(a15=float("nan")) == call(a15=-1e-3) == -1
    assert call(a6=65536, a7=32768, a3=32768, a4=2 ** 31, a10=3 * 32768, a11=3 * 2 ** 31) == -3


# ---- evaluate_files(wls=...) with the kernels restated ----------------------------------------------------------------
def test_evaluate_files_rejects_unknown_wls_keys():
    import dcanet_b200 as d
    with pytest.raises(ValueError, match="wls"):
        d.evaluate_files(torch.nn.Identity(), [], wls=dict(lam=1.0, radius=3))
