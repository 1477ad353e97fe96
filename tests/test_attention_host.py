"""CPU: the float64 restatement of the semantic-level context (tests/_attention_restatement.py) against the oracle and
torch, how far its output moves under modelled kernel bugs compared with the GPU tests' tolerance, and the argument
checks of dca_class_stats / dca_disp_attention / dca_self_attention, which return before any CUDA call."""
import importlib
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import _attention_restatement as R
from oracle import dcanet_oracle as O

_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")

PREFIX = "cva.slc_net.cross_attention"


def _rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def _weights():
    m = R.seeded_cva(1)
    return m, R.fold64(m.slc_net.cross_attention, m.fuse[0][0].weight)


# ---- the restatement against the oracle and torch --------------------------------------------------------------
@pytest.mark.parametrize("B,D,H,W", [(2, 24, 5, 11), (3, 7, 4, 6), (1, 33, 3, 5)])
def test_restatement_matches_the_oracle(B, D, H, W):
    """class_stats64 + disp_attention64 equal oracle.semantic_level_key + disparity_attention in float64, the two-input
    form equals disparity_attention on an explicit key, and has_wa equals the first 32 input channels of cva.fuse's
    conv applied to the output."""
    m, (Wm, sc, sh) = _weights()
    sd = {"cva." + k: (v.double() if v.is_floating_point() else v) for k, v in m.state_dict().items()}
    ctx = O._Ctx(sd)
    rng = np.random.default_rng(B * 100 + D)
    x = rng.standard_normal((B, 32, D, H, W))
    logits = rng.standard_normal((B, D, H, W)) * 3
    logits[0, :, 0, 0] = 1.5                                   # a constant pixel: first index of an exact tie
    xt, lt = torch.from_numpy(x), torch.from_numpy(logits)

    _, k_o, e_o, S_o, _ = O.class_stats(lt)
    k, e, S = R.class_stats64(logits)
    assert np.array_equal(k, k_o.numpy()) and k[0, 0, 0] == 0
    assert np.abs(e - e_o.numpy()).max() <= 1e-15 * 3 and np.abs(S - S_o.numpy()).max() <= 1e-12 * np.abs(S).max()

    key, _ = O.semantic_level_key(xt, lt)
    ref = O.disparity_attention(ctx, PREFIX, xt, key).numpy()
    got = R.disp_attention64(x, k, e, S, Wm, sc, sh, has_wa=0)
    assert _rel(got, ref) <= 1e-12
    assert _rel(R.dca_key64(x, k, e, S), key.numpy()) <= 1e-15

    wa = F.conv3d(torch.from_numpy(ref), m.fuse[0][0].weight.detach().double()[:, :32]).numpy()
    assert _rel(R.disp_attention64(x, k, e, S, Wm, sc, sh, has_wa=1), wa) <= 1e-12

    k2 = rng.standard_normal(x.shape)
    ref2 = O.disparity_attention(ctx, PREFIX, xt, torch.from_numpy(k2)).numpy()
    assert _rel(R.disp_attention64(x, None, None, None, Wm, sc, sh, 0, key=k2), ref2) <= 1e-12


def test_packed_buffer_layout_round_trips():
    """unpack reads the layout engine.PackedAttention writes: 7 matrices [ci][co], then 6 x (scale[32], shift[32])."""
    _, (Wm, sc, sh) = _weights()
    buf = np.concatenate([Wm.ravel(), np.stack([sc, sh], 1).ravel()])
    W2, sc2, sh2 = R.unpack(buf.astype(np.float32))
    assert np.abs(W2 - Wm).max() <= 2 ** -24 * np.abs(Wm).max()
    assert np.abs(sc2 - sc).max() <= 2 ** -24 * 2 and np.abs(sh2 - sh).max() <= 2 ** -24


@pytest.mark.parametrize("D", [1, 2, 5, 24])
def test_store_layouts_match_torch(D):
    y = np.random.default_rng(D).standard_normal((2, 32, D, 3, 4))
    yt = torch.from_numpy(y)
    assert np.array_equal(R.store64(y, 0), y)
    assert np.array_equal(R.store64(y, 1), F.pad(yt, (1, 1, 1, 1, 1, 1), mode="replicate").numpy())
    up = F.interpolate(yt, scale_factor=(2, 1, 1), mode="trilinear", align_corners=False)
    assert np.abs(R.store64(y, 2) - F.pad(up, (1, 1, 1, 1, 0, 0), mode="replicate").numpy()).max() <= 1e-15


# ---- sensitivity: the GPU tolerance must see each modelled bug ---------------------------------------------------
_REFS = {}


def _case(D):
    """The inputs and reference of the GPU test's route case at disparity count D (same shapes and seeds)."""
    if D not in _REFS:
        _, (Wm, sc, sh) = _weights()
        B, H, W = R.shape_for(D)
        x, k, e, S = R.inputs(B, D, H, W, seed=D)
        _REFS[D] = (x, k, e, S, (Wm, sc, sh), R.disp_attention64(x, k, e, S, Wm, sc, sh, 1))
    return _REFS[D]


@pytest.mark.parametrize("D", R.ROUTE_D + (24,))
def test_tolerance_sees_the_neighbouring_pixels_class_and_weight(D):
    """Bug 1: every pixel uses k and e of pixel pix + 1 (the prefetch hand-over off by one), S still of its own image."""
    x, k, e, S, w, ref = _case(D)
    shifted = [np.roll(a.ravel(), -1).reshape(a.shape) for a in (k, e)]
    assert _rel(R.disp_attention64(x, *shifted, S, *w, 1), ref) >= 10 * R.TOL2


@pytest.mark.parametrize("D", [d for d in R.ROUTE_D + (24,) if R.shape_for(d)[0] > 1])
def test_tolerance_sees_image_zeros_class_sums(D):
    """Bug 2: w_p = e_p / S[0, k_p] for every image."""
    x, k, e, S, w, ref = _case(D)
    assert _rel(R.disp_attention64(x, k, e, np.broadcast_to(S[:1], S.shape), *w, 1), ref) >= 10 * R.TOL2


@pytest.mark.parametrize("D", [d for d in R.ROUTE_D + (24,) if d % 16])
def test_tolerance_sees_the_padded_key_rows(D):
    """Bug 3: the buffer rows [D, 16 MT), zero on input, enter the softmax as keys (and their values the sum)."""
    x, k, e, S, w, ref = _case(D)
    key = R.dca_key64(x, k, e, S)
    pad = np.zeros(key.shape[:2] + (16 * ((D + 15) // 16) - D,) + key.shape[3:])
    assert _rel(R.disp_attention64(x, k, e, S, *w, 1, key=np.concatenate([key, pad], 2)), ref) >= 10 * R.TOL2


@pytest.mark.parametrize("D", [24, 17])
def test_tolerance_sees_swapped_depth_weights(D):
    """Bug 4: the pad-2 store weights 0.25 and 0.75 swapped (the GPU store test runs D = 24 and 17)."""
    *_, ref = _case(D)
    swapped = np.pad(R.depth_x2(ref, near=0.25), ((0, 0), (0, 0), (0, 0), (1, 1), (1, 1)), mode="edge")
    assert _rel(swapped, R.store64(ref, 2)) >= 10 * R.TOL2


@pytest.mark.parametrize("D", R.ROUTE_D + (24,))
def test_tolerance_sees_the_lost_lo_plane(D):
    """Bug 5: parity mode drops the input's lo plane, i.e. x is rounded to fp16.  Measured: 15x the tolerance at D = 1,
    30x to 78x at the other route cases."""
    x, k, e, S, w, ref = _case(D)
    x16 = x.astype(np.float16).astype(np.float64)
    assert _rel(R.disp_attention64(x16, k, e, S, *w, 1), ref) >= 3 * R.TOL2


# ---- argument checks (no device needed) ------------------------------------------------------------------------
def test_entry_points_reject_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    ARG, UNSUPPORTED = -1, -3

    def attn(D=24, C=32, pad=0, planes=2, B=1):
        return lib.dca_disp_attention(p, p, p, p, p, 0, p, pad, planes, B, C, D, 4, 4, None)

    assert attn(D=65) == attn(D=65, pad=2) == attn(C=31) == attn(C=64) == UNSUPPORTED
    assert attn(pad=3) == attn(pad=-1) == attn(D=0) == attn(D=-1) == attn(planes=3) == attn(B=0) == ARG
    assert lib.dca_disp_attention(p, None, p, p, p, 0, p, 0, 2, 1, 32, 24, 4, 4, None) == ARG
    assert lib.dca_self_attention(p, p, p, p, 2, 1, 32, 65, 4, 4, None) == UNSUPPORTED
    assert lib.dca_self_attention(p, p, p, p, 2, 1, 31, 24, 4, 4, None) == UNSUPPORTED
    assert lib.dca_self_attention(p, None, p, p, 2, 1, 32, 24, 4, 4, None) == ARG
    assert lib.dca_self_attention(p, p, p, p, 2, 1, 32, 0, 4, 4, None) == ARG

    def stats(D=24, scratch=p, B=1, H=4, W=4):
        return lib.dca_class_stats(p, p, p, p, scratch, B, D, H, W, None)

    assert stats(D=257) == stats(D=0) == stats(scratch=p + 4) == stats(B=0) == stats(H=0) == stats(W=0) == ARG
