"""GPU: the semantic-level context -- dca_class_stats, dca_disp_attention and dca_self_attention -- against its float64
restatement (tests/_attention_restatement.py).

The attention kernel is persistent: at most one CTA per SM, each with a few teams that walk the pixels with a stride of
the whole grid, and the D = 24 core route prefetches the next pixel's rows, class and weight while it works on the
current one.  So every attention case here is sized so that every team walks at least 3 pixels (asserted from the SM
count and the team count the launcher picks): the hand-over between pixels, the buffer rows [D, 16 MT) a team reuses
and the per-image S index beyond the first wave all run.  The inputs draw S directly, so w_p = e_p / S[b, k_p] is of
order 1 and a wrong class or weight moves the output far beyond the tolerance (tests/test_attention_host.py).

Tolerances, relative to max |ref| of a case:
  planes = 2: R.TOL2 = 2e-5.
  planes = 1: per element 2^-11 |ref| (the fp16 rounding of the store) plus R.TOL2; the kernel keeps its
              intermediates as hi/lo pairs in either mode.
The reference input is the value the planes hold, so the split of the input is not counted as error.  Measured maxima
of max |err| / max |ref| on an NVIDIA B200 at a 1,000 W power limit, planes = 2 (DCA key form / two-input form):
  D = 24, team mode 1 (core)      1.05e-6 / 1.11e-6
  D = 24, team mode 2             1.01e-6 / 1.00e-6
  D = 24, team mode 0             1.01e-6 / 1.00e-6
  MT 1: D = 1, 8, 16              5.1e-7, 6.9e-7, 8.7e-7
  MT 2: D = 17, 30, 32            1.20e-6, 1.37e-6, 1.31e-6 / D = 17: 1.32e-6
  MT 3: D = 33, 40, 48            9.5e-7, 1.41e-6, 1.05e-6 / D = 40: 1.84e-6
  MT 4: D = 49, 64                1.84e-6, 2.03e-6 / D = 64: 1.28e-6
  pad 0 / 1 / 2 x has_wa          D = 24: 1.00e-6 to 1.13e-6; D = 17: 7.9e-7 to 1.20e-6
  class_stats -> disp_attention   1.08e-6 (D = 24), 1.02e-6 (D = 40)
planes = 1: at most 5.2e-7 beyond the 2^-11 |ref| of the store's rounding on every route above (the error itself is
2.5e-4 to 4.6e-4 of max |ref|, the fp16 store).  No route stands out: the error grows slowly with D.  dca_class_stats:
every k equal to the float64 argmax where it is decided and on every constructed tie, e at most 5.23 ulps off (D = 256,
B = 3, 7,488 pixels).
"""
import contextlib

import numpy as np
import pytest
import torch

import _attention_restatement as R

pytestmark = pytest.mark.gpu

# bytes of the attention kernel's shared memory, restated from attention_launch (csrc/dca_ops.cu)
_W_BYTES = 7 * 2 * 32 * 40 * 2 + 6 * 64 * 4
_SMEM_CAP = 224 * 1024


def _mods():
    import dcanet_b200 as d
    return d, d.engine, d._lib


def _teams(D, team):
    """Teams per CTA that attention_launch picks: 9 on the core route (D = 24, team mode 1), else 8, fewer when their
    buffers do not fit next to the weights."""
    MT = (D + 15) // 16
    core = D == 24 and team == 1
    pair = 2 * 16 * MT * 40 * 2
    per_team = 4 * pair if core else 2 * pair + 3 * 16 * MT * 32 * 4
    n = 9 if core else 8
    while n > 1 and _W_BYTES + n * per_team > _SMEM_CAP:
        n -= 1
    return n


def _min_pixels_per_team(B, D, H, W, team):
    n = B * H * W
    teams = _teams(D, team)
    grid = min(-(-n // teams), torch.cuda.get_device_properties(0).multi_processor_count)
    return n // (grid * teams)


@contextlib.contextmanager
def _team_mode(team):
    lib = _mods()[2].load()
    if team is not None:
        lib.dca_attention_set_team(team)
    try:
        yield
    finally:
        lib.dca_attention_set_team(1)


_PACK = {}


def _weights():
    """engine.PackedAttention of the seeded cva stage: the buffer the kernel reads and the float64 numbers in it."""
    if not _PACK:
        _, E, _ = _mods()
        m = R.seeded_cva(1).cuda()
        pk = E.PackedAttention(m.slc_net.cross_attention, m.fuse[0][0].weight)
        _PACK["buf"], _PACK["w"] = pk.buf, R.unpack(pk.buf.cpu().numpy())
    return _PACK["buf"], _PACK["w"]


def _eps16():
    _, E, _ = _mods()
    return 2.0 ** -11 if E.plane_dtype() == torch.float16 else 2.0 ** -8


def _launch(xp, buf, pad=0, has_wa=0, kce=None, keyp=None):
    """One launch through the C ABI into an output filled with NaN first: every element, border included, must be
    written.  kce = (k, e, S) device tensors of the DCA key form, keyp = the key planes of the two-input form."""
    _, E, L = _mods()
    B, D, H, W = xp.B, xp.D, xp.H, xp.W
    shape = (B, 2 * D, H + 2, W + 2) if pad == 2 else (B, D + 2 * pad, H + 2 * pad, W + 2 * pad)
    y = E.Planes(*shape, 32, xp.planes, xp.t.device)
    y.t.fill_(float("nan"))
    if keyp is None:
        k, e, S = kce
        L.call("dca_disp_attention", xp.ptr, k.data_ptr(), e.data_ptr(), S.data_ptr(), buf.data_ptr(), has_wa, y.ptr,
               pad, xp.planes, B, 32, D, H, W, E._stream())
    else:
        L.call("dca_self_attention", xp.ptr, keyp.ptr, buf.data_ptr(), y.ptr, xp.planes, B, 32, D, H, W, E._stream())
    return y


_CASES = {}


def _case(D, planes, two_input):
    """Device inputs of the route case at D (shape R.shape_for(D), seed D, as the CPU sensitivity tests) and the float64
    view of what the planes hold."""
    key = (D, planes, two_input)
    if key not in _CASES:
        _, E, _ = _mods()
        B, H, W = R.shape_for(D)
        x, k, e, S = R.inputs(B, D, H, W, seed=D)
        xp = E.Planes.from_ncdhw(torch.from_numpy(x).float().cuda(), planes)
        dev = dict(xp=xp, x64=xp.to_ncdhw().double().cpu().numpy())
        if two_input:
            kp = E.Planes.from_ncdhw(torch.from_numpy(R.key_input(B, D, H, W, seed=D)).float().cuda(), planes)
            dev.update(keyp=kp, key64=kp.to_ncdhw().double().cpu().numpy())
        else:
            k32 = torch.from_numpy(k.astype(np.int32)).cuda()
            e32, S32 = torch.from_numpy(e.astype(np.float32)).cuda(), torch.from_numpy(S.astype(np.float32)).cuda()
            dev.update(kce=(k32, e32, S32), k=k, e=e.astype(np.float32), S=S.astype(np.float32))
        dev["ref"] = {}
        _CASES[key] = dev
    return _CASES[key]


def _reference(c, has_wa):
    if has_wa not in c["ref"]:
        _, w = _weights()
        if "keyp" in c:
            c["ref"][has_wa] = R.disp_attention64(c["x64"], None, None, None, *w, has_wa, key=c["key64"])
        else:
            c["ref"][has_wa] = R.disp_attention64(c["x64"], c["k"], c["e"], c["S"], *w, has_wa)
    return c["ref"][has_wa]


def _check(y, ref, planes, what):
    """|got - ref| <= TOL2 max|ref| (+ 2^-11 |ref| with planes = 1) everywhere; returns the measured error."""
    got = y.to_ncdhw().double().cpu().numpy()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert not np.isnan(got).any(), f"{what}: {int(np.isnan(got).sum())} elements not written"
    scale = float(np.abs(ref).max())
    err = np.abs(got - ref)
    rounding = _eps16() * np.abs(ref) if planes == 1 else 0.0
    excess = float((err - rounding).max()) / scale
    print(f"{what}: max err / max|ref| = {float(err.max()) / scale:.3e}, beyond the store rounding {excess:.3e}")
    assert excess <= R.TOL2, f"{what}: {excess:.3e} of max|ref| = {scale:.3e} beyond the bound"
    return excess


def _borders_bit_equal(y, pad, what):
    t = y.t.view(torch.int16)                                     # [planes][B][D'][H'][W'][C]: compare the bits
    for ax in ((2, 3, 4) if pad == 1 else (3, 4)):
        n = t.shape[ax]
        assert torch.equal(t.select(ax, 0), t.select(ax, 1)), (what, "low border", ax)
        assert torch.equal(t.select(ax, n - 1), t.select(ax, n - 2)), (what, "high border", ax)


# ---- every route at sizes where each team walks several pixels ---------------------------------------------------
_ROUTES = [(24, 1), (24, 2), (24, 0)] + [(D, None) for D in R.ROUTE_D]


@pytest.mark.parametrize("planes", [2, 1])
@pytest.mark.parametrize("D,team", _ROUTES)
def test_disp_attention_route(D, team, planes):
    """The DCA key form on every route: D = 24 in team mode 1 (two warps, mma.sync core, prefetch), 2 (two warps, FMA
    core) and 0 (one warp); MT = 1..4 with exact (16, 32, 48, 64) and partial tiles, B = 1, 2 and 3."""
    B, H, W = R.shape_for(D)
    assert _min_pixels_per_team(B, D, H, W, team if team is not None else 1) >= 3
    c = _case(D, planes, False)
    buf, _ = _weights()
    with _team_mode(team):
        y = _launch(c["xp"], buf, kce=c["kce"])
    _check(y, _reference(c, 0), planes, f"disp_attention D={D} team={team} planes={planes} B={B} {H}x{W}")


@pytest.mark.parametrize("planes", [2, 1])
@pytest.mark.parametrize("D,team", [(24, 1), (24, 2), (24, 0), (17, None), (40, None), (64, None)])
def test_self_attention_route(D, team, planes):
    """The two-input form (explicit key tensor), on the core route too."""
    B, H, W = R.shape_for(D)
    assert _min_pixels_per_team(B, D, H, W, team if team is not None else 1) >= 3
    c = _case(D, planes, True)
    buf, _ = _weights()
    with _team_mode(team):
        y = _launch(c["xp"], buf, keyp=c["keyp"])
    _check(y, _reference(c, 0), planes, f"self_attention D={D} team={team} planes={planes} B={B} {H}x{W}")


# ---- every store -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("has_wa", [0, 1])
@pytest.mark.parametrize("pad", [0, 1, 2])
@pytest.mark.parametrize("planes", [2, 1])
@pytest.mark.parametrize("D", [24, 17])
def test_disp_attention_store(D, planes, pad, has_wa):
    """pad 0 / 1 / 2 x has_wa on the core route (two warps share the store) and on a one-warp partial tile: every
    element written, every border copy bit-equal to the voxel it replicates, the values as store64 lays them out."""
    c = _case(D, planes, False)
    buf, _ = _weights()
    y = _launch(c["xp"], buf, pad=pad, has_wa=has_wa, kce=c["kce"])
    what = f"store D={D} planes={planes} pad={pad} has_wa={has_wa}"
    _check(y, R.store64(_reference(c, has_wa), pad), planes, what)
    if pad:
        _borders_bit_equal(y, pad, what)


def test_core_route_is_deterministic_at_kitti_size():
    """Two launches, the second through engine.disp_attention, give bit-identical planes."""
    _, E, _ = _mods()
    c = _case(24, 2, False)
    buf, _ = _weights()
    a = _launch(c["xp"], buf, pad=2, has_wa=1, kce=c["kce"])
    b = E.disp_attention(c["xp"], *c["kce"], buf, True, pad=2)
    assert torch.equal(a.t.view(torch.int16), b.t.view(torch.int16))


# ---- class statistics --------------------------------------------------------------------------------------------
def _logits(B, D, HW, seed):
    """fp32 logits [B, D, HW] whose pixels cycle through five kinds: 0 random N(0, 9); 1 an exact tie of the two largest
    at d1 < d2; 2 constant (every class ties); 3 +-1e4 + N(0, 1) (exp overflows without the max subtraction); 4 exactly
    +-1e4 (the +1e4 classes tie).  Returns the logits and the mask of the constructed ties (kinds 1, 2, 4)."""
    rng = np.random.default_rng(seed)
    z = rng.standard_normal((B, HW, D)) * 3
    kind = (np.arange(B * HW) % 5).reshape(B, HW)
    sign = np.where(rng.random((B, HW, D)) < 0.5, 1.0, -1.0)
    sign[np.arange(B)[:, None], np.arange(HW)[None, :], rng.integers(0, D, (B, HW))] = 1.0   # at least one +1e4
    d1, d2 = rng.integers(0, D, (2, B, HW))
    m1 = kind == 1
    top = z[m1].max(axis=1, keepdims=True) + 1.0
    z[m1] = np.where((np.arange(D) == d1[m1][:, None]) | (np.arange(D) == d2[m1][:, None]), top, z[m1])
    z[kind == 2] = rng.standard_normal((int((kind == 2).sum()), 1))
    z[kind == 3] = 1e4 * sign[kind == 3] + rng.standard_normal((int((kind == 3).sum()), D))
    z[kind == 4] = 1e4 * sign[kind == 4]
    return np.ascontiguousarray(z.astype(np.float32).transpose(0, 2, 1)), (kind == 1) | (kind == 2) | (kind == 4)


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("H,W", [(1, 1), (1, 31), (3, 11), (48, 156)])
@pytest.mark.parametrize("D", [1, 7, 24, 64, 65, 130, 256])
def test_class_stats(D, H, W, B):
    """k = the float64 first argmax wherever the top two probabilities differ by more than 1e-5 relative, and exactly on
    the constructed ties; e within 8 fp32 ulps of exp(P[k]) (expf's 2 ulps and the fp32 softmax's rounding: at most
    5.2 ulps in an exact-exp fp32 emulation of the kernel's summation order up to D = 256); S within N 2^-41 + 2^-23 S
    of the float64 sum of the kernel's own e over its own classes (the 2^-40 fixed point and the conversion to fp32);
    two runs bit-identical.  D > 64 takes the re-read loop, HW = 31 / 33 partial warps, B = 3 the ticketed conversion
    of every image."""
    _, E, _ = _mods()
    HW = H * W
    z, tie = _logits(B, D, HW, seed=D * 1000 + HW + B)
    P = R.softmax64(z[..., None])[..., 0]                              # [B, D, HW]
    k64, e64, _ = R.class_stats64(z[..., None])
    k64, e64 = k64[..., 0], e64[..., 0]
    top2 = np.sort(P, axis=1)[:, -2:] if D > 1 else np.concatenate([np.zeros_like(P), P], 1)
    decided = (top2[:, 1] - top2[:, 0]) > 1e-5 * top2[:, 1]

    logits = torch.from_numpy(z).reshape(B, D, H, W).cuda()
    cls, e, S = E.class_stats(logits)
    cls2, e2, S2 = E.class_stats(logits)
    assert torch.equal(cls, cls2) and torch.equal(e.view(torch.int32), e2.view(torch.int32))
    assert torch.equal(S.view(torch.int32), S2.view(torch.int32))
    k, e, S = cls.cpu().numpy().reshape(B, HW), e.cpu().numpy().reshape(B, HW), S.cpu().numpy()

    assert np.array_equal(k[tie], k64[tie]), "first index of a constructed tie"
    assert np.array_equal(k[decided], k64[decided])
    assert (decided | tie).mean() > 0.9
    ulp = 2.0 ** (np.floor(np.log2(e64)) - 23)
    assert (np.abs(e - e64) <= 8 * ulp).all(), f"e: {float((np.abs(e - e64) / ulp).max()):.2f} ulps"
    sums, count = np.zeros((B, D)), np.zeros((B, D))
    for b in range(B):
        np.add.at(sums[b], k[b], e[b].astype(np.float64))
        np.add.at(count[b], k[b], 1)
    assert (np.abs(S - sums) <= count * 2.0 ** -41 + 2.0 ** -23 * sums).all()
    print(f"class_stats D={D} B={B} HW={HW}: e {float((np.abs(e - e64) / ulp).max()):.2f} ulps, "
          f"{int((~decided).sum())} undecided pixels")


@pytest.mark.parametrize("D", [24, 40])
def test_class_stats_then_attention(D):
    """The chain the forward runs, on a small image where S sums few pixels (w_p of order 1): dca_class_stats ->
    dca_disp_attention against class_stats64 -> disp_attention64."""
    _, E, _ = _mods()
    B, H, W = 2, 5, 7
    rng = np.random.default_rng(D)
    x = rng.standard_normal((B, 32, D, H, W))
    z = (rng.standard_normal((B, D, H, W)) * 3).astype(np.float32)
    k64, e64, S64 = R.class_stats64(z)
    xp = E.Planes.from_ncdhw(torch.from_numpy(x).float().cuda(), 2)
    cls, e, S = E.class_stats(torch.from_numpy(z).cuda())
    assert np.array_equal(cls.cpu().numpy(), k64)
    buf, w = _weights()
    y = _launch(xp, buf, pad=0, has_wa=1, kce=(cls, e, S))
    ref = R.disp_attention64(xp.to_ncdhw().double().cpu().numpy(), k64, e64, S64, *w, 1)
    _check(y, ref, 2, f"class_stats -> disp_attention D={D}")
