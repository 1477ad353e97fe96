"""float64 restatement of the semantic-level context (include/dca_b200.h section 2, csrc/dca_ops.cu) -- TEST
INFRASTRUCTURE.

  class_stats64      (k, e, S) of dca_class_stats from logits [B, D, H, W]
  disp_attention64   the closed form of dca_disp_attention (key built from k, e, S) and of dca_self_attention (explicit
                     key) on x [B, 32, D, H, W]
  store64            the output layouts of the attention's store: pad 0, pad 1 (replicated border), pad 2 (depth x2)
  unpack / fold64    the (W, scale, shift) the kernel reads: from the packed fp32 buffer of engine.PackedAttention, or
                     folded in float64 from the modules
  inputs             seeded x, k, e, S with w_p = e_p / S[b, k_p] of order 1, and the shapes the kernel tests run
  seeded_cva         the seeded module whose attention weights both sides use
"""
import numpy as np

C = 32
HEADS, HEAD_DIM = 4, 8
LEAK = 0.1
# order of the 7 matrices and 6 (scale, shift) pairs in the packed buffer: q0, q1, k0, k1, v, o (+ Wa, no affine)
Q0, Q1, K0, K1, V, O, WA = range(7)

# (B, H, W) per 16-row tile count MT = ceil(D / 16): every team of the persistent attention kernel walks at least 3
# pixels on a 148-SM part (the GPU test computes and asserts the count).  KITTI = 1/8 of a 384x1248 pair at D = 24.
KITTI = (2, 48, 156)
BY_MT = {1: (3, 29, 43), 2: (1, 61, 59), 3: (3, 25, 31), 4: (2, 29, 31)}
# The attention routes the kernel tests run: D = 24 in its three team modes, and MT 1-4 with exact and partial tiles.
ROUTE_D = (1, 8, 16, 17, 30, 32, 33, 40, 48, 49, 64)
# Tolerance of the parity mode (planes = 2) relative to max |ref| of a case; planes = 1 adds the fp16 rounding of the
# store.  The CPU tests hold every modelled indexing bug at 10x this bound, and dropping the input's lo plane at 3x.
TOL2 = 2e-5


def shape_for(D):
    """(B, H, W) the kernel tests run disparity count D at."""
    return KITTI if D == 24 else BY_MT[(D + 15) // 16]


def inputs(B, D, H, W, seed):
    """x [B, 32, D, H, W], k [B, H, W], e [B, H, W] in (1, e], S [B, D] uniform in [1, 4]: drawn independently, so that
    w_p = e_p / S[b, k_p] is of order 1 (S of a real image sums hundreds of pixels and hides a wrong k_p or w_p)."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, C, D, H, W))
    k = rng.integers(0, D, (B, H, W))
    e = np.exp(1.0 - rng.random((B, H, W)))
    S = rng.uniform(1.0, 4.0, (B, D))
    return x, k, e, S


def key_input(B, D, H, W, seed):
    """The second input of the two-input form."""
    return np.random.default_rng(seed + 7919).standard_normal((B, C, D, H, W))


# ---- class statistics ------------------------------------------------------------------------------------------
def softmax64(logits):
    z = np.asarray(logits, np.float64)
    p = np.exp(z - z.max(axis=1, keepdims=True))
    return p / p.sum(axis=1, keepdims=True)


def class_stats64(logits):
    """k = first argmax over d of P = softmax_d(logits), e = exp(P[k]), S[b, c] = sum of e over the pixels of class c
    in image b."""
    P = softmax64(logits)
    B, D = P.shape[:2]
    k = P.argmax(axis=1)
    e = np.exp(np.take_along_axis(P, k[:, None], 1)[:, 0])
    S = np.zeros((B, D))
    for b in range(B):
        np.add.at(S[b], k[b].ravel(), e[b].ravel())
    return k, e, S


# ---- attention -------------------------------------------------------------------------------------------------
def unpack(buf):
    """The flat fp32 buffer of engine.PackedAttention -> W [7][ci][co], scale [6][32], shift [6][32] (float64)."""
    b = np.asarray(buf, np.float64).ravel()
    assert b.size == 7 * C * C + 6 * 2 * C
    ss = b[7 * C * C:].reshape(6, 2, C)
    return b[:7 * C * C].reshape(7, C, C), ss[:, 0], ss[:, 1]


def fold64(attn, fuse_weight=None):
    """The same numbers from a SelfAttentionBlock (and cva.fuse's conv weight, whose first 32 input channels act on the
    attention output), BatchNorm folded in float64: scale = gamma / sqrt(var + eps), shift = beta - mean * scale."""
    seqs = [attn.query_project[0], attn.query_project[1], attn.key_project[0], attn.key_project[1],
            attn.value_project, attn.out_project]
    W = np.zeros((7, C, C))
    scale, shift = np.zeros((6, C)), np.zeros((6, C))
    for i, (conv, bn) in enumerate(s[:2] for s in seqs):
        W[i] = conv.weight.detach().double().numpy()[:, :, 0, 0, 0].T
        g, bt = bn.weight.detach().double().numpy(), bn.bias.detach().double().numpy()
        m, v = bn.running_mean.detach().double().numpy(), bn.running_var.detach().double().numpy()
        scale[i] = g / np.sqrt(v + bn.eps)
        shift[i] = bt - m * scale[i]
    if fuse_weight is not None:
        W[WA] = fuse_weight.detach().double().numpy()[:, :C, 0, 0, 0].T
    return W, scale, shift


def _project(xl, W, scale, shift, i):
    """1x1x1 conv + folded BN + LeakyReLU(0.1) on channels-last rows."""
    y = (xl @ W[i]) * scale[i] + shift[i]
    return np.where(y > 0, y, LEAK * y)


def _heads(t):
    """[HW, D, 32] -> [HW, 4, D, 8]: channel = head * 8 + c."""
    return t.reshape(t.shape[0], t.shape[1], HEADS, HEAD_DIM).transpose(0, 2, 1, 3)


def dca_key64(x, k, e, S):
    """key[d] = x[d] * (1 + [d == k_p] * e_p / S[b, k_p])."""
    x = np.asarray(x, np.float64)
    B, _, D, H, W = x.shape
    k = np.asarray(k)
    w = np.asarray(e, np.float64) / np.take_along_axis(np.asarray(S, np.float64), k.reshape(B, -1), 1).reshape(B, H, W)
    onehot = np.arange(D)[None, :, None, None] == k[:, None]
    return x * (1.0 + onehot * w[:, None])[:, None]


def disp_attention64(x, k, e, S, W, scale, shift, has_wa, key=None):
    """q = Pq1(Pq0(x)), k = Pk1(Pk0(key)), v = Pv(key); per pixel and head (4 x 8 channels) the softmax over the keys of
    q k^T / sqrt(8), times v; out = Po(ctx); with has_wa t = Wa out (no affine).  key = the explicit key tensor, or the
    DCA key of (k, e, S).  Queries and keys may differ in depth (rows D of x, Dk of key).  -> [B, 32, D, H, W]"""
    x = np.asarray(x, np.float64)
    key = dca_key64(x, k, e, S) if key is None else np.asarray(key, np.float64)
    B, _, D, H, Wd = x.shape
    Dk = key.shape[2]
    out = np.empty((B, D, H, Wd, C))
    for b in range(B):                                            # one image at a time: the scores are B*HW*4*D*Dk
        xl = np.moveaxis(x[b], 0, -1).reshape(D, H * Wd, C).transpose(1, 0, 2)      # [HW, D, 32]
        kl = np.moveaxis(key[b], 0, -1).reshape(Dk, H * Wd, C).transpose(1, 0, 2)
        q = _project(_project(xl, W, scale, shift, Q0), W, scale, shift, Q1)
        kk = _project(_project(kl, W, scale, shift, K0), W, scale, shift, K1)
        v = _project(kl, W, scale, shift, V)
        s = _heads(q) @ _heads(kk).transpose(0, 1, 3, 2) * HEAD_DIM ** -0.5                       # [HW, 4, D, Dk]
        p = np.exp(s - s.max(axis=-1, keepdims=True))
        ctx = (p / p.sum(axis=-1, keepdims=True)) @ _heads(v)                                    # [HW, 4, D, 8]
        ctx = ctx.transpose(0, 2, 1, 3).reshape(H * Wd, D, C)
        o = _project(ctx, W, scale, shift, O)
        if has_wa:
            o = o @ W[WA]
        out[b] = o.transpose(1, 0, 2).reshape(D, H, Wd, C)
    return np.moveaxis(out, -1, 1)


# ---- store layouts ---------------------------------------------------------------------------------------------
def depth_x2(y, near=0.75):
    """x2 along depth (axis 2), align_corners=False: output 2i + 1 = near * y[i] + (1 - near) * y[i + 1], 2i =
    (1 - near) * y[i - 1] + near * y[i], the neighbour index clamped to [0, D)."""
    D = y.shape[2]
    i = np.arange(D)
    lo, hi = y[:, :, np.maximum(i - 1, 0)], y[:, :, np.minimum(i + 1, D - 1)]
    out = np.empty(y.shape[:2] + (2 * D,) + y.shape[3:])
    out[:, :, 0::2] = (1 - near) * lo + near * y
    out[:, :, 1::2] = near * y + (1 - near) * hi
    return out


def store64(y, pad):
    """pad 0: y [B, C, D, H, W]; pad 1: a replicated 1-voxel border on D, H and W; pad 2: depth_x2 and a replicated
    border on H and W."""
    if pad == 0:
        return y
    if pad == 1:
        return np.pad(y, ((0, 0), (0, 0), (1, 1), (1, 1), (1, 1)), mode="edge")
    assert pad == 2
    return np.pad(depth_x2(y), ((0, 0), (0, 0), (0, 0), (1, 1), (1, 1)), mode="edge")


# ---- the seeded module the kernel tests pack ---------------------------------------------------------------------
def seeded_cva(seed):
    """A cva stage with seeded conv weights and BatchNorm statistics away from the identity (eval mode, on the CPU)."""
    import torch
    import dcanet_b200 as d
    torch.manual_seed(seed)
    m = d.cva(192, 32)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm3d):
            mod.weight.data.uniform_(0.75, 1.25)
            mod.bias.data.normal_(0, 0.1)
            mod.running_mean.normal_(0, 0.1)
            mod.running_var.uniform_(0.5, 1.5)
        if isinstance(mod, (torch.nn.Conv3d, torch.nn.ConvTranspose3d)):
            mod.weight.data.normal_(0, (2.0 / (mod.weight[0].numel())) ** 0.5)
    return m.eval()
