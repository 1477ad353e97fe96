"""fp64 restatements of the confidence maps and the sparsification tables -- TEST INFRASTRUCTURE.

  confidence                  peak / std of dca_softmax_confidence_upsample (include/dca_b200.h section 4) from the same
                              fp32 logits and mask, in float64
  prop_mask                   the prop net's mask logits, channels-last [B,H,W,144], computed with the oracle's own conv
                              and BN primitives (the two lines at the top of oracle.convex_upsample)
  confidence_histograms       the tables of dca_confidence_histograms, integer-exact (fp32 error, as the kernel)
  sparsification_bruteforce   sparsification curves by sorting the pixels (numpy)
"""
import numpy as np
import torch
import torch.nn.functional as F

import _eval_restatement as E


def confidence_quarter(logits):
    """logits [B,D,H,W] -> (peak_q, std_q) [B,H,W] float64: max_d p and sqrt(sum_d p (d - mu)^2), p = softmax_d."""
    lg = torch.as_tensor(logits).double()
    p = F.softmax(lg, dim=1)
    d = torch.arange(lg.shape[1], dtype=torch.float64).view(1, -1, 1, 1)
    mu = (p * d).sum(dim=1, keepdim=True)
    return p.max(dim=1).values, ((p * (d - mu) ** 2).sum(dim=1)).sqrt()


def convex_up(mask, v):
    """mask channels-last [B,H,W,144] (c = n*16 + i*4 + j), v [B,H,W] -> [B,1,4H,4W] float64: the 9-neighbour softmax
    blend of convex_upsample_kernel, zero outside the image."""
    m = torch.as_tensor(mask).double()
    B, H, W, _ = m.shape
    m = F.softmax(m.view(B, H, W, 9, 4, 4), dim=3)
    vp = F.pad(torch.as_tensor(v).double(), (1, 1, 1, 1))
    out = torch.zeros(B, H, W, 4, 4, dtype=torch.float64)
    for n in range(9):
        dy, dx = n // 3, n % 3
        out += m[:, :, :, n] * vp[:, dy:dy + H, dx:dx + W, None, None]
    return out.permute(0, 1, 3, 2, 4).reshape(B, 1, 4 * H, 4 * W)


def confidence(logits, mask):
    """-> (peak_q [B,H,W], std_q [B,H,W], peak [B,1,4H,4W], std [B,1,4H,4W]), float64."""
    pq, sq = confidence_quarter(logits)
    return pq, sq, convex_up(mask, pq), convex_up(mask, 4.0 * sq)


def prop_mask(sd, g):
    """PropgationNet_4x.conv (gwcnet_dca_g.py:112-115) on the guidance features g [B,64,H,W] with the oracle's
    primitives -> fp32 channels-last [B,H,W,144], the layout the kernels read."""
    from oracle import dcanet_oracle as O
    ctx = O._Ctx(sd)
    m = ctx.bn(ctx.conv2d(g, "prop.conv.0.0.weight"), "prop.conv.0.1")
    m = ctx.conv2d(F.relu(m), "prop.conv.2.weight")
    return m.permute(0, 2, 3, 1).contiguous()


CONF_BINS, ERR_BINS = 256, 2049


def confidence_histograms(pred, gt, peak, max_valid):
    """(conf_hist [256,2], err_hist [2049,2]) int64 over the pixels of SUM_ABS (valid GT, finite prediction): fixed-point
    |E| as _eval_restatement.disparity_metric_counts, conf bin min(floor(peak * 256), 255) (non-finite or negative: 0),
    error bin min(F >> 15, 2048)."""
    p, g, c = E._np32(pred).ravel(), E._np32(gt).ravel(), E._np32(peak).ravel()
    keep = E.gt_valid_mask(g, max_valid) & np.isfinite(p)
    p, g, c = p[keep], g[keep], c[keep]
    with np.errstate(invalid="ignore", over="ignore"):
        e = np.abs(p - g)
        fix = np.rint(np.minimum(e, np.float32(2.0 ** 20)) * np.float32(2.0 ** 20)).astype(np.uint64)
        ok = np.isfinite(c) & (c >= 0)
        cb = np.where(ok, np.minimum(np.floor(np.where(ok, c, 0) * np.float32(256)), np.float32(255)), 0).astype(np.int64)
    eb = np.minimum(fix >> np.uint64(15), np.uint64(ERR_BINS - 1)).astype(np.int64)
    out = []
    for bins, nb in ((cb, CONF_BINS), (eb, ERR_BINS)):
        h = np.zeros((nb, 2), np.int64)
        np.add.at(h[:, 0], bins, 1)
        np.add.at(h[:, 1], bins, fix.astype(np.int64))
        out.append(h)
    return tuple(out)


def sparsification_bruteforce(err_px, conf, densities):
    """EPE of the round(N q) pixels with the highest conf (and with the lowest error: the oracle), by sorting."""
    err_px, conf = np.asarray(err_px, np.float64), np.asarray(conf, np.float64)
    n = err_px.size
    by_conf = err_px[np.argsort(-conf, kind="stable")]
    by_err = np.sort(err_px)
    curve, oracle = [], []
    for q in densities:
        k = int(round(n * q))
        curve.append(float(by_conf[:k].mean()))
        oracle.append(float(by_err[:k].mean()))
    return curve, oracle
