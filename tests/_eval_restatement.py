"""CPU restatement of the two evaluation kernels (dca_disparity_metrics, dca_class_confusion) -- TEST INFRASTRUCTURE.

Float32 numpy / torch restatements of the definitions in include/dca_b200.h (section 7), which follow the reference's
evaluation loop (main_dca.py `mytest` :143-232, utils/metrics.py:45-63).  The GPU tests compare the kernels against
these bit for bit; the CPU tests check them against the GwcNet metric formulas and drive evaluate_files with them.
Kept beside the tests rather than in oracle/, whose hot-path restatement is pinned on the reference fixtures.
"""
import numpy as np
import torch
import torch.nn.functional as F


def _np32(x):
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().numpy()
    return np.asarray(x, dtype=np.float32)


def gt_valid_mask(gt, max_valid):
    """isfinite(gt) & gt > 0 & (gt < max_valid unless max_valid <= 0), all in fp32."""
    g = _np32(gt)
    mv = np.float32(max_valid)
    with np.errstate(invalid="ignore"):
        return np.isfinite(g) & (g > 0) & ((mv <= 0) | (g < mv))


def disparity_metric_counts(pred, gt, max_valid):
    """The counters of dca_disparity_metrics, restated in fp32 numpy: pred / gt [B,H,W] (or [B,1,H,W]) ->
    int64 [B, 7] = (valid, sum_abs, gt1, gt2, gt3, d1, pred_nonfinite).  sum_abs is sum of
    rint(min(|pred - gt|, 2^20) * 2^20) over valid pixels with a finite prediction (exact in fp32: a power-of-two
    scaling, rounded half to even); a non-finite prediction counts in gt1..d1."""
    p, g = _np32(pred), _np32(gt)
    B = g.shape[0]
    p, g = p.reshape(B, -1), g.reshape(B, -1)
    valid = gt_valid_mask(g, max_valid)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        e = np.abs(p - g)
        bad = ~np.isfinite(p)
        fix = np.rint(np.minimum(e, np.float32(2.0 ** 20)) * np.float32(2.0 ** 20))
        d1 = (e > np.float32(3)) & (e / np.abs(g) > np.float32(0.05))
    out = np.zeros((B, 7), np.int64)
    for b in range(B):
        v, bb = valid[b], bad[b]
        out[b, 0] = v.sum()
        out[b, 1] = int(fix[b][v & ~bb].astype(np.uint64).sum(dtype=np.uint64))
        for j, t in enumerate((1, 2, 3)):
            out[b, 2 + j] = (v & (bb | (e[b] > np.float32(t)))).sum()
        out[b, 5] = (v & (bb | d1[b])).sum()
        out[b, 6] = (v & bb).sum()
    return out


def class_confusion(logits, gt, D8, max_valid):
    """The confusion matrix of dca_class_confusion: logits [B,D8,H8,W8], gt [B,8*H8,8*W8] -> int64 [D8,D8]
    (row = GT class, column = predicted class).  Predicted class = first argmax of the fp32 softmax (as class_stats);
    GT = F.interpolate(gt, scale_factor=1/8, mode='nearest'), class min(floor(g / 8 + 0.5), D8 - 1) of the valid pixels."""
    logits = torch.as_tensor(logits).float().cpu()
    k = F.softmax(logits, dim=1).argmax(dim=1).numpy()
    g8 = F.interpolate(torch.as_tensor(_np32(gt))[:, None], scale_factor=1 / 8, mode="nearest")[:, 0].numpy()
    assert g8.shape == k.shape, (g8.shape, k.shape)
    valid = gt_valid_mask(g8, max_valid)
    with np.errstate(invalid="ignore", over="ignore"):
        cls = np.minimum(np.floor(g8 * np.float32(0.125) + np.float32(0.5)), np.float32(D8 - 1))
    idx = cls[valid].astype(np.int64) * D8 + k[valid]
    return np.bincount(idx, minlength=D8 * D8).reshape(D8, D8).astype(np.int64)
