"""float32 numpy restatement of the left-right consistency check and background fill (include/dca_b200.h section 8) --
TEST INFRASTRUCTURE.

  lr_check     (label uint8, filled float32) of dca_lr_consistency from D_L and D_R [..., W] in their own views: the same
               IEEE fp32 operations in the same order, so the kernel must match it bit for bit
  scene        a background plane with a nearer box in front of it, seen from both cameras: integer disparities, and the
               labels the geometry implies
"""
import numpy as np

CONSISTENT, OCCLUDED, MISMATCH, OUT_OF_VIEW = 0, 1, 2, 3


def lr_check(disp_left, disp_right, tau=1.0):
    dl = np.ascontiguousarray(np.asarray(disp_left, np.float32))
    dr = np.ascontiguousarray(np.asarray(disp_right, np.float32))
    W = dl.shape[-1]
    tau = np.float32(tau)
    with np.errstate(invalid="ignore", over="ignore"):
        xr = np.arange(W, dtype=np.float32) - dl
        inview = (xr >= np.float32(0)) & (xr <= np.float32(W - 1))
        xs = np.where(inview, xr, np.float32(0))
        x0f = np.floor(xs)
        x0 = x0f.astype(np.int64)
        r0 = np.take_along_axis(dr, x0, -1)
        r1 = np.take_along_axis(dr, np.minimum(x0 + 1, W - 1), -1)
        v = np.where(x0 == W - 1, r0, r0 + (xs - x0f) * (r1 - r0))
        label = np.full(dl.shape, MISMATCH, np.uint8)
        label[(v - dl) > tau] = OCCLUDED
        label[np.abs(dl - v) <= tau] = CONSISTENT
        label[~inview] = OUT_OF_VIEW
    return label, background_fill(dl, label)


def background_fill(dl, label):
    """Consistent pixels keep D_L; the others take min(D_L[l], D_L[r]) of the nearest consistent pixels l < x < r on the
    row, the one that exists, or D_L when the row has none."""
    W = dl.shape[-1]
    idx = np.broadcast_to(np.arange(W), dl.shape)
    cons = label == CONSISTENT
    left = np.maximum.accumulate(np.where(cons, idx, -1), axis=-1)
    right = np.minimum.accumulate(np.where(cons, idx, W)[..., ::-1], axis=-1)[..., ::-1]
    vl = np.take_along_axis(dl, np.clip(left, 0, W - 1), -1)
    vr = np.take_along_axis(dl, np.clip(right, 0, W - 1), -1)
    has_l, has_r = left >= 0, right < W
    with np.errstate(invalid="ignore"):
        f = np.where(has_l & has_r, np.minimum(vl, vr), np.where(has_l, vl, np.where(has_r, vr, dl)))
    return np.where(cons, dl, f).astype(np.float32)


def scene(H, W, a, b, d_b, d_f):
    """Background plane at disparity d_b, a box over columns [a, b) at d_f > d_b (integers, a >= d_f, b - a > d_f - d_b,
    b <= W).  Returns D_L, D_R [H, W] float32 and the expected labels: OCCLUDED on [a - (d_f - d_b), a), OUT_OF_VIEW
    for x < d_b, CONSISTENT elsewhere (for any tau < d_f - d_b)."""
    assert a >= d_f > d_b >= 0 and b - a > d_f - d_b and b <= W
    x = np.arange(W)
    dl = np.where((x >= a) & (x < b), d_f, d_b).astype(np.float32)
    dr = np.where((x >= a - d_f) & (x < b - d_f), d_f, d_b).astype(np.float32)     # box seen at x - d_f
    want = np.full(W, CONSISTENT, np.uint8)
    want[a - (d_f - d_b):a] = OCCLUDED
    want[:d_b] = OUT_OF_VIEW
    tile = lambda r: np.ascontiguousarray(np.broadcast_to(r, (H, W)))
    return tile(dl), tile(dr), tile(want)
