"""float32 / float64 numpy restatement of the LiDAR guidance (include/dca_b200.h section 14) -- TEST INFRASTRUCTURE.

  fma32          the correctly rounded fp32 fused multiply-add (an exact float64 product, TwoSum, and the one tie the
                 double rounding can break)
  lidar_hints    dca_lidar_hints: the same fp32 operations in the same order (z-buffer included), so the kernel must
                 match it bit for bit
  quarter        dca_guide_quarter (exact)
  factor         the modulation factor k exp(-(d - hq)^2 s) per (b, d, h, w) in float64, 1 where hq <= 0
  camera_points  synthetic velodyne scans: points spread over a camera's view, moved into the velodyne frame
  guided_hot_path  the oracle's forward from feature maps with the guided volume (float64 factor)
"""
import numpy as np

F32 = np.float32


def fma32(a, b, c):
    """fmaf(a, b, c) for float32 arrays: round(a b + c) once."""
    a, b, c = (np.asarray(x, F32).astype(np.float64) for x in (a, b, c))
    p = a * b                                   # exact: 24 + 24 significand bits
    r = p + c
    bb = r - p
    e = (p - (r - bb)) + (c - bb)               # TwoSum: r + e == p + c exactly
    r32 = r.astype(F32)
    d = r - r32.astype(np.float64)
    nxt = np.nextafter(r32, np.where(d > 0, F32(np.inf), F32(-np.inf)).astype(F32))
    half = (nxt.astype(np.float64) - r32.astype(np.float64)) / 2
    # r itself is the exact midpoint between two fp32 values only when d == half; then e decides the side
    fix = (d != 0) & (d == half) & (np.sign(e) == np.sign(d))
    return np.where(fix, nxt, r32).astype(F32)


def transform(M, pts):
    """X_i = fmaf(M_i2, z, fmaf(M_i1, y, fmaf(M_i0, x, M_i3))) per row i -> float32 [N, 3]."""
    M = np.asarray(M, F32).reshape(3, 4)
    x, y, z = (np.asarray(pts[:, i], F32) for i in range(3))
    return np.stack([fma32(M[i, 2], z, fma32(M[i, 1], y, fma32(M[i, 0], x, M[i, 3]))) for i in range(3)], -1)


def lidar_hints(scans, M, fx, fy, cx, cy, fB, doffs, H, W, window=None, view="left", min_depth=1.0, max_depth=80.0):
    """-> float32 [B, H, W] of dca_lidar_hints; fx .. doffs are rounded to float32 as the C ABI does."""
    fx, fy, cx, cy, fB, doffs = (F32(v) for v in (fx, fy, cx, cy, fB, doffs))
    y0, x0, h, w, vo = (0, 0, H, W, 0) if window is None else window
    out = np.zeros((len(scans), H, W), F32)
    for b, pts in enumerate(scans):
        pts = np.asarray(pts, F32)
        X, Y, Z = transform(M, pts).T
        with np.errstate(all="ignore"):
            keep = (Z >= F32(min_depth)) & (Z <= F32(max_depth))
            u = (fx * X) / Z + cx
            v = (fy * Y) / Z + cy
            disp = fB / Z - doffs
            if view == "right":
                u = u - disp
            fu, fv = np.floor(u + F32(0.5)), np.floor(v + F32(0.5))
            keep &= (fu >= F32(x0)) & (fu < F32(x0 + w)) & (fv >= F32(vo)) & (fv < F32(vo + h))
        idx = np.flatnonzero(keep)
        rows = y0 + (fv[idx].astype(np.int64) - vo)
        cols = fu[idx].astype(np.int64)
        pix = rows * W + cols
        order = np.lexsort((idx, Z[idx], pix))          # per pixel: smallest Z, then smallest point index
        pix, win = pix[order], idx[order]
        first = np.ones(len(pix), bool)
        first[1:] = pix[1:] != pix[:-1]
        zw = Z[win[first]]
        out[b].reshape(-1)[pix[first]] = fB / zw - doffs
    return out


def quarter(hints, maxdisp):
    """[B, H, W] -> [B, H/4, W/4]: the largest valid hint (finite, 0 < h < maxdisp) of each 4x4 block, times 0.25."""
    h = np.asarray(hints, F32)
    B, H, W = h.shape
    with np.errstate(invalid="ignore"):
        v = np.where(np.isfinite(h) & (h > 0) & (h < F32(maxdisp)), h, F32(0))
    return (v.reshape(B, H // 4, 4, W // 4, 4).max(axis=(2, 4)) * F32(0.25)).astype(F32)


def factor(hq, D, k, s):
    """float64 [B, D, H, W]: k exp(-(d - hq)^2 s) where hq > 0, else 1."""
    hq = np.asarray(hq, np.float64)[:, None]
    d = np.arange(D, dtype=np.float64)[None, :, None, None]
    return np.where(hq > 0, k * np.exp(-((d - hq) ** 2) * s), 1.0)


def camera_points(seed, n, fx, fy, cx, cy, W, H, rect_to_velo, zmin=2.0, zmax=60.0):
    """n points spread over a W x H view (rectified cam-2 frame, depths in [zmin, zmax]), moved into the velodyne frame
    with rect_to_velo (float64) -> float32 [n, 4] with a reflectance column."""
    rng = np.random.default_rng(seed)
    u = rng.uniform(-20, W + 20, n)
    v = rng.uniform(-20, H + 20, n)
    Z = rng.uniform(zmin, zmax, n)
    P = np.stack([(u - cx) * Z / fx, (v - cy) * Z / fy, Z, np.ones(n)], -1)
    T = np.vstack([np.asarray(rect_to_velo, np.float64).reshape(3, 4), [0, 0, 0, 1]])
    V = P @ T.T
    return np.hstack([V[:, :3], rng.uniform(0, 1, (n, 1))]).astype(F32)


def guided_hot_path(sd, gwc_l, gwc_r, cat_l, cat_r, g, maxdisp, hq, k, s, num_groups=40, collect=None):
    """oracle.dcanet_oracle.hot_path (3 cva stages) with the guided volume: every channel of plane d at a 1/4-res pixel
    with hq > 0 multiplied by k exp(-(d - hq)^2 s) in float64 (torch [B,H,W] hq), the rest of the path the oracle's own
    functions, in the oracle's order."""
    import torch
    import torch.nn.functional as F
    from oracle import dcanet_oracle as O
    ctx = O._Ctx(sd, None, False)
    D4 = maxdisp // 4
    vol = torch.cat([O.build_gwc_volume(gwc_l, gwc_r, D4, num_groups), O.build_concat_volume(cat_l, cat_r, D4)], dim=1)
    f = torch.from_numpy(factor(hq.numpy(), D4, k, s))[:, None]                        # [B,1,D,H,W]
    vol = (vol.double() * f).to(vol.dtype)
    c = ctx.convbn3d(vol, "dres0.0", 1, 1, "relu")
    c = ctx.convbn3d(c, "dres0.2", 1, 1, "relu")
    r = ctx.convbn3d(c, "dres1.0", 1, 1, "relu")
    cost0 = ctx.convbn3d(r, "dres1.2", 1, 1, None) + c
    cur, pvs = cost0, []
    for i in range(3):
        pv, out = O.cva_forward(ctx, f"cva{i + 1}", cur, collect)
        cur = cost0 + out if i == 0 else out
        pvs.append(pv)
    h = ctx.convbn3d(cur, "classif3.0", 1, 1, "relu")
    logits = ctx.conv3d(h, "classif3.2.weight", 1, 1).squeeze(1)
    pred_q = O.disparity_regression(F.softmax(logits, dim=1), D4)
    return O.convex_upsample(ctx, "prop", g, pred_q), pvs[1].squeeze(1)
