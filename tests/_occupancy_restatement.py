"""numpy restatement of the occupancy-grid update (include/dca_b200.h section 17) -- TEST INFRASTRUCTURE.

  integrate   dca_occupancy_integrate: the same IEEE fp32 operations in the same order (numpy float32, every step
              rounded), integer sums in int64 (they stay below 2^31 in the kernel), so the kernel must match it bit for
              bit; log_odds / updates are updated in place
"""
import numpy as np

F32 = np.float32


def _row(m, a, b, c):
    return ((m[0] * a + m[1] * b) + m[2] * c) + m[3]


def nbins(max_depth, range_res):
    return int(np.floor(F32(max_depth) / F32(range_res))) + 1


def integrate(log_odds, updates, origin, cs, depth, M, Minv, intr, u0=0, v0=0, weight=None, camera_height=1.65,
              band=(0.3, 2.5), col_width=5, range_res=0.1, max_depth=40.0, min_hits=10, l_hit=0.85, l_miss=-0.4,
              l_min=-2.0, l_max=3.5, box=None):
    """log_odds float32 / updates int32 [ny,nx] updated in place; depth (weight) float32 [B,H,W]; M, Minv float32
    [B,12] (grid <- camera, camera <- grid); box (i0, j0, bi, bj) or None (the whole grid).  Returns the per-frame
    intermediates (hits [B,bj,bi], occ [B,ncols,nbins], near, far, first [B,ncols]; near / far -1 when empty)."""
    ny, nx = log_odds.shape
    i0, j0, bi, bj = box if box is not None else (0, 0, nx, ny)
    ox, oy, cs = F32(origin[0]), F32(origin[1]), F32(cs)
    fx, fy, cx, cy = (F32(v) for v in intr)
    fu0, fv0 = F32(u0), F32(v0)
    h_lo, h_hi = F32(band[0]), F32(band[1])
    rr, md = F32(range_res), F32(max_depth)
    l_hit, l_miss, l_min, l_max = F32(l_hit), F32(l_miss), F32(l_min), F32(l_max)
    depth = np.asarray(depth, F32)
    B, H, W = depth.shape
    M = np.asarray(M, F32).reshape(B, 12)
    Minv = np.asarray(Minv, F32).reshape(B, 12)
    road = (M[:, 11] - F32(camera_height)).astype(F32)
    nb = nbins(max_depth, range_res)
    ncols = (W + col_width - 1) // col_width
    thr = 256 * int(min_hits)
    hits = np.zeros((B, bj, bi), np.int64)
    occ = np.zeros((B, ncols, nb), np.int64)
    near = np.full((B, ncols), -1, np.int64)
    far = np.full((B, ncols), -1, np.int64)
    first = np.full((B, ncols), nb, np.int64)
    y, x = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    xf32, yf32 = x.astype(F32), y.astype(F32)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        for b in range(B):
            z = depth[b]
            ok = np.isfinite(z) & (z > 0) & (z <= md)
            if weight is None:
                w = np.ones_like(z)
            else:
                wm = np.asarray(weight, F32)[b]
                w = np.where(np.isnan(wm), F32(0), np.minimum(np.maximum(wm, F32(0)), F32(1))).astype(F32)
            ok &= w > 0
            px = (((xf32 + fu0) - cx) * z) / fx
            py = (((yf32 + fv0) - cy) * z) / fy
            m = M[b]
            h = _row(m[8:12], px, py, z) - road[b]
            ok &= h <= h_hi
            obst = ok & (h >= h_lo)
            q = np.rint(F32(256) * w).astype(np.int64)
            c = x // col_width
            k = np.floor(np.where(ok, z, 0) / rr).astype(np.int64)
            gx, gy = _row(m[0:4], px, py, z), _row(m[4:8], px, py, z)
            fi = np.floor(((gx - ox) / cs) + F32(0.5))
            fj = np.floor(((gy - oy) / cs) + F32(0.5))
            inbox = obst & (fi >= i0) & (fi < i0 + bi) & (fj >= j0) & (fj < j0 + bj)
            ii = np.where(inbox, fi, i0).astype(np.int64) - i0
            jj = np.where(inbox, fj, j0).astype(np.int64) - j0
            np.add.at(hits[b], (jj[inbox], ii[inbox]), q[inbox])
            np.add.at(occ[b], (c[obst], k[obst]), q[obst])
            np.maximum.at(far[b], c[ok], k[ok])
            nr = np.full(ncols, nb, np.int64)
            np.minimum.at(nr, c[ok], k[ok])
            near[b] = np.where(nr < nb, nr, -1)
            above = occ[b] >= thr
            first[b] = np.where(above.any(1), above.argmax(1), nb)
        # cells
        jg, ig = np.meshgrid(np.arange(j0, j0 + bj), np.arange(i0, i0 + bi), indexing="ij")
        sx = ox + cs * ig.astype(F32)
        sy = oy + cs * jg.astype(F32)
        L = log_odds[j0:j0 + bj, i0:i0 + bi].copy()
        n = updates[j0:j0 + bj, i0:i0 + bi].astype(np.int64)
        for b in range(B):
            mi = Minv[b]
            sz = road[b]
            occd = hits[b] >= thr
            Zc = _row(mi[8:12], sx, sy, sz)
            Xc, Yc = _row(mi[0:4], sx, sy, sz), _row(mi[4:8], sx, sy, sz)
            xx = ((fx * Xc) / Zc + cx) - fu0
            yy = ((fy * Yc) / Zc + cy) - fv0
            xf, yf = np.floor(xx + F32(0.5)), np.floor(yy + F32(0.5))
            kf = np.floor(Zc / rr)
            seen = (Zc > 0) & (xf >= 0) & (xf < F32(W)) & (yf >= 0) & (yf < F32(H)) & (kf < F32(nb))
            col = np.where(seen, xf, 0).astype(np.int64) // col_width
            kk = np.where(seen, kf, 0).astype(np.int64)
            nr, fr, fs = near[b][col], far[b][col], first[b][col]
            free = ~occd & seen & (fr >= 0) & (nr <= kk) & (kk < fs) & (kk <= fr)
            L = np.where(occd, np.minimum(L + l_hit, l_max), L)
            L = np.where(free, np.maximum(L + l_miss, l_min), L).astype(F32)
            n = n + (occd | free)
        log_odds[j0:j0 + bj, i0:i0 + bi] = L
        updates[j0:j0 + bj, i0:i0 + bi] = n.astype(np.int32)
    return dict(hits=hits, occ=occ, near=near, far=far, first=first)
