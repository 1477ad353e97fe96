"""float32 / float64 numpy restatement of the raycast and of ICP tracking (include/dca_b200.h section 13) -- TEST
INFRASTRUCTURE.

  raycast   dca_tsdf_raycast: the march, the hit, the normal and the colour with the same IEEE fp32 operations in the same
            order, so the kernel must match it bit for bit
  icp       dca_icp_track: every iteration's fixed-point sums (exact int64), the fp64 Cholesky solve and the pose update in
            Python floats (IEEE float64, correctly rounded), the stats and the ok flag
"""
import math

import numpy as np

F32 = np.float32
NAN = F32(np.nan)

TILE = 1024                          # DCA_ICP_TILE
WORKSPACE_ROW = 32                   # DCA_ICP_WORKSPACE_ROW
MAX_DEPTH = 256.0                    # DCA_ICP_MAX_DEPTH
MAX_GATE = 16.0                      # DCA_ICP_MAX_GATE
MAX_PIXELS = 1 << 24                 # DCA_ICP_MAX_PIXELS
MAX_NORMAL2 = F32(1.0625)            # DCA_ICP_MAX_NORMAL2
SCALE_H, SCALE_G, SCALE_E, SCALE_W = 2.0 ** 18, 2.0 ** 24, 2.0 ** 30, 2.0 ** 30
PIVOT_REL = 5e-5                     # DCA_ICP_PIVOT_REL
FEW_INLIERS, DEGENERATE = 1, 2


def _row(m, a, b, c):
    return ((m[0] * a + m[1] * b) + m[2] * c) + m[3]


def _lerp(p, q, t):
    return p + t * (q - p)


def _tri(plane, i, j, k, a, b, c):
    c00 = _lerp(plane[k, j, i], plane[k, j, i + 1], a)
    c10 = _lerp(plane[k, j + 1, i], plane[k, j + 1, i + 1], a)
    c01 = _lerp(plane[k + 1, j, i], plane[k + 1, j, i + 1], a)
    c11 = _lerp(plane[k + 1, j + 1, i], plane[k + 1, j + 1, i + 1], a)
    return _lerp(_lerp(c00, c10, b), _lerp(c01, c11, b), c)


def _clamped(plane, gx, gy, gz):
    nz, ny, nx = plane.shape
    g = []
    for v, n in ((gx, nx), (gy, ny), (gz, nz)):
        v = np.minimum(np.maximum(v, F32(0)), F32(n - 1))
        v0 = np.minimum(np.floor(v), F32(n - 2))
        g.append((v0.astype(np.int64), v - v0))
    (i, a), (j, b), (k, c) = g
    return _tri(plane, i, j, k, a, b, c)


def _grid(M, origin, vs, xn, yn, z):
    cx, cy = xn * z, yn * z
    o = [F32(v) for v in origin]
    return tuple((_row(M[4 * a:4 * a + 4], cx, cy, z) - o[a]) / vs for a in range(3))


def raycast(state, origin, vs, trunc, min_weight, intrinsics, u0, v0, H, W, cam_to_world, min_depth=0.0,
            max_depth=40.0):
    """-> depth float32 [H,W], vertex float32 [H,W,3], normal float32 [H,W,3], rgb uint8 [H,W,3] (None without colour)
    of dca_tsdf_raycast; cam_to_world float32 [12] (or [3,4])."""
    P, nz, ny, nx = state.shape
    T, Wt = state[0], state[1]
    vs, trunc, mw = F32(vs), F32(trunc), F32(min_weight)
    fx, fy, cx, cy = (F32(v) for v in intrinsics)
    M = np.asarray(cam_to_world, F32).reshape(12)
    y, x = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    x, y = x.ravel(), y.ravel()
    xn = ((x.astype(F32) + F32(u0)) - cx) / fx
    yn = ((y.astype(F32) + F32(v0)) - cy) / fy
    L = np.sqrt((xn * xn + yn * yn) + F32(1))
    half = F32(0.5) * vs
    n = x.size
    z = np.full(n, F32(min_depth), F32)
    zh = np.zeros(n, F32)
    have = np.zeros(n, bool)
    zp = np.zeros(n, F32)
    Tp = np.zeros(n, F32)
    act = np.flatnonzero(z <= F32(max_depth))
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        while act.size:
            za = z[act]
            gx, gy, gz = _grid(M, origin, vs, xn[act], yn[act], za)
            x0, y0, z0 = np.floor(gx), np.floor(gy), np.floor(gz)
            known = (x0 >= 0) & (x0 < F32(nx - 1)) & (y0 >= 0) & (y0 < F32(ny - 1)) & (z0 >= 0) & (z0 < F32(nz - 1))
            i = np.where(known, x0, 0).astype(np.int64)
            j = np.where(known, y0, 0).astype(np.int64)
            k = np.where(known, z0, 0).astype(np.int64)
            for dz in (0, 1):
                for dy in (0, 1):
                    for dx in (0, 1):
                        known &= Wt[k + dz, j + dy, i + dx] >= mw
            Ts = _tri(T, i, j, k, gx - x0, gy - y0, gz - z0)
            hv, tp = have[act], Tp[act]
            hit = known & hv & (tp >= 0) & (Ts < 0)
            back = known & hv & (tp < 0) & (Ts >= 0)
            zpa = zp[act]
            zh[act[hit]] = (zpa + (za - zpa) * (tp / (tp - Ts)))[hit]
            s = np.where(known, np.maximum(half, np.abs(Ts) * trunc), trunc).astype(F32)
            have[act] = known
            zp[act] = np.where(known, za, zpa)
            Tp[act] = np.where(known, Ts, tp)
            zn = za + s / L[act]
            go = ~hit & ~back & (zn > za) & (zn <= F32(max_depth))
            z[act] = zn
            act = act[go]
        hit = zh > 0
        depth = np.zeros(n, F32)
        vertex = np.full((n, 3), NAN, F32)
        normal = np.full((n, 3), NAN, F32)
        rgb = np.zeros((n, 3), np.uint8) if P == 5 else None
        h = np.flatnonzero(hit)
        if h.size:
            zz = zh[h]
            gx, gy, gz = _grid(M, origin, vs, xn[h], yn[h], zz)
            one = F32(1)
            ax = _clamped(T, gx + one, gy, gz) - _clamped(T, gx - one, gy, gz)
            ay = _clamped(T, gx, gy + one, gz) - _clamped(T, gx, gy - one, gz)
            az = _clamped(T, gx, gy, gz + one) - _clamped(T, gx, gy, gz - one)
            ln = np.sqrt((ax * ax + ay * ay) + az * az)
            ok = ln > 0
            h, zz, gx, gy, gz, ax, ay, az, ln = (a[ok] for a in (h, zz, gx, gy, gz, ax, ay, az, ln))
            wx, wy, wz = ax / ln, ay / ln, az / ln
            depth[h] = zz
            vertex[h] = np.stack([xn[h] * zz, yn[h] * zz, zz], -1)
            normal[h] = np.stack([(M[c] * wx + M[4 + c] * wy) + M[8 + c] * wz for c in range(3)], -1)
            if rgb is not None:
                rgb[h] = np.stack([np.clip(np.rint(_clamped(state[2 + c], gx, gy, gz)), 0, 255) for c in range(3)],
                                  -1).astype(np.uint8)
    return (depth.reshape(H, W), vertex.reshape(H, W, 3), normal.reshape(H, W, 3),
            None if rgb is None else rgb.reshape(H, W, 3))


def _sums(depth, weight, intr, u0, v0, max_depth, mvert, mnorm, A, stride, gate):
    """int64 [30]: the 21 + 6 + 3 fixed-point sums of one iteration (exact, so the order of the kernel's CTAs does not
    matter)."""
    H, W = depth.shape
    fx, fy, cx, cy = (F32(v) for v in intr)
    md = F32(max_depth)
    Q = F32(2) * md
    Af = np.array(A, np.float64).astype(F32)
    y, x = np.meshgrid(np.arange(0, H, stride), np.arange(0, W, stride), indexing="ij")
    x, y = x.ravel(), y.ravel()
    z = depth[y, x]
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        keep = np.isfinite(z) & (z > 0) & (z <= md)
        if weight is None:
            w = np.ones_like(z)
        else:
            wm = weight[y, x]
            w = np.where(np.isnan(wm), F32(0), np.minimum(np.maximum(wm, F32(0)), F32(1))).astype(F32)
        keep &= w > 0
        px = (((x.astype(F32) + F32(u0)) - cx) * z) / fx
        py = (((y.astype(F32) + F32(v0)) - cy) * z) / fy
        qx, qy, qz = _row(Af[0:4], px, py, z), _row(Af[4:8], px, py, z), _row(Af[8:12], px, py, z)
        keep &= (qz > 0) & (qz <= Q) & (np.abs(qx) <= Q) & (np.abs(qy) <= Q)
        mx = (((fx * qx) / qz) + cx) - F32(u0)
        my = (((fy * qy) / qz) + cy) - F32(v0)
        xf, yf = np.floor(mx + F32(0.5)), np.floor(my + F32(0.5))
        keep &= (xf >= 0) & (xf < F32(W)) & (yf >= 0) & (yf < F32(H))
        xi = np.where(keep, xf, 0).astype(np.int64)
        yi = np.where(keep, yf, 0).astype(np.int64)
        m, n = mvert[yi, xi], mnorm[yi, xi]
        nx, ny, nz = n[:, 0], n[:, 1], n[:, 2]
        keep &= ((nx * nx + ny * ny) + nz * nz) <= MAX_NORMAL2
        dx, dy, dz = qx - m[:, 0], qy - m[:, 1], qz - m[:, 2]
        g = F32(gate)
        keep &= ((dx * dx + dy * dy) + dz * dz) <= g * g
        k = np.flatnonzero(keep)
        w, qx, qy, qz, nx, ny, nz, dx, dy, dz = (a[k] for a in (w, qx, qy, qz, nx, ny, nz, dx, dy, dz))
        r = (nx * dx + ny * dy) + nz * dz
        J = [qy * nz - qz * ny, qz * nx - qx * nz, qx * ny - qy * nx, nx, ny, nz]

    def fixed(t, scale):
        return int(np.rint(t.astype(np.float64) * scale).astype(np.int64).sum())

    out = []
    for i in range(6):
        wj = w * J[i]
        for j in range(i, 6):
            out.append(fixed(wj * J[j], SCALE_H))
    for i in range(6):
        out.append(fixed((w * J[i]) * r, SCALE_G))
    out.append(fixed((w * r) * r, SCALE_E))
    out.append(fixed(w, SCALE_W))
    out.append(int(k.size))
    return out


def _solve(s, A, min_inliers):
    """One solve of dca_icp_track in Python floats -> (A', stats row, flag)."""
    count = s[29]
    H = [[0.0] * 6 for _ in range(6)]
    o = 0
    for i in range(6):
        for j in range(i, 6):
            H[i][j] = H[j][i] = float(s[o]) * (1.0 / SCALE_H)
            o += 1
    g = [float(s[21 + i]) * (1.0 / SCALE_G) for i in range(6)]
    E = float(s[27]) * (1.0 / SCALE_E)
    Sw = float(s[28]) * (1.0 / SCALE_W)
    flag = FEW_INLIERS if count < min_inliers else 0
    if not flag:
        thr = PIVOT_REL * max(H[i][i] for i in range(6))
        L = [[0.0] * 6 for _ in range(6)]
        for j in range(6):
            v = H[j][j]
            for k in range(j):
                v = v - L[j][k] * L[j][k]
            if not v > thr:
                flag = DEGENERATE
                break
            d = math.sqrt(v)
            L[j][j] = d
            for i in range(j + 1, 6):
                u = H[i][j]
                for k in range(j):
                    u = u - L[i][k] * L[j][k]
                L[i][j] = u / d
    if not flag:
        yv = [0.0] * 6
        xi = [0.0] * 6
        for i in range(6):
            u = -g[i]
            for k in range(i):
                u = u - L[i][k] * yv[k]
            yv[i] = u / L[i][i]
        for i in range(5, -1, -1):
            u = yv[i]
            for k in range(i + 1, 6):
                u = u - L[k][i] * xi[k]
            xi[i] = u / L[i][i]
        hx, hy, hz = xi[0] * 0.5, xi[1] * 0.5, xi[2] * 0.5
        nq = math.sqrt(((1.0 + hx * hx) + hy * hy) + hz * hz)
        qw, qx, qy, qz = 1.0 / nq, hx / nq, hy / nq, hz / nq
        xx, yy, zz = qx * qx, qy * qy, qz * qz
        xy, xz, yz = qx * qy, qx * qz, qy * qz
        wx, wy, wz = qw * qx, qw * qy, qw * qz
        R = [1.0 - 2.0 * (yy + zz), 2.0 * (xy - wz), 2.0 * (xz + wy),
             2.0 * (xy + wz), 1.0 - 2.0 * (xx + zz), 2.0 * (yz - wx),
             2.0 * (xz - wy), 2.0 * (yz + wx), 1.0 - 2.0 * (xx + yy)]
        An = []
        for i in range(3):
            for j in range(4):
                v = (R[3 * i] * A[j] + R[3 * i + 1] * A[4 + j]) + R[3 * i + 2] * A[8 + j]
                if j == 3:
                    v = v + xi[3 + i]
                An.append(v)
        A = An
    return A, [float(count), Sw, E, float(flag)], flag


def icp(depth, weight, intrinsics, u0, v0, max_depth, mvert, mnorm, A0, levels, min_inliers):
    """-> (pose float64 [12], stats float64 [iterations, 4], ok bool) of dca_icp_track.  depth, weight float32 [H,W];
    mvert, mnorm float32 [H,W,3]; A0 [3,4] or [12] float64; levels = ((stride, iterations, gate), ...)."""
    depth = np.asarray(depth, F32)
    weight = None if weight is None else np.asarray(weight, F32)
    A = [float(v) for v in np.asarray(A0, np.float64)[:3].reshape(12)] if np.asarray(A0).size != 12 else \
        [float(v) for v in np.asarray(A0, np.float64).reshape(12)]
    stats, ok = [], True
    for stride, iters, gate in levels:
        for _ in range(iters):
            s = _sums(depth, weight, intrinsics, u0, v0, max_depth, mvert, mnorm, A, stride, gate)
            A, row, flag = _solve(s, A, min_inliers)
            stats.append(row)
            ok = ok and flag == 0
    return np.array(A, np.float64), np.array(stats, np.float64), ok
