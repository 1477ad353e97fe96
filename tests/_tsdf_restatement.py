"""float32 numpy restatement of TSDF fusion and surface extraction (include/dca_b200.h section 12) -- TEST
INFRASTRUCTURE.

  integrate   dca_tsdf_integrate: the same IEEE fp32 operations in the same order, frame after frame, so the kernel must
              match it bit for bit
  surface     dca_tsdf_count_surface + dca_tsdf_extract_surface: (xyz, normal, rgb) of every crossing, ordered by voxel
              then axis
  new_state   a fresh state [planes, nz, ny, nx]
"""
import numpy as np

F32 = np.float32


def new_state(dims, colour=True):
    nx, ny, nz = dims
    s = np.zeros((5 if colour else 2, nz, ny, nx), F32)
    s[0] = 1
    return s


def _row(m, a, b, c):
    return ((m[0] * a + m[1] * b) + m[2] * c) + m[3]


def _centres(origin, vs, i, j, k):
    o = [F32(v) for v in origin]
    vs = F32(vs)
    return o[0] + vs * i.astype(F32), o[1] + vs * j.astype(F32), o[2] + vs * k.astype(F32)


def integrate(state, origin, vs, depth, T, intrinsics, u0=0, v0=0, weight=None, rgb=None, trunc=0.3,
              max_weight=np.inf, max_depth=np.inf, box=None):
    """state float32 [planes, nz, ny, nx] updated in place and returned; depth (weight) float32 [B,H,W], rgb uint8
    [B,H,W,3|4] (required iff planes = 5), T float32 [B,12] world-to-camera, box (i0, j0, k0, bi, bj, bk) or None."""
    P, nz, ny, nx = state.shape
    i0, j0, k0, bi, bj, bk = box if box is not None else (0, 0, 0, nx, ny, nz)
    k, j, i = (a.ravel() for a in np.meshgrid(np.arange(k0, k0 + bk), np.arange(j0, j0 + bj), np.arange(i0, i0 + bi),
                                              indexing="ij"))
    px, py, pz = _centres(origin, vs, i, j, k)
    fx, fy, cx, cy = (F32(v) for v in intrinsics)
    fu0, fv0 = F32(u0), F32(v0)
    trunc, max_weight, max_depth = F32(trunc), F32(max_weight), F32(max_depth)
    depth = np.asarray(depth, F32)
    B, H, W = depth.shape
    T = np.asarray(T, F32).reshape(B, 12)
    Tv = state[0, k, j, i].copy()
    Wv = state[1, k, j, i].copy()
    C = [state[2 + c, k, j, i].copy() for c in range(3)] if P == 5 else []
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        for b in range(B):
            m = T[b]
            Zc = _row(m[8:12], px, py, pz)
            ok = Zc > 0
            Xc, Yc = _row(m[0:4], px, py, pz), _row(m[4:8], px, py, pz)
            x = ((fx * Xc) / Zc + cx) - fu0
            y = ((fy * Yc) / Zc + cy) - fv0
            xf, yf = np.floor(x + F32(0.5)), np.floor(y + F32(0.5))
            ok &= (xf >= 0) & (xf < F32(W)) & (yf >= 0) & (yf < F32(H))
            xi = np.where(ok, xf, 0).astype(np.int64)
            yi = np.where(ok, yf, 0).astype(np.int64)
            z = depth[b, yi, xi]
            ok &= np.isfinite(z) & (z > 0) & (z <= max_depth)
            if weight is None:
                w = np.ones_like(z)
            else:
                wm = np.asarray(weight, F32)[b, yi, xi]
                w = np.where(np.isnan(wm), F32(0), np.minimum(np.maximum(wm, F32(0)), F32(1))).astype(F32)
            ok &= w > 0
            sdf = z - Zc
            ok &= ~(sdf < -trunc)
            f = np.minimum(F32(1), sdf / trunc)
            Wn = Wv + w
            Tv = np.where(ok, ((Tv * Wv) + (f * w)) / Wn, Tv).astype(F32)
            if P == 5:
                for c in range(3):
                    q = np.asarray(rgb)[b, yi, xi, c].astype(F32)
                    C[c] = np.where(ok, ((C[c] * Wv) + (q * w)) / Wn, C[c]).astype(F32)
            Wv = np.where(ok, np.minimum(Wn, max_weight), Wv).astype(F32)
    state[0, k, j, i] = Tv
    state[1, k, j, i] = Wv
    for c in range(len(C)):
        state[2 + c, k, j, i] = C[c]
    return state


def crossings(state, min_weight):
    """bool [nz, ny, nx, 3]: the crossing of each voxel along x, y, z."""
    T, Wt = state[0], state[1]
    mw = F32(min_weight)
    ok = Wt >= mw
    neg = T < 0
    m = np.zeros(T.shape + (3,), bool)
    for a, ax in enumerate((2, 1, 0)):
        n = T.shape[ax]
        sl_v = [slice(None)] * 3
        sl_n = [slice(None)] * 3
        sl_v[ax], sl_n[ax] = slice(0, n - 1), slice(1, n)
        sl_v, sl_n = tuple(sl_v), tuple(sl_n)
        m[sl_v + (a,)] = ok[sl_v] & ok[sl_n] & (neg[sl_v] != neg[sl_n])
    return m


def surface(state, origin, vs, min_weight=0.5, normals=True, colours=True):
    """-> (xyz float32 [n,3], normal float32 [n,3] or None, rgb uint8 [n,3] or None) of dca_tsdf_extract_surface."""
    P, nz, ny, nx = state.shape
    T = state[0]
    flat = np.flatnonzero(crossings(state, min_weight))
    v, a = flat // 3, flat % 3
    i, j, k = v % nx, (v // nx) % ny, v // (nx * ny)
    step = np.array([1, nx, nx * ny])[a]
    Tf = T.ravel()
    Tv, Tn = Tf[v], Tf[v + step]
    with np.errstate(invalid="ignore", divide="ignore"):
        t = Tv / (Tv - Tn)
    p = np.stack(_centres(origin, vs, i, j, k), -1)
    xyz = p.copy()
    xyz[np.arange(len(v)), a] = p[np.arange(len(v)), a] + t * F32(vs)
    normal = None
    if normals:
        ip, im = np.minimum(i + 1, nx - 1), np.maximum(i - 1, 0)
        jp, jm = np.minimum(j + 1, ny - 1), np.maximum(j - 1, 0)
        kp, km = np.minimum(k + 1, nz - 1), np.maximum(k - 1, 0)
        g = np.stack([T[k, j, ip] - T[k, j, im], T[k, jp, i] - T[k, jm, i], T[kp, j, i] - T[km, j, i]], -1)
        ln = np.sqrt((g[:, 0] * g[:, 0] + g[:, 1] * g[:, 1]) + g[:, 2] * g[:, 2])
        with np.errstate(invalid="ignore", divide="ignore"):
            normal = np.where((ln > 0)[:, None], g / ln[:, None], F32(0)).astype(F32)
    rgb = None
    if colours:
        out = []
        for c in range(3):
            Cf = state[2 + c].ravel()
            cv, cn = Cf[v], Cf[v + step]
            out.append(np.clip(np.rint(cv + t * (cn - cv)), 0, 255))
        rgb = np.stack(out, -1).astype(np.uint8)
    return xyz.astype(F32), normal, rgb
