"""numpy restatement of the moving-object test (include/dca_b200.h section 16) -- TEST INFRASTRUCTURE.

  labels       dca_motion_labels: the same IEEE fp32 operations in the same order (numpy float32 with explicit
               rounding of every step), so the kernel must match it bit for bit
  components   dca_motion_components: scipy.sparse.csgraph.connected_components on the gated 4-neighbour edge graph,
               numbered in raster order of each component's smallest pixel, object statistics in int64
"""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

F32 = np.float32
STATIC, APPEARED, BEHIND, UNSEEN, INVALID = 0, 1, 2, 3, 4
MAX_OBJECTS = 256
RES_CLAMP = F32(1048576.0)


def _row(m, a, b, c):
    return ((m[0] * a + m[1] * b) + m[2] * c) + m[3]


def _valid(z):
    with np.errstate(invalid="ignore"):
        return np.isfinite(z) & (z > 0)


def _disp(z, fB, doffs):
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        return (F32(fB) / z).astype(F32) - F32(doffs)


def backproject(H, W, z, intr, u0, v0):
    """p = ((((x + u0) - cx) z) / fx, (((y + v0) - cy) z) / fy, z), float32 [H,W] each."""
    fx, fy, cx, cy = (F32(v) for v in intr)
    y, x = np.meshgrid(np.arange(H, dtype=F32), np.arange(W, dtype=F32), indexing="ij")
    with np.errstate(invalid="ignore", over="ignore"):
        px = (((x + F32(u0)) - cx) * z) / fx
        py = (((y + F32(v0)) - cy) * z) / fy
    return px.astype(F32), py.astype(F32), z


def labels(depth, prev, intr, fB, doffs, u0, v0, A, tau=3.0, tau_rel=0.05, radius=1):
    """depth, prev float32 [B,H,W]; A float32 [B,12] -> (label uint8 [B,H,W], residual float32 [B,H,W])."""
    B, H, W = depth.shape
    fx, fy, cx, cy = (F32(v) for v in intr)
    tau, tau_rel = F32(tau), F32(tau_rel)
    lab = np.full((B, H, W), INVALID, np.uint8)
    res = np.full((B, H, W), np.nan, F32)
    for b in range(B):
        z = depth[b].astype(F32)
        ok = _valid(z)
        px, py, _ = backproject(H, W, z, intr, u0, v0)
        m = np.asarray(A[b], F32)
        with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
            qx, qy, qz = _row(m[0:4], px, py, z), _row(m[4:8], px, py, z), _row(m[8:12], px, py, z)
            seen = ok & (qz > 0)
            mx = (((fx * qx) / qz) + cx) - F32(u0)
            my = (((fy * qy) / qz) + cy) - F32(v0)
            xf, yf = np.floor(mx + F32(0.5)), np.floor(my + F32(0.5))
            inside = seen & (xf >= 0) & (xf < W) & (yf >= 0) & (yf < H)
        lab[b][ok] = UNSEEN
        ys, xs = np.nonzero(inside)
        xm, ym = xf[ys, xs].astype(np.int64), yf[ys, xs].astype(np.int64)
        e = _disp(qz[ys, xs], fB, doffs)
        with np.errstate(invalid="ignore", over="ignore"):
            tol = np.fmax(tau, (tau_rel * e).astype(F32))      # fmaxf: a NaN product gives tau
        n = len(ys)
        anyv = np.zeros(n, bool)
        stat = np.zeros(n, bool)
        appd = np.ones(n, bool)
        best = np.zeros(n, F32)
        dprev = _disp(prev[b].astype(F32), fB, doffs)
        vprev = _valid(prev[b])
        for dy in range(-radius, radius + 1):
            for dx in range(-radius, radius + 1):
                yy, xx = ym + dy, xm + dx
                inw = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
                yc, xc = np.clip(yy, 0, H - 1), np.clip(xx, 0, W - 1)
                v = inw & vprev[yc, xc]
                with np.errstate(invalid="ignore", over="ignore"):
                    s = (dprev[yc, xc] - e).astype(F32)
                    take = v & (~anyv | (np.abs(s) < np.abs(best)))
                    best = np.where(take, s, best)
                    anyv |= v
                    stat |= v & (np.abs(s) <= tol)
                    appd &= ~v | (s < -tol)
        l = np.where(stat, STATIC, np.where(appd, APPEARED, BEHIND)).astype(np.uint8)
        lab[b, ys[anyv], xs[anyv]] = l[anyv]
        res[b, ys[anyv], xs[anyv]] = best[anyv]
    return lab, res


def _key(f):
    i = np.asarray(f, F32).view(np.int32).astype(np.int64)
    return np.where(i >= 0, i, i ^ 0x7fffffff)


def _unkey(k):
    k = np.asarray(k, np.int64)
    return np.where(k >= 0, k, k ^ 0x7fffffff).astype(np.int32).view(F32)


def components(depth, label, residual, intr, fB, doffs, u0, v0, gate=1.0, min_pixels=100):
    """-> dict(instance int32 [B,H,W], count int32 [B], dropped int32 [B], ints int32 [B,MAX,8], extent float32
    [B,MAX,6], res_sum int64 [B,MAX]) as dca_motion_components writes them."""
    B, H, W = label.shape
    out = dict(instance=np.zeros((B, H, W), np.int32), count=np.zeros(B, np.int32), dropped=np.zeros(B, np.int32),
               ints=np.zeros((B, MAX_OBJECTS, 8), np.int32), extent=np.full((B, MAX_OBJECTS, 6), np.nan, F32),
               res_sum=np.zeros((B, MAX_OBJECTS), np.int64))
    gate = F32(gate)
    for b in range(B):
        z = depth[b].astype(F32)
        mov = (label[b] == APPEARED) | (label[b] == BEHIND)
        d = _disp(z, fB, doffs)
        idx = np.arange(H * W).reshape(H, W)
        rows, cols = [], []
        with np.errstate(invalid="ignore"):
            ex = mov[:, 1:] & mov[:, :-1] & (np.abs((d[:, 1:] - d[:, :-1]).astype(F32)) <= gate)
            ey = mov[1:, :] & mov[:-1, :] & (np.abs((d[1:, :] - d[:-1, :]).astype(F32)) <= gate)
        rows += [idx[:, 1:][ex], idx[1:, :][ey]]
        cols += [idx[:, :-1][ex], idx[:-1, :][ey]]
        r, c = np.concatenate(rows), np.concatenate(cols)
        g = coo_matrix((np.ones(len(r), np.int8), (r, c)), shape=(H * W, H * W))
        _, comp = connected_components(g, directed=False)
        flat = mov.ravel()
        pix = np.nonzero(flat)[0]
        cid = comp[pix]
        # the root of each component: its smallest pixel; components in raster order of their roots
        roots, first, sizes = np.unique(cid, return_index=True, return_counts=True)
        root_pix = pix[first]
        order = np.argsort(root_pix, kind="stable")
        kept = [roots[i] for i in order if sizes[i] >= min_pixels]
        K = min(len(kept), MAX_OBJECTS)
        out["count"][b], out["dropped"][b] = K, len(kept) - K
        ident = np.zeros(comp.max() + 1, np.int32)
        ident[np.array(kept[:K], np.int64)] = np.arange(1, K + 1, dtype=np.int32)
        inst = ident[cid]
        out["instance"][b].ravel()[pix] = inst
        px, py, _ = backproject(H, W, z, intr, u0, v0)
        lab = label[b].ravel()
        res = residual[b].ravel()
        for k in range(K):
            sel = pix[inst == k + 1]
            ys, xs = sel // W, sel % W
            out["ints"][b, k] = (len(sel), int((lab[sel] == APPEARED).sum()), int((lab[sel] == BEHIND).sum()),
                                 xs.min(), ys.min(), xs.max(), ys.max(), 0)
            ext = []
            for a in (px.ravel()[sel], py.ravel()[sel], z.ravel()[sel]):
                kk = _key(a)
                ext += [kk.min(), kk.max()]
            out["extent"][b, k] = _unkey(np.array(ext))
            rr = np.clip(res[sel], -RES_CLAMP, RES_CLAMP).astype(F32)
            out["res_sum"][b, k] = int(np.rint((rr * F32(256)).astype(F32)).astype(np.int64).sum())
    return out
