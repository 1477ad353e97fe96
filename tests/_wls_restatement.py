"""Float32 numpy restatement of dca_wls_filter (include/dca_b200.h section 11) in the kernels' exact operation order,
its float64 reference (scipy.linalg.solve_banded on every line), the host weight table and a synthetic scene.  Test
infrastructure only."""
import numpy as np

f32 = np.float32
LUT_SIZE = 3 * 255 * 255 + 1
K = 64                             # DCA_WLS_SEGMENT
CONSISTENT = 0


def lut(sigma, dtype=np.float32):
    k = np.arange(LUT_SIZE, dtype=np.float64)
    return np.exp(-np.sqrt(k) / float(sigma)).astype(dtype)


def schedule(lam, T):
    lam64 = float(f32(lam))
    return [f32(((lam64 * 1.5) * 4.0 ** (T - t)) / (4.0 ** T - 1.0)) for t in range(1, T + 1)]


def start(disp, peak=None, label=None, dtype=np.float32):
    """(c, U, V) of step 1-2: disp / peak / label [B,H,W]."""
    d = np.asarray(disp, np.float32)
    if peak is None:
        c = np.ones(d.shape, np.float32)
    else:
        p = np.asarray(peak, np.float32)
        c = np.where(np.isnan(p), f32(0), np.minimum(np.maximum(p, f32(0)), f32(1))).astype(np.float32)
    if label is not None:
        c = np.where(np.asarray(label) == CONSISTENT, c, f32(0))
    c = np.where(np.isfinite(d) & (c > 0), c, f32(0)).astype(np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        U = np.where(c > 0, c.astype(dtype) * d.astype(dtype), 0).astype(dtype)
    return c.astype(dtype), U, c.astype(dtype)


def weights(guide, table):
    """(wh, wv) [B,H,W]: weight to the right / lower neighbour, 0 at the last column / row."""
    g = np.asarray(guide)[..., :3].astype(np.int64)
    B, H, W, _ = g.shape
    wh = np.zeros((B, H, W), table.dtype)
    wv = np.zeros((B, H, W), table.dtype)
    wh[:, :, :-1] = table[((g[:, :, 1:] - g[:, :, :-1]) ** 2).sum(-1)]
    wv[:, :-1, :] = table[((g[:, 1:] - g[:, :-1]) ** 2).sum(-1)]
    return wh, wv


def segments(n):
    """[(a, c)] of a line of n elements: separators at K-1, 2K-1, ... <= n-2 (K = DCA_WLS_SEGMENT)."""
    S = (n - 1) // K + 1
    return [(s * K, (s + 1) * K - 1 if s + 1 < S else n) for s in range(S)]


def _thomas(f_u, f_v, e, b, eL, a, c):
    """THOMAS of the segment [a, c) of every line: forward from e_{a-1} = eL, backward from u_c = 0."""
    one = f32(1)
    L = e.shape[0]
    P = np.empty((L, c - a), np.float32)
    GU = np.empty((L, c - a), np.float32)
    GV = np.empty((L, c - a), np.float32)
    ep, pp = eL, np.zeros(L, np.float32)
    gu = np.zeros(L, np.float32)
    gv = np.zeros(L, np.float32)
    for k, i in enumerate(range(a, c)):
        m = one / (b[:, i] - ep * pp)
        gu = (f_u[:, k] + ep * gu) * m
        gv = (f_v[:, k] + ep * gv) * m
        pp = e[:, i] * m
        ep = e[:, i]
        P[:, k], GU[:, k], GV[:, k] = pp, gu, gv
    u = np.zeros(L, np.float32)
    v = np.zeros(L, np.float32)
    U = np.empty((L, c - a), np.float32)
    V = np.empty((L, c - a), np.float32)
    for k in range(c - a - 1, -1, -1):
        u = GU[:, k] + P[:, k] * u
        v = GV[:, k] + P[:, k] * v
        U[:, k], V[:, k] = u, v
    return U, V


def thomas(f_u, f_v, w, lam):
    """Solve every line of [L, n] arrays (the axis of the recurrence last) by the partitioned solve of
    include/dca_b200.h section 11, in the kernels' order."""
    L, n = w.shape
    one = f32(1)
    zero = np.zeros(L, np.float32)
    e = lam * w
    b = (one + np.concatenate([zero[:, None], e[:, :-1]], 1)) + e
    segs = segments(n)
    S = len(segs)
    U = np.empty((L, n), np.float32)
    V = np.empty((L, n), np.float32)
    if S == 1:
        U[:], V[:] = _thomas(f_u, f_v, e, b, zero, 0, n)
        return U, V
    bd = []                                   # boundary values of each segment
    for a, c in segs:
        eL = e[:, a - 1] if a > 0 else zero
        eR = e[:, c - 1]
        ep, pp = eL, zero
        gu = gv = gphi = zero
        for i in range(a, c):
            m = one / (b[:, i] - ep * pp)
            gu = (f_u[:, i] + ep * gu) * m
            gv = (f_v[:, i] + ep * gv) * m
            gphi = eL * m if i == a else (ep * gphi) * m
            pp = e[:, i] * m
            ep = e[:, i]
        rn = hu = hv = hpsi = zero
        for i in range(c - 1, a - 1, -1):
            em = e[:, i - 1] if i > 0 else zero
            q = one / (b[:, i] - e[:, i] * rn)
            hu = (f_u[:, i] + e[:, i] * hu) * q
            hv = (f_v[:, i] + e[:, i] * hv) * q
            hpsi = eR * q if i == c - 1 else (e[:, i] * hpsi) * q
            rn = em * q
        bd.append(dict(yU_f=hu, yV_f=hv, phi_f=eL * q, psi_f=hpsi, yU_l=gu, yV_l=gv, phi_l=gphi, psi_l=eR * m))
    P, GU, GV = [], [], []
    pp = gU = gV = zero
    for s in range(S - 1):
        c = segs[s][1]
        em, ec = e[:, c - 1], e[:, c]
        lo = em * bd[s]["phi_l"]
        up = ec * bd[s + 1]["psi_f"]
        D = (b[:, c] - em * bd[s]["psi_l"]) - ec * bd[s + 1]["phi_f"]
        rU = (f_u[:, c] + em * bd[s]["yU_l"]) + ec * bd[s + 1]["yU_f"]
        rV = (f_v[:, c] + em * bd[s]["yV_l"]) + ec * bd[s + 1]["yV_f"]
        m = one / (D - lo * pp)
        pp = up * m
        gU = (rU + lo * gU) * m
        gV = (rV + lo * gV) * m
        P.append(pp), GU.append(gU), GV.append(gV)
    xU, xV = [None] * (S - 1), [None] * (S - 1)
    u = v = zero
    for s in range(S - 2, -1, -1):
        u = GU[s] + P[s] * u
        v = GV[s] + P[s] * v
        xU[s], xV[s] = u, v
        U[:, segs[s][1]], V[:, segs[s][1]] = u, v
    for s, (a, c) in enumerate(segs):
        eL = e[:, a - 1] if a > 0 else zero
        fu, fv = f_u[:, a:c].copy(), f_v[:, a:c].copy()
        if a > 0:
            fu[:, 0] = fu[:, 0] + eL * xU[s - 1]
            fv[:, 0] = fv[:, 0] + eL * xV[s - 1]
        if c < n:
            fu[:, -1] = fu[:, -1] + e[:, c - 1] * xU[s]
            fv[:, -1] = fv[:, -1] + e[:, c - 1] * xV[s]
        U[:, a:c], V[:, a:c] = _thomas(fu, fv, e, b, eL, a, c)
    return U, V


def wls(disp, guide, peak=None, label=None, lam=8000.0, sigma=1.5, T=3, min_support=1e-3):
    """-> (refined, support) float32 [B,H,W], bit for bit what dca_wls_filter computes."""
    d = np.asarray(disp, np.float32)
    B, H, W = d.shape
    with np.errstate(over="ignore", invalid="ignore", divide="ignore", under="ignore"):
        _, U, V = start(d, peak, label)
        wh, wv = weights(guide, lut(sigma))
        for lt in schedule(lam, T):
            U, V = thomas(U.reshape(B * H, W), V.reshape(B * H, W), wh.reshape(B * H, W), lt)
            U, V = U.reshape(B, H, W), V.reshape(B, H, W)
            tr = lambda a: np.ascontiguousarray(a.transpose(0, 2, 1)).reshape(B * W, H)
            U, V = thomas(tr(U), tr(V), tr(wv), lt)
            U = U.reshape(B, W, H).transpose(0, 2, 1)
            V = V.reshape(B, W, H).transpose(0, 2, 1)
        ok = V >= f32(min_support)
        refined = np.where(ok, U / np.where(ok, V, f32(1)), d)
    return np.ascontiguousarray(refined, dtype=np.float32), np.ascontiguousarray(V, dtype=np.float32)


def wls64(disp, guide, peak=None, label=None, lam=8000.0, sigma=1.5, T=3):
    """Float64 reference: every line solved by scipy.linalg.solve_banded with the same lambda_t -> (U / V, V)."""
    from scipy.linalg import solve_banded
    d = np.asarray(disp, np.float32)
    B, H, W = d.shape
    _, U, V = start(d, peak, label, dtype=np.float64)
    wh, wv = weights(guide, lut(sigma, np.float64))

    def solve(F1, F2, w, lt):
        out1, out2 = np.empty_like(F1), np.empty_like(F2)
        lt = float(lt)
        for k in range(F1.shape[0]):
            e = lt * w[k]
            e[-1] = 0.0
            ab = np.zeros((3, len(e)))
            ab[0, 1:] = -e[:-1]
            ab[1] = 1.0 + e + np.concatenate([[0.0], e[:-1]])
            ab[2, :-1] = -e[:-1]
            sol = solve_banded((1, 1), ab, np.stack([F1[k], F2[k]], 1))
            out1[k], out2[k] = sol[:, 0], sol[:, 1]
        return out1, out2

    for lt in schedule(lam, T):
        U, V = solve(U.reshape(B * H, W), V.reshape(B * H, W), wh.reshape(B * H, W), lt)
        U, V = U.reshape(B, H, W), V.reshape(B, H, W)
        tr = lambda a: np.ascontiguousarray(a.transpose(0, 2, 1)).reshape(B * W, H)
        U, V = solve(tr(U), tr(V), tr(wv), lt)
        U = U.reshape(B, W, H).transpose(0, 2, 1)
        V = V.reshape(B, W, H).transpose(0, 2, 1)
    with np.errstate(invalid="ignore", divide="ignore"):
        return U / V, V


def scene(H, W, B=1, seed=0, confident=0.7, noise=0.5, blocks=(6, 10), slope=0.01):
    """Colour-block guide aligned with piecewise-planar disparities (tilts up to `slope` px per px) plus noise ->
    (guide uint8 [B,H,W,3], disp noisy float32 [B,H,W], clean float32 [B,H,W], peak float32 [B,H,W])."""
    rng = np.random.default_rng(seed)
    by, bx = blocks
    ys = np.sort(rng.choice(np.arange(1, H), min(by - 1, H - 1), replace=False)) if H > 1 else np.array([], int)
    xs = np.sort(rng.choice(np.arange(1, W), min(bx - 1, W - 1), replace=False)) if W > 1 else np.array([], int)
    ry = np.searchsorted(ys, np.arange(H), side="right")
    rx = np.searchsorted(xs, np.arange(W), side="right")
    region = ry[:, None] * (len(xs) + 1) + rx[None, :]
    n = region.max() + 1
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    guide = np.empty((B, H, W, 3), np.uint8)
    clean = np.empty((B, H, W), np.float32)
    for b in range(B):
        col = rng.integers(0, 256, (n, 3))
        plane = np.stack([rng.uniform(5, 80, n), rng.uniform(-slope, slope, n), rng.uniform(-slope, slope, n)], 1)
        guide[b] = col[region].astype(np.uint8)
        p = plane[region]
        clean[b] = (p[..., 0] + p[..., 1] * (xx - W / 2) + p[..., 2] * (yy - H / 2)).astype(np.float32)
    disp = (clean + rng.normal(0, noise, clean.shape)).astype(np.float32)
    peak = np.where(rng.random(clean.shape) < confident, rng.uniform(0.3, 1.0, clean.shape), 0.0).astype(np.float32)
    return guide, disp, clean, peak
