"""numpy restatement of include/dca_b200.h section 15 (ground profile, stixels, render), int64 throughout once the
disparity is quantised; the fp64 solve of the ground line in the kernel's operation order.  The GPU tests compare the
kernels with it bit for bit; the host tests check the model's properties with it."""
import itertools

import numpy as np

A_MIN, A_STEP, NA = np.float32(1 / 64), np.float32(1 / 256), 253
GROUND, OBJECT, SKY = 0, 1, 2
MIN_SLOPE = 0.0625
BIG = np.int64(1) << 60


def valid_pixels(disp, peak=None, label=None, min_peak=0.0, max_disp=192):
    """disp fp32 [B,H,W] -> (valid bool, d fp32 with 0 where invalid)."""
    d = np.asarray(disp, np.float32)
    with np.errstate(invalid="ignore"):
        ok = (d >= 0) & (d < np.float32(max_disp))
        if peak is not None:
            ok &= np.asarray(peak, np.float32) >= np.float32(min_peak)
    if label is not None:
        ok &= np.asarray(label) == 0
    return ok, np.where(ok, d, np.float32(0))


def quantise(d):
    return np.rint(np.asarray(d, np.float32) * np.float32(256)).astype(np.int64)


def ground_profile(disp, peak=None, label=None, min_peak=0.0, max_disp=192, min_inliers=1000, details=False):
    """-> (profile fp32 [B,H], line fp64 [B,2], inliers int64 [B], ok bool [B]) (+ the Hough winners (i, j) [B,2])."""
    ok_px, d = valid_pixels(disp, peak, label, min_peak, max_disp)
    B, H, W = d.shape
    D = int(max_disp)
    a = (A_MIN + np.arange(NA, dtype=np.float32) * A_STEP).astype(np.float64)         # exact
    t = np.arange(H, dtype=np.float64)
    R = np.minimum(np.rint(a[:, None] * t[None, :]).astype(np.int64), D + 1)           # [NA, H] by y - j
    prof = np.zeros((B, H), np.float32)
    line = np.zeros((B, 2), np.float64)
    inl = np.zeros(B, np.int64)
    good = np.zeros(B, bool)
    win = np.zeros((B, 2), np.int64)
    ys = np.broadcast_to(np.arange(H)[:, None], (H, W))
    for b in range(B):
        hist = np.zeros((H, D), np.int64)
        fd = d[b].astype(np.int64)
        np.add.at(hist, (ys[ok_px[b]], fd[ok_px[b]]), 1)
        h3 = np.zeros((H, D + 2), np.int64)                 # h3[y, r] = hist[r-1] + hist[r] + hist[r+1], r <= D
        h3[:, :D] += hist
        h3[:, 1:D + 1] += hist
        h3[:, :D - 1] += hist[:, 1:]
        scores = np.zeros((NA, H), np.int64)
        for j in range(H - 1):
            tt = np.arange(1, H - j)
            scores[:, j] = h3[j + tt[None, :], R[:, tt]].sum(axis=1)
        i, j = np.unravel_index(int(np.argmax(scores)), scores.shape)      # first maximum: smallest i, then j
        win[b] = i, j
        r = np.rint(a[i] * (ys - j)).astype(np.int64)
        sel = ok_px[b] & (ys > j) & (np.abs(fd - r) <= 1)
        yy = ys[sel].astype(np.int64)
        q = quantise(d[b][sel])
        n, Sy, Syy, Sq, Syq = len(yy), int(yy.sum()), int((yy * yy).sum()), int(q.sum()), int((q * yy).sum())
        N, Y, YY, Q, YQ = (np.float64(v) for v in (n, Sy, Syy, Sq, Syq))
        with np.errstate(all="ignore"):
            den = N * YY - Y * Y
            alpha = (N * YQ - Y * Q) / den
            beta = (Q - alpha * Y) / N
            ag = alpha * np.float64(1 / 256)
            yh = (-beta) / alpha
        g = bool(n >= min_inliers and den > 0 and ag >= MIN_SLOPE and np.isfinite(yh))
        inl[b], good[b] = n, g
        if g:
            line[b] = ag, yh
            tt = np.arange(H, dtype=np.float64) - yh
            prof[b] = np.where(tt > 0, (ag * tt).astype(np.float32), np.float32(0))
    out = (prof, line, inl, good)
    return out + (win,) if details else out


def cost(r, s, tau):
    r = np.abs(np.asarray(r, np.int64))
    return np.where(r >= tau * s, tau * tau * 1024, (r * r * 1024) // (s * s))


def column_samples(disp, peak=None, label=None, min_peak=0.0, max_disp=192, width=5):
    """-> int64 [B, ncols, H] by n = H - 1 - y: the lower median of each row's valid q, -1 for none."""
    ok_px, d = valid_pixels(disp, peak, label, min_peak, max_disp)
    B, H, W = d.shape
    ncols = -(-W // width)
    q = np.where(ok_px, quantise(d), BIG)
    pad = np.full((B, H, ncols * width), BIG, np.int64)
    pad[:, :, :W] = q
    s = np.sort(pad.reshape(B, H, ncols, width), axis=-1)
    m = (s < BIG).sum(-1)
    med = np.take_along_axis(s, np.maximum(m - 1, 0)[..., None] // 2, -1)[..., 0]
    med = np.where(m > 0, med, -1)
    return med[:, ::-1, :].transpose(0, 2, 1).copy()


def quantise_profile(profile, max_disp):
    p = np.asarray(profile, np.float32)
    with np.errstate(invalid="ignore"):
        ok = np.isfinite(p) & (p > 0)
    v = np.minimum(np.where(ok, p, np.float32(0)), np.float32(max_disp)) * np.float32(256)
    return np.where(ok, np.rint(v), 0).astype(np.int64)


DEFAULTS = dict(s_ground=256, s_object=512, s_sky=512, tau=3, p_seg=16384, p_gravity=8192, p_order=8192,
                eps_gravity=512, eps_order=256)


def dp(samples, g, max_disp, s_ground, s_object, s_sky, tau, p_seg, p_gravity, p_order, eps_gravity, eps_order,
       chunk=64):
    """samples int64 [M, H] (by n, -1 = invalid), g int64 [M, H] (by n) -> (C [M,H,3], BP [M,H,3], DM [M,H]) with
    C = BIG for unreachable states; vectorised over the columns and n_b."""
    M, H = samples.shape
    C = np.full((M, H, 3), BIG, np.int64)
    BP = np.zeros((M, H, 3), np.int64)
    DM = np.zeros((M, H), np.int64)
    for c0 in range(0, M, chunk):
        sl = slice(c0, min(c0 + chunk, M))
        _dp_chunk(samples[sl], g[sl], max_disp, s_ground, s_object, s_sky, tau, p_seg, p_gravity, p_order,
                  eps_gravity, eps_order, C[sl], BP[sl], DM[sl])
    return C, BP, DM


def _prefix(v):
    out = np.zeros(v.shape[:-1] + (v.shape[-1] + 1,), np.int64)
    out[..., 1:] = np.cumsum(v, axis=-1)
    return out


def _dp_chunk(q, g, D, s_g, s_o, s_s, tau, p_seg, p_grav, p_ord, eps_g, eps_o, C, BP, DM):
    M, H = q.shape
    valid = q >= 0
    qv = np.where(valid, q, 0)
    PV, PQ = _prefix(valid.astype(np.int64)), _prefix(qv)
    PG = _prefix(np.where(valid, cost(qv - g, s_g, tau), 0))
    PS = _prefix(np.where(valid, cost(qv, s_s, tau), 0))
    PZ = _prefix((g <= 0).astype(np.int64))
    lvl = np.arange(D + 1, dtype=np.int64)
    lut = _prefix(np.where(valid[:, None, :], cost(qv[:, None, :] - 256 * lvl[None, :, None], s_o, tau), 0))
    rows = np.arange(M)[:, None]
    for nt in range(H):
        nb = np.arange(nt + 1)
        key = nb[None, :] * 4
        first = (nb == 0)[None, :]
        prevC = np.zeros((M, nt + 1, 3), np.int64)
        prevC[:, 1:] = C[:, :nt]
        prevC[:, 0] = BIG
        prev_dm = np.zeros((M, nt + 1), np.int64)
        prev_dm[:, 1:] = DM[:, :nt]
        reach = prevC < BIG
        cands = []                          # (class, cost, key) candidate arrays [M, nt+1]
        # ground
        okg = PZ[:, nt + 1, None] == PZ[:, nb]
        dg = PG[:, nt + 1, None] - PG[:, nb] + p_seg
        cands.append((GROUND, np.where(okg & first, dg, BIG), key))
        cands.append((GROUND, np.where(okg & reach[..., OBJECT], prevC[..., OBJECT] + dg, BIG), key + OBJECT))
        # object
        cnt = PV[:, nt + 1, None] - PV[:, nb]
        S = PQ[:, nt + 1, None] - PQ[:, nb]
        m = (2 * S + cnt) // np.maximum(2 * cnt, 1)
        lv = np.minimum((m + 128) >> 8, D)
        do = lut[rows, lv, nt + 1] - lut[rows, lv, nb[None, :]] + p_seg
        has = cnt > 0
        grav = np.where(np.abs(m - g[:, nb]) > eps_g, p_grav, 0)
        order = np.where(m > prev_dm + eps_o, p_ord, 0)
        cands.append((OBJECT, np.where(has & first, do, BIG), key))
        cands.append((OBJECT, np.where(has & reach[..., GROUND], prevC[..., GROUND] + do + grav, BIG), key + GROUND))
        cands.append((OBJECT, np.where(has & reach[..., OBJECT], prevC[..., OBJECT] + do + order, BIG), key + OBJECT))
        # sky
        ds = PS[:, nt + 1, None] - PS[:, nb] + p_seg
        cands.append((SKY, np.where(first, ds, BIG), key))
        cands.append((SKY, np.where(reach[..., GROUND], prevC[..., GROUND] + ds, BIG), key + GROUND))
        cands.append((SKY, np.where(reach[..., OBJECT], prevC[..., OBJECT] + ds, BIG), key + OBJECT))
        for c in (GROUND, OBJECT, SKY):
            cc = [(cst, np.broadcast_to(k, cst.shape)) for cl, cst, k in cands if cl == c]
            cst = np.concatenate([a for a, _ in cc], axis=1)
            kk = np.concatenate([b for _, b in cc], axis=1)
            order_key = np.where(cst < BIG, (cst << 16) | kk, BIG << 2)
            best = np.argmin(order_key, axis=1)
            bc = cst[np.arange(M), best]
            C[:, nt, c] = bc
            BP[:, nt, c] = np.where(bc < BIG, kk[np.arange(M), best], 0)
            if c == OBJECT:
                bnb = BP[:, nt, c] >> 2
                mm = m[np.arange(M), np.minimum(bnb, nt)]
                DM[:, nt] = np.where(bc < BIG, mm, 0)


def backtrack(C, BP, DM, H):
    """-> list per column of segments (n_b, n_t, class, m) from the bottom up."""
    out = []
    for col in range(C.shape[0]):
        c = int(np.argmin(C[col, H - 1]))            # first minimum: ground < object < sky
        segs = []
        nt = H - 1
        while nt >= 0:
            key = int(BP[col, nt, c])
            nb = key >> 2
            segs.append((nb, nt, c, int(DM[col, nt]) if c == OBJECT else 0))
            c = key & 3
            nt = nb - 1
        out.append(segs[::-1])
    return out


def stixels(disp, profile, peak=None, label=None, min_peak=0.0, width=5, max_disp=192, **priors):
    """-> dict of count [B,ncols], bottom / top / cls [B,ncols,H] (-1 past count), disp fp32 (m / 256), free_space,
    and segs (the per-column lists of backtrack) and energy [B,ncols]."""
    pr = dict(DEFAULTS, **priors)
    samp = column_samples(disp, peak, label, min_peak, max_disp, width)
    B, ncols, H = samp.shape
    g = quantise_profile(profile, max_disp)[:, ::-1]                     # by n
    gcol = np.repeat(g[:, None, :], ncols, axis=1).reshape(B * ncols, H)
    C, BP, DM = dp(samp.reshape(B * ncols, H), gcol, max_disp, **pr)
    segs = backtrack(C, BP, DM, H)
    count = np.zeros((B, ncols), np.int64)
    bottom = np.full((B, ncols, H), -1, np.int64)
    top = np.full((B, ncols, H), -1, np.int64)
    cls = np.full((B, ncols, H), -1, np.int64)
    sd = np.zeros((B, ncols, H), np.float32)
    free = np.full((B, ncols), H, np.int64)
    for idx, sg in enumerate(segs):
        b, k = divmod(idx, ncols)
        count[b, k] = len(sg)
        for i, (nb, nt, c, m) in enumerate(sg):
            bottom[b, k, i], top[b, k, i], cls[b, k, i] = H - 1 - nb, H - 1 - nt, c
            sd[b, k, i] = np.float32(m) / np.float32(256) if c == OBJECT else 0
        if sg[0][2] == GROUND:
            free[b, k] = H - 1 - sg[0][1]
    energy = C[:, H - 1].min(axis=1).reshape(B, ncols)
    return dict(count=count, bottom=bottom, top=top, cls=cls, disp=sd, free_space=free, segs=segs, energy=energy,
                samples=samp)


def render(st, profile, W, width):
    count, bottom, top, cls, sd = st["count"], st["bottom"], st["top"], st["cls"], st["disp"]
    B, ncols, H = bottom.shape
    out = np.zeros((B, H, W), np.float32)
    oc = np.full((B, H, W), SKY, np.uint8)
    prof = np.asarray(profile, np.float32)
    for b in range(B):
        for k in range(ncols):
            x0, x1 = k * width, min((k + 1) * width, W)
            for i in range(count[b, k]):
                t, bt, c = top[b, k, i], bottom[b, k, i], cls[b, k, i]
                oc[b, t:bt + 1, x0:x1] = c
                v = prof[b, t:bt + 1, None] if c == GROUND else (sd[b, k, i] if c == OBJECT else 0)
                out[b, t:bt + 1, x0:x1] = v
    return out, oc


# ---- exhaustive check of the DP --------------------------------------------------------------------------------
def segmentation_energy(q, g, segs, max_disp, s_ground, s_object, s_sky, tau, p_seg, p_gravity, p_order, eps_gravity,
                        eps_order):
    """The exact energy of one segmentation [(n_b, n_t, c)] of a column (q, g by n), or None when it is forbidden."""
    valid = q >= 0
    e, prev = 0, None
    for nb, nt, c in segs:
        rows = slice(nb, nt + 1)
        qq = q[rows][valid[rows]]
        if c == GROUND:
            if (g[rows] <= 0).any() or (prev is not None and prev[0] != OBJECT):
                return None
            e += int(cost(qq - g[rows][valid[rows]], s_ground, tau).sum())
            m = None
        elif c == OBJECT:
            if len(qq) == 0 or (prev is not None and prev[0] == SKY):
                return None
            m = (2 * int(qq.sum()) + len(qq)) // (2 * len(qq))
            lv = min((m + 128) >> 8, max_disp)
            e += int(cost(qq - 256 * lv, s_object, tau).sum())
            if prev is not None and prev[0] == GROUND and abs(m - int(g[nb])) > eps_gravity:
                e += p_gravity
            if prev is not None and prev[0] == OBJECT and m > prev[1] + eps_order:
                e += p_order
        else:
            if prev is not None and prev[0] == SKY:
                return None
            e += int(cost(qq, s_sky, tau).sum())
            m = None
        e += p_seg
        prev = (c, m)
    return e


def all_segmentations(H):
    for cuts in itertools.product((0, 1), repeat=H - 1):
        bounds = [0] + [i + 1 for i, c in enumerate(cuts) if c] + [H]
        spans = [(bounds[i], bounds[i + 1] - 1) for i in range(len(bounds) - 1)]
        for labels in itertools.product((GROUND, OBJECT, SKY), repeat=len(spans)):
            yield [(nb, nt, c) for (nb, nt), c in zip(spans, labels)]


# ---- synthetic scenes ------------------------------------------------------------------------------------------
KITTI = dict(fx=721.5377, fy=721.5377, cx=609.5593, cy=172.854, baseline=0.5327)
# (left column, right column, camera depth Z in m, height in m): fronto-parallel boxes standing on the road
BOXES = ((100, 260, 8.0, 1.5), (400, 520, 15.0, 1.8), (700, 800, 22.0, 1.5), (900, 980, 30.0, 2.5),
         (1050, 1110, 38.0, 1.6))


def driving_scene(seed=0, H=375, W=1242, cam_height=1.65, pitch_deg=1.0, wall_z=60.0, wall_height=10.0, noise=0.3,
                  outliers=0.05, invalid=0.10, boxes=BOXES, road=True):
    """A flat road seen from a camera cam_height above it and pitched down by pitch_deg, boxes on the road, a far wall
    and sky (disparity 0), with uniform +-noise px, a fraction of uniform outliers in [0, 100) px and a fraction of
    invalid pixels (NaN, -1, +inf).  The road's disparity is exactly a (y - y_h) with a = fx B cos(pitch) / (fy h) and
    y_h = cy - fy tan(pitch).  road=False extends the far wall down to the bottom edge (no ground).  -> (disp float32 [H,W], info)"""
    rng = np.random.default_rng(seed)
    fx, fy, cy, B = KITTI["fx"], KITTI["fy"], KITTI["cy"], KITTI["baseline"]
    th = np.deg2rad(pitch_deg)
    a = fx * B * np.cos(th) / (fy * cam_height)
    yh = cy - fy * np.tan(th)
    fB = fx * B
    y = np.arange(H, dtype=np.float64)[:, None] * np.ones((1, W))
    d = np.zeros((H, W))                                            # sky
    dw = fB / wall_z
    wall_foot = yh + dw / a
    wall_top = wall_foot - wall_height * fy / wall_z
    d[(y >= wall_top) & (y <= wall_foot)] = dw
    if road:
        d = np.where(y > wall_foot, a * (y - yh), d)
    else:
        d = np.where(y > wall_foot, dw, d)
    info = dict(a=a, yh=yh, wall_foot=wall_foot, wall_top=wall_top, wall_disp=dw, boxes=[])
    for u0, u1, z, hb in boxes:
        db = fB / z
        foot = int(np.floor(yh + db / a))
        top = int(np.ceil(foot - hb * fy / z))
        d[top:foot + 1, u0:u1 + 1] = db
        info["boxes"].append(dict(u0=u0, u1=u1, disp=db, foot=foot, top=top))
    d = d + rng.uniform(-noise, noise, d.shape)
    out = rng.random(d.shape) < outliers
    d[out] = rng.uniform(0, 100, int(out.sum()))
    bad = rng.random(d.shape) < invalid
    d[bad] = rng.choice(np.array([np.nan, -1.0, np.inf]), int(bad.sum()))
    return d.astype(np.float32), info
