"""float32 numpy restatement of the reprojection (include/dca_b200.h section 9) and of the depth errors of
dca_depth_metrics (section 7) -- TEST INFRASTRUCTURE.

  reproject       (xyz, index, count, depth) of dca_reproject: the same IEEE fp32 operations in the same order, so the
                  kernel must match it bit for bit
  depth_metrics   the DCA_DEPTH_* rows, plus the per-pixel ln-ratio the log-error bound of the GPU test is computed from
  kitti_scene     a synthetic KITTI calibration (P2, P3, R0_rect, Tr_velo_to_cam) and its files in both key styles
"""
import numpy as np

from _eval_restatement import _np32, gt_valid_mask

CONSISTENT = 0
F32 = np.float32


def _row(m, a, b, c):
    return ((m[0] * a + m[1] * b) + m[2] * c) + m[3]


def keep_and_points(disp, peak, label, u0, v0, Q, T, min_peak, min_depth, max_depth):
    """Per-pixel (keep, P [..., 3], Z) over [B,H,W] maps."""
    d = _np32(disp)
    B, H, W = d.shape
    Q = np.asarray(Q, F32).reshape(4, 4)
    u = np.broadcast_to((np.arange(W) + u0).astype(F32), d.shape)
    v = np.broadcast_to((np.arange(H) + v0).astype(F32)[:, None], d.shape)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        w = _row(Q[3], u, v, d)
        X, Y, Z = (_row(Q[i], u, v, d) / w for i in range(3))
        keep = np.isfinite(d) & (w > 0) & (Z >= F32(min_depth)) & (Z <= F32(max_depth))
        if peak is not None:
            keep &= _np32(peak) >= F32(min_peak)
        if label is not None:
            keep &= np.asarray(label) == CONSISTENT
        if T is not None:
            T = np.asarray(T, F32).reshape(3, 4)
            P = np.stack([_row(T[i], X, Y, Z) for i in range(3)], -1)
        else:
            P = np.stack([X, Y, Z], -1)
    return keep, P.astype(F32), Z.astype(F32)


def reproject(disp, peak=None, label=None, u0=0, v0=0, Q=None, T=None, min_peak=0.0, min_depth=0.0,
              max_depth=np.inf):
    """-> (xyz list of [count_b, 3], index list of int32 [count_b], count int64 [B], depth float32 [B,H,W]); the points of
    image b are those of np.flatnonzero(keep[b]), in that order."""
    keep, P, Z = keep_and_points(disp, peak, label, u0, v0, Q, T, min_peak, min_depth, max_depth)
    B = keep.shape[0]
    xyz, index = [], []
    for b in range(B):
        idx = np.flatnonzero(keep[b])
        index.append(idx.astype(np.int32))
        xyz.append(P[b].reshape(-1, 3)[idx])
    depth = np.where(keep, Z, F32(0)).astype(F32)
    return xyz, index, np.array([len(i) for i in index], np.int64), depth


def _fix(v):
    with np.errstate(invalid="ignore", over="ignore"):
        return np.rint(np.fmin(v, F32(2.0 ** 20)) * F32(2.0 ** 20)).astype(np.uint64)


def depth_metrics(pred, gt, max_valid, fb, doffs, min_depth, max_depth):
    """-> (rows int64 [B, 8] of DCA_DEPTH_*, lg float32 [B, H*W] = ln Zp - ln Zg (0 off the scored pixels))."""
    p, g = _np32(pred), _np32(gt)
    B = g.shape[0]
    p, g = p.reshape(B, -1), g.reshape(B, -1)
    fb, doffs, lo, hi = F32(fb), F32(doffs), F32(min_depth), F32(max_depth)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        zg = fb / (g + doffs)
        m = gt_valid_mask(g, max_valid) & (zg >= lo) & (zg <= hi)
        pd = p + doffs
        zp = np.where(np.isfinite(pd) & (pd > 0), fb / pd, hi)
        zp = np.minimum(np.maximum(zp, lo), hi).astype(F32)
        e = zp - zg
        e2 = e * e
        lg = np.log(zp) - np.log(zg)
        ratio = np.maximum(zp / zg, zg / zp)
        terms = [np.abs(e) / zg, e2 / zg, e2, lg * lg]
    out = np.zeros((B, 8), np.int64)
    for b in range(B):
        mb = m[b]
        out[b, 0] = mb.sum()
        for j, t in enumerate(terms):
            out[b, 1 + j] = int(_fix(t[b][mb]).sum(dtype=np.uint64))
        for j, thr in enumerate((1.25, 1.5625, 1.953125)):
            out[b, 5 + j] = (mb & (ratio[b] < F32(thr))).sum()
    return out, np.where(m, lg, F32(0)).astype(F32)


# ---- a synthetic KITTI calibration ----------------------------------------------------------------------------
def _rot(ax, ay, az):
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def kitti_scene():
    """A KITTI-like rig in float64: K of the rectified colour cameras, P2 = K [I | t2], P3 = K [I | t3] with t2, t3
    differing in x only (camera 2 at +0.06 m, camera 3 at -0.47 m), a small R0_rect and a velodyne-to-camera rigid
    transform."""
    fx, fy, cx, cy = 721.5377, 721.5377, 609.5593, 172.854
    K = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1.0]])
    t2, t3 = np.array([0.0598, -0.0003, 0.0]), np.array([-0.4731, -0.0003, 0.0])    # rectified: x offsets differ
    P2 = K @ np.hstack([np.eye(3), t2[:, None]])
    P3 = K @ np.hstack([np.eye(3), t3[:, None]])
    R0 = _rot(0.004, -0.009, 0.0075)
    Rv = _rot(-np.pi / 2 + 0.01, 0.02, -np.pi / 2 - 0.005)
    tv = np.array([-0.004, -0.076, -0.27])
    V2C = np.hstack([Rv, tv[:, None]])
    return {"P2": P2, "P3": P3, "R0_rect": R0, "Tr_velo_to_cam": V2C, "fx": fx, "fy": fy, "cx": cx, "cy": cy,
            "t2": t2, "t3": t3, "Rv": Rv, "tv": tv}


def write_kitti_calib(path, s, style="object"):
    fmt = lambda a: " ".join("%.12e" % v for v in np.asarray(a).ravel())
    if style == "object":
        lines = ["P0: " + fmt(s["P2"]), "P1: " + fmt(s["P3"]), "P2: " + fmt(s["P2"]), "P3: " + fmt(s["P3"]),
                 "R0_rect: " + fmt(s["R0_rect"]), "Tr_velo_to_cam: " + fmt(s["Tr_velo_to_cam"]),
                 "Tr_imu_to_velo: " + fmt(np.eye(4)[:3])]
    else:                                   # stereo 2015 / raw calib_cam_to_cam.txt
        lines = ["calib_time: 09-Jan-2012 13:57:47", "corner_dist: 9.950000e-02",
                 "S_rect_02: 1.242000e+03 3.750000e+02", "R_rect_02: " + fmt(np.eye(3)),
                 "P_rect_02: " + fmt(s["P2"]), "P_rect_03: " + fmt(s["P3"])]
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
