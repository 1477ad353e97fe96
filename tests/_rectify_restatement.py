"""float32 numpy restatement of the rectification kernels (include/dca_b200.h section 10) -- TEST INFRASTRUCTURE.

  remap              (rgb, moments) of dca_rectify: the same IEEE fp32 operations in the same order, integer moments
  standardise_frame  (left, right) of dca_standardise_frame: mean, 128-bit-exact variance (Python ints), fp64 outputs
                     rounded once to fp32
  framing            the kernel's framing parameters and the reproject window, restated from kitti_io's fit_to_crop /
                     pad_to_multiple
  kitti_raw_rig      a KITTI-raw-like two-camera rig (distorted raw cameras, rectifying rotations, rectified P) and its
                     calib_cam_to_cam.txt with the real key layout
"""
import math

import numpy as np

F32 = np.float32


def remap(raw_left, raw_right, maps):
    """raw uint8 [B, Hs, Ws, C>=3] x2, maps float32 [2, H, W, 2] -> (rgb uint8 [B, 2, H, W, 3], moments int64
    [B, 2, 3, 2] of (sum q, sum q^2))."""
    maps = np.asarray(maps, F32)
    B = raw_left.shape[0]
    H, W = maps.shape[1:3]
    rgb = np.zeros((B, 2, H, W, 3), np.uint8)
    for v, raw in enumerate((raw_left, raw_right)):
        src = np.asarray(raw)[..., :3]
        Hs, Ws = src.shape[1:3]
        sx, sy = maps[v, ..., 0], maps[v, ..., 1]
        inside = (sx > F32(-1)) & (sx < F32(Ws)) & (sy > F32(-1)) & (sy < F32(Hs))       # NaN: False
        sx, sy = np.where(inside, sx, F32(-2)), np.where(inside, sy, F32(-2))
        fx, fy = np.floor(sx), np.floor(sy)
        x0, y0 = fx.astype(np.int64), fy.astype(np.int64)
        ax, ay = sx - fx, sy - fy
        wx0, wy0 = F32(1) - ax, F32(1) - ay

        def tap(yy, xx):
            ok = (yy >= 0) & (yy < Hs) & (xx >= 0) & (xx < Ws)
            g = src[:, np.clip(yy, 0, Hs - 1), np.clip(xx, 0, Ws - 1)].astype(F32)       # [B, H, W, 3]
            return np.where(ok[None, ..., None], g, F32(0))

        p00, p01, p10, p11 = tap(y0, x0), tap(y0, x0 + 1), tap(y0 + 1, x0), tap(y0 + 1, x0 + 1)
        e = lambda a: a[None, ..., None]
        top = e(wx0) * p00 + e(ax) * p01
        bot = e(wx0) * p10 + e(ax) * p11
        val = e(wy0) * top + e(ay) * bot
        assert val.dtype == F32
        rgb[:, v] = np.clip(np.rint(val), 0, 255).astype(np.uint8)
    q = rgb.astype(np.int64)
    moments = np.stack([q.sum(axis=(2, 3)), (q * q).sum(axis=(2, 3))], -1)               # [B, 2, 3, 2]
    return rgb, moments


def channel_stats(S, SS, N):
    """(mean, std) in fp64 by the header's definition: exact integer numerator, each fp64 operation rounded once."""
    S, SS, N = int(S), int(SS), int(N)
    mean = S / N                                    # Python int / int: correctly rounded
    var = float(N * SS - S * S) / (float(N) * float(N))
    return mean, math.sqrt(var)


def standardise(rgb, moments):
    """rgb uint8 [B, 2, H, W, 3] -> float32 [B, 2, 3, H, W] standardised images (no framing)."""
    B, _, H, W, _ = rgb.shape
    out = np.empty((B, 2, 3, H, W), F32)
    for b in range(B):
        for v in range(2):
            for c in range(3):
                mean, std = channel_stats(moments[b, v, c, 0], moments[b, v, c, 1], H * W)
                with np.errstate(invalid="ignore", divide="ignore"):        # a constant channel: 0 / 0 = NaN
                    lut = ((np.arange(256, dtype=np.float64) - mean) / np.float64(std)).astype(F32)
                out[b, v, c] = lut[rgb[b, v, :, :, c]]
    return out


def standardise_frame(rgb, moments, frame):
    """(left, right) float32 [B, 3, Hn, Wn] of dca_standardise_frame with frame = (Hn, Wn, dst_y0, src_y0, h, w)."""
    Hn, Wn, dst_y0, src_y0, h, w = frame
    s = standardise(rgb, moments)
    B = rgb.shape[0]
    out = np.zeros((B, 2, 3, Hn, Wn), F32)
    out[..., dst_y0:dst_y0 + h, :w] = s[..., src_y0:src_y0 + h, :w]
    return out[:, 0], out[:, 1]


def framing(H, W, mode, ch=384, cw=1248):
    """(frame, window) restated from kitti_io: fit_to_crop pads a smaller image at the top and right and crops a larger
    one around the row centre from column 0; pad_to_multiple(16) pads at the top and right."""
    if mode == "pad16":
        top, right = (-H) % 16, (-W) % 16
        return (H + top, W + right, top, 0, H, W), (top, 0, H, W, 0)
    if H <= ch and W <= cw:
        return (ch, cw, ch - H, 0, H, W), (ch - H, 0, H, W, 0)
    y = int((H - ch) / 2)
    return (ch, cw, 0, y, ch, cw), (0, 0, ch, cw, y)


# ---- a KITTI-raw-like rig ---------------------------------------------------------------------------------------
def _rot(ax, ay, az):
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def kitti_raw_rig(raw_size=(1392, 512), rect_size=(1242, 375)):
    """Cameras 00..03 in float64 with KITTI raw's magnitudes: raw K with distortion, rectifying rotations R_rect_0i,
    rectified projections P_rect_0i = K_rect [I | t_i] with t_i along x only."""
    Kr = np.array([[7.215377e2, 0, 6.095593e2], [0, 7.215377e2, 1.72854e2], [0, 0, 1]])
    cams = {}
    for i, (tx, ang, dist) in enumerate([(0.0, (0.002, -0.003, 0.001), (-0.37, 0.20, 0.001, -0.001, -0.07)),
                                         (-0.537, (0.001, 0.002, -0.002), (-0.37, 0.21, 0.0005, 0.0008, -0.075)),
                                         (0.0598, (0.004, -0.009, 0.0075), (-0.369, 0.197, 0.0013, -0.0006, -0.068)),
                                         (-0.4731, (-0.003, 0.006, -0.004), (-0.364, 0.180, 0.0014, 0.0004, -0.055))]):
        K = np.array([[9.597910e2 + 3 * i, 0.0, 6.960217e2 - 2 * i], [0.0, 9.569251e2 - i, 2.241806e2 + i],
                      [0.0, 0.0, 1.0]])
        cams[i] = {"S": np.array(raw_size, float), "K": K, "D": np.array(dist), "R": _rot(*ang) @ _rot(0.01, 0.0, 0.0),
                   "T": np.array([tx, 0.001 * i, -0.002 * i]), "S_rect": np.array(rect_size, float),
                   "R_rect": _rot(*ang), "P_rect": Kr @ np.hstack([np.eye(3), [[tx], [0.0], [0.0]]])}
    return cams


def write_kitti_raw_calib(path, cams, drop=None, d_len=5):
    fmt = lambda a: " ".join("%.12e" % v for v in np.asarray(a).ravel())
    lines = ["calib_time: 09-Jan-2012 13:57:47", "corner_dist: 9.950000e-02"]
    for i in sorted(cams):
        c = cams[i]
        for key in ("S", "K", "D", "R", "T", "S_rect", "R_rect", "P_rect"):
            name = f"{key}_{i:02d}"
            if name == drop:
                continue
            val = c[key][:d_len] if key == "D" else c[key]
            lines.append(f"{name}: " + fmt(val))
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
