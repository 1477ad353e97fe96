"""The Stixel World from the disparity on the GPU (include/dca_b200.h section 15).

  ground_profile   disparity (+ Confidence.peak, + LRCheck.label as filters) -> GroundProfile(disp, line, inliers, ok):
                   the flat-road V-disparity line d_g(y) = a (y - y_h) of Labayrade et al. (2002), found by a Hough search
                   and refined by an exact least-squares fit.  One dca_ground_profile (six launches), no host sync
  stixels          disparity + a per-row ground profile -> Stixels: each column of `width` pixels split bottom-up into
                   ground, object and sky segments by dynamic programming (Pfeiffer & Franke 2011, made GPU-parallel as in
                   Hernandez-Juarez et al. 2017, in a simplified model).  One dca_stixels (three launches), no host sync
  Stixels.render   the dense disparity and class maps of the segments (one dca_stixel_render)
  Stixels.metric   per-segment Z, column-centre X and the Y of the top and bottom rows in the camera frame

Everything after the quantisation to 1/256 px is integer, so the results do not depend on the order of any atomic or
reduction.  The default priors are starting values chosen on a synthetic driving scene; they are not tuned for DCANet or
KITTI.
"""
import math
from typing import NamedTuple

import numpy as np
import torch

from . import _lib, engine, geometry

GROUND, OBJECT, SKY = 0, 1, 2        # DCA_STIXEL_GROUND / OBJECT / SKY
MAX_WIDTH = 16                       # DCA_STIXEL_MAX_WIDTH
MAX_ROWS = 768                       # DCA_STIXEL_MAX_ROWS: the DP's shared memory per column
MAX_DISP = 1024                      # DCA_STIXEL_MAX_DISP
MAX_SIGMA = 16384                    # DCA_STIXEL_MAX_SIGMA, 1/256 px
MAX_TAU = 8                          # DCA_STIXEL_MAX_TAU
MAX_PRIOR = 1 << 20                  # DCA_STIXEL_MAX_PRIOR
GROUND_NA = 253                      # DCA_GROUND_NA: Hough slopes 1/64 + i / 256, i < 253
GROUND_MAX_ROWS = 4096               # DCA_GROUND_MAX_ROWS


def ground_workspace_bytes(B, H, max_disp):
    """DCA_GROUND_WORKSPACE_BYTES."""
    return 4 * B * H * (max_disp + GROUND_NA) + 48 * B


def stixel_workspace_bytes(B, H, W, width, max_disp):
    """DCA_STIXEL_WORKSPACE_BYTES: the column samples and the object lut [B][ncols][max_disp + 1][H + 1] (72 MB for one
    375 x 1242 window at max_disp 192)."""
    return 4 * B * -(-W // width) * (H + (max_disp + 1) * (H + 1))


class GroundProfile(NamedTuple):
    """disp fp32 [B,h]: the ground disparity of each window row (0 above the horizon, and everywhere when not ok);
    line fp64 [B,2]: (a, y_h), (0, 0) when not ok; inliers int32 [B]: the pixels of the fit; ok bool [B]."""
    disp: torch.Tensor
    line: torch.Tensor
    inliers: torch.Tensor
    ok: torch.Tensor


class StixelMetric(NamedTuple):
    """fp32 [B, ncols, h] per segment, in metres in the rectified left camera frame (X right, Y down, Z forward); NaN for
    ground and sky segments and past count."""
    z: torch.Tensor
    x: torch.Tensor
    y_top: torch.Tensor
    y_bottom: torch.Tensor


class Stixels(NamedTuple):
    """The segments of every column, bottom-up: segment i < count[b, k] of column k spans window rows top[b, k, i] ..
    bottom[b, k, i] (int16, bottom >= top) with class cls (uint8: GROUND, OBJECT, SKY) and disparity disp (fp32, px; 0
    for ground and sky).  Entries past count are not written.  free_space int32 [B, ncols]: the top row of the ground
    segment touching the bottom edge, or h when the bottom segment is not ground.  width: the column width; window: the
    (y0, x0, h, w, v_origin) of the maps ((0, 0, H, W, 0) when stixels() had no window)."""
    count: torch.Tensor
    bottom: torch.Tensor
    top: torch.Tensor
    cls: torch.Tensor
    disp: torch.Tensor
    free_space: torch.Tensor
    width: int
    window: tuple

    def render(self, ground):
        """(disp fp32 [B,h,w], cls uint8 [B,h,w]) of the window: ground rows take the profile's value, objects their
        disparity, sky 0.  ground = the GroundProfile (or fp32 [B,h] profile) the stixels were computed with."""
        B, ncols, h = self.bottom.shape
        prof = _profile(ground, B, h, self.bottom.device)
        w = self.window[3]
        out = torch.empty((B, h, w), dtype=torch.float32, device=prof.device)
        cls = torch.empty((B, h, w), dtype=torch.uint8, device=prof.device)
        engine._require_cuda(self.count, prof)
        _lib.call("dca_stixel_render", self.count.data_ptr(), self.bottom.data_ptr(), self.top.data_ptr(),
                  self.cls.data_ptr(), self.disp.data_ptr(), prof.data_ptr(), B, h, w, self.width, ncols,
                  out.data_ptr(), cls.data_ptr(), torch.cuda.current_stream(prof.device).cuda_stream)
        return out, cls

    def metric(self, calib):
        """StixelMetric of the object segments: Z = fB / (d + doffs), X = (u_c - cx) Z / fx at the column centre
        u_c = x0 + (k w + min((k+1) w, W) - 1) / 2, Y = (v - cy) Z / fy at the top and bottom rows v = v_origin + row
        (the window's image coordinates, as in geometry.reproject).  Element-wise torch ops on the device."""
        B, ncols, h = self.bottom.shape
        _, x0, _, W, vo = self.window
        dev = self.disp.device
        k = torch.arange(ncols, device=dev, dtype=torch.float32)
        uc = x0 + (k * self.width + torch.clamp((k + 1) * self.width, max=W) - 1) * 0.5
        keep = (torch.arange(h, device=dev)[None, None] < self.count[..., None]) & (self.cls == OBJECT)
        z = torch.where(keep, calib.focal_baseline / (self.disp + calib.doffs), float("nan"))
        x = (uc[None, :, None] - calib.cx) * z / calib.fx
        yt = (vo + self.top.float() - calib.cy) * z / calib.fy
        yb = (vo + self.bottom.float() - calib.cy) * z / calib.fy
        return StixelMetric(z, x, yt, yb)


def _int(v, what, lo, hi):
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not lo <= v <= hi:
        raise ValueError(f"{what} must be an int in {lo}..{hi}, got {v!r}")
    return int(v)


def _q256(v, what, lo, hi):
    """A non-negative length in px -> rint(256 v), checked against [lo, hi]."""
    if not (isinstance(v, (int, float, np.floating, np.integer)) and math.isfinite(v)):
        raise ValueError(f"{what} must be a finite number, got {v!r}")
    q = int(np.rint(256.0 * float(v)))
    if not lo <= q <= hi:
        raise ValueError(f"{what} = {v!r} px is outside [{lo / 256}, {hi / 256}] px")
    return q


def _min_peak(confidence, min_confidence):
    if confidence is None:
        return 0.0
    if not isinstance(min_confidence, (int, float, np.floating, np.integer)) or math.isnan(min_confidence):
        raise ValueError(f"min_confidence must be a number, got {min_confidence!r}")
    return float(min_confidence)


def _profile(ground, B, h, device):
    g = ground.disp if isinstance(ground, GroundProfile) else ground
    if not torch.is_tensor(g) or g.dtype != torch.float32 or tuple(g.shape) != (B, h):
        raise ValueError(f"ground: expected a GroundProfile or fp32 [{B},{h}], got "
                         f"{getattr(g, 'dtype', type(g).__name__)} {tuple(getattr(g, 'shape', ()))}")
    if g.device != device:
        raise ValueError(f"ground on {g.device}, disp on {device}")
    return g.contiguous()


def _layout(m):
    B, H, _ = m.shape
    return m.stride(1), (m.stride(0) if B > 1 else H * m.stride(1))


def ground_profile(disp, *, confidence=None, min_confidence=0.0, label=None, max_disp=192, min_inliers=1000,
                   window=None):
    """disp fp32 [B,H,W] or [B,1,H,W] (pred4, or LRCheck.filled) -> GroundProfile of the window, on the same device,
    without a host sync.

    confidence, min_confidence   a Confidence.peak map: pixels with peak < min_confidence are left out
    label        LRCheck.label: only DCA_LR_CONSISTENT pixels are used
    max_disp     pixels with d >= max_disp are left out (the histogram's width)
    min_inliers  fewer fitted pixels than this give ok = False
    window       (y0, x0, h, w, v_origin) as in geometry.reproject; the profile has one value per window row
    ok is also False when the fitted slope is below 1/16 px per row (a baseline of 1/16 of the camera height): a
    fronto-parallel surface fills a band of the flattest lines too, and the fit of that band follows the band's slope.  The profile is then all zeros, so stixels() finds only objects and sky."""
    maps = geometry._window_maps(disp, confidence, label, window)[0]
    min_peak = _min_peak(confidence, min_confidence)
    max_disp = _int(max_disp, "max_disp", 1, MAX_DISP)
    min_inliers = _int(min_inliers, "min_inliers", 1, 2 ** 31 - 1)
    B, h, w = maps[0].shape
    if h > GROUND_MAX_ROWS:
        raise ValueError(f"the window has {h} rows; ground_profile supports at most {GROUND_MAX_ROWS}")
    engine._require_cuda(*maps)
    dev = maps[0].device
    pitch_row, pitch_img = _layout(maps[0])
    prof = torch.empty((B, h), dtype=torch.float32, device=dev)
    line = torch.empty((B, 2), dtype=torch.float64, device=dev)
    inliers = torch.empty((B,), dtype=torch.int32, device=dev)
    ok = torch.empty((B,), dtype=torch.bool, device=dev)
    ws = torch.empty((ground_workspace_bytes(B, h, max_disp),), dtype=torch.uint8, device=dev)
    _lib.call("dca_ground_profile", maps[0].data_ptr(), 0 if maps[1] is None else maps[1].data_ptr(),
              0 if maps[2] is None else maps[2].data_ptr(), pitch_row, pitch_img, B, h, w, min_peak, max_disp,
              min_inliers, prof.data_ptr(), line.data_ptr(), inliers.data_ptr(), ok.data_ptr(), ws.data_ptr(),
              torch.cuda.current_stream(dev).cuda_stream)
    return GroundProfile(prof, line, inliers, ok)


def stixels(disp, ground, *, confidence=None, min_confidence=0.0, label=None, width=5, max_disp=192,
            sigma_ground=1.0, sigma_object=2.0, sigma_sky=2.0, tau=3, p_seg=16384, p_gravity=8192, p_order=8192,
            eps_gravity=2.0, eps_order=1.0, window=None):
    """disp fp32 [B,H,W] or [B,1,H,W] and a ground profile of the window (a GroundProfile, or any fp32 [B,h] per-row
    ground disparity such as a calibrated rig's own) -> Stixels, on the same device, without a host sync.

    confidence, min_confidence, label, max_disp, window   the pixel filters and window of ground_profile
    width        the column width in px (1..16; 5 is the value of Hernandez-Juarez et al.)
    sigma_*      the disparity noise of each class in px: a row costs floor(min(r^2, (tau sigma)^2) 1024 / sigma^2)
                 for a residual r (all in 1/256 px), so 1024 is one sigma^2 and tau sigma the outlier cut-off
    p_seg        the cost of every segment, in 1/1024 sigma^2
    p_gravity    the cost of an object on ground whose disparity differs from the ground's at its foot by more than
                 eps_gravity px
    p_order      the cost of an object above a farther object by more than eps_order px
    The defaults are starting values chosen on a synthetic driving scene, not tuned for DCANet or KITTI."""
    maps = geometry._window_maps(disp, confidence, label, window)[0]
    min_peak = _min_peak(confidence, min_confidence)
    width = _int(width, "width", 1, MAX_WIDTH)
    max_disp = _int(max_disp, "max_disp", 1, MAX_DISP)
    sig = [_q256(s, n, 1, MAX_SIGMA) for s, n in ((sigma_ground, "sigma_ground"), (sigma_object, "sigma_object"),
                                                    (sigma_sky, "sigma_sky"))]
    tau = _int(tau, "tau", 1, MAX_TAU)
    pri = [_int(v, n, 0, MAX_PRIOR) for v, n in ((p_seg, "p_seg"), (p_gravity, "p_gravity"), (p_order, "p_order"))]
    eps = [_q256(v, n, 0, MAX_PRIOR) for v, n in ((eps_gravity, "eps_gravity"), (eps_order, "eps_order"))]
    B, h, w = maps[0].shape
    if h > MAX_ROWS:
        raise ValueError(f"the window has {h} rows; stixels supports at most {MAX_ROWS}")
    prof = _profile(ground, B, h, maps[0].device)
    engine._require_cuda(*maps)
    dev = maps[0].device
    ncols = -(-w // width)
    pitch_row, pitch_img = _layout(maps[0])
    count = torch.empty((B, ncols), dtype=torch.int32, device=dev)
    bottom = torch.empty((B, ncols, h), dtype=torch.int16, device=dev)
    top = torch.empty((B, ncols, h), dtype=torch.int16, device=dev)
    cls = torch.empty((B, ncols, h), dtype=torch.uint8, device=dev)
    sdisp = torch.empty((B, ncols, h), dtype=torch.float32, device=dev)
    free = torch.empty((B, ncols), dtype=torch.int32, device=dev)
    ws = torch.empty((stixel_workspace_bytes(B, h, w, width, max_disp),), dtype=torch.uint8, device=dev)
    _lib.call("dca_stixels", maps[0].data_ptr(), 0 if maps[1] is None else maps[1].data_ptr(),
              0 if maps[2] is None else maps[2].data_ptr(), pitch_row, pitch_img, B, h, w, min_peak, prof.data_ptr(),
              width, max_disp, *sig, tau, *pri, *eps, count.data_ptr(), bottom.data_ptr(), top.data_ptr(),
              cls.data_ptr(), sdisp.data_ptr(), free.data_ptr(), ws.data_ptr(),
              torch.cuda.current_stream(dev).cuda_stream)
    win = tuple(int(v) for v in window) if window is not None else (0, 0, h, w, 0)
    return Stixels(count, bottom, top, cls, sdisp, free, width, win)
