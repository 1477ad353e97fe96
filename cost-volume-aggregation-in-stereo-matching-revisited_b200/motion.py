"""Moving objects between consecutive depth maps on the GPU (include/dca_b200.h section 16).

  motion          the current and the previous depth map and the ego-motion between them -> Motion(label, residual,
                  instance, objects): every pixel with depth moved into the previous camera and compared with the
                  previous frame's disparity around where it lands (dca_motion_labels, one launch per 16 images), then
                  the 4-connected components of the pixels that fail the test, numbered per image in raster order
                  (dca_motion_components, eight launches).  No host sync
  MovingObjects   the per-object table on the device; .counts() and .numpy() read it back on request

Labels: STATIC (the previous frame holds the point), APPEARED (the previous camera saw through it: something moved into
empty space), BEHIND (hidden at t-1, or the surface moved away), UNSEEN (no previous depth where it lands), INVALID (no
depth).  The default thresholds are starting values chosen on synthetic scenes; they are not tuned for DCANet or KITTI.
"""
import math
from typing import NamedTuple

import numpy as np
import torch

from . import _lib, engine, geometry
from .fusion import _poses, _window_origin

STATIC, APPEARED, BEHIND, UNSEEN, INVALID = 0, 1, 2, 3, 4   # DCA_MOTION_*
MAX_FRAMES = 16                  # DCA_MOTION_MAX_FRAMES: images per dca_motion_labels call
MAX_RADIUS = 4                   # DCA_MOTION_MAX_RADIUS
MAX_OBJECTS = 256                # DCA_MOTION_MAX_OBJECTS: rows of the object table per image
TILE = 1024                      # DCA_MOTION_TILE


def workspace_bytes(B, h, w):
    """DCA_MOTION_WORKSPACE_BYTES: union-find parents and component sizes int32 [B][h w], tile counts int32."""
    return 8 * B * h * w + 4 * B * ((h * w + TILE - 1) // TILE)


class MovingObjects(NamedTuple):
    """The objects of each image, on the device: count int32 [B] (K), dropped int32 [B] (components large enough but
    past the 256 rows); per row k < K (instance id k + 1): ints int32 [B,256,8] = (pixels, APPEARED pixels, BEHIND
    pixels, x_min, y_min, x_max, y_max, 0) in window pixels, extent fp32 [B,256,6] = (min X, max X, min Y, max Y, min Z,
    max Z) in metres in the current camera frame, res_sum int64 [B,256] = the sum of rint(256 residual).  Rows past K
    are 0 (extent NaN)."""
    count: torch.Tensor
    dropped: torch.Tensor
    ints: torch.Tensor
    extent: torch.Tensor
    res_sum: torch.Tensor

    def counts(self):
        """K of every image, int64 [B] on the host (synchronises)."""
        return self.count.cpu().numpy().astype(np.int64)

    def numpy(self, b=0):
        """The K objects of image b on the host (synchronises): dict of pixels, appeared, behind (int64 [K]), box
        int64 [K,4] (x_min, y_min, x_max, y_max), extent float32 [K,6] and mean_residual float64 [K] (px)."""
        k = int(self.count[b])
        ints = self.ints[b, :k].cpu().numpy().astype(np.int64)
        rs = self.res_sum[b, :k].cpu().numpy()
        return dict(pixels=ints[:, 0], appeared=ints[:, 1], behind=ints[:, 2], box=ints[:, 3:7],
                    extent=self.extent[b, :k].cpu().numpy(), mean_residual=rs / 256.0 / np.maximum(ints[:, 0], 1))


class Motion(NamedTuple):
    """label uint8 [B,h,w] (STATIC, APPEARED, BEHIND, UNSEEN, INVALID), residual fp32 [B,h,w] (px: the previous
    disparity nearest the expected one, minus the expected one; NaN without one), instance int32 [B,h,w] (0 = none,
    else the object's id), objects: MovingObjects."""
    label: torch.Tensor
    residual: torch.Tensor
    instance: torch.Tensor
    objects: MovingObjects


def _layout(m):
    B, H, _ = m.shape
    return m.stride(1), (m.stride(0) if B > 1 else H * m.stride(1))


def _labels_kernel(depth, prev, intrinsics, fB, doffs, u0, v0, A, tau, tau_rel, radius, label, residual):
    """One dca_motion_labels of B <= 16 images: depth and prev fp32 [B,h,w] sharing one layout (unit column stride),
    A float32 [B,12]; label uint8 and residual fp32 [B,h,w] contiguous."""
    engine._require_cuda(depth, prev, label, residual)
    B, h, w = depth.shape
    pitch_row, pitch_img = _layout(depth)
    a = np.ascontiguousarray(A, np.float32)
    _lib.call("dca_motion_labels", depth.data_ptr(), prev.data_ptr(), pitch_row, pitch_img, B, h, w, *intrinsics, u0,
              v0, fB, doffs, a.ctypes.data, tau, tau_rel, radius, label.data_ptr(), residual.data_ptr(),
              torch.cuda.current_stream(depth.device).cuda_stream)


def _components_kernel(depth, label, residual, intrinsics, fB, doffs, u0, v0, gate, min_pixels, instance, objects):
    """One dca_motion_components over [B,h,w]: depth in its layout, label / residual / instance contiguous; objects =
    the MovingObjects to fill."""
    engine._require_cuda(depth, label, residual, instance)
    B, h, w = depth.shape
    pitch_row, pitch_img = _layout(depth)
    ws = torch.empty((workspace_bytes(B, h, w),), dtype=torch.uint8, device=depth.device)
    o = objects
    _lib.call("dca_motion_components", depth.data_ptr(), pitch_row, pitch_img, label.data_ptr(), residual.data_ptr(),
              B, h, w, *intrinsics, u0, v0, fB, doffs, gate, min_pixels, instance.data_ptr(), o.count.data_ptr(),
              o.dropped.data_ptr(), o.ints.data_ptr(), o.extent.data_ptr(), o.res_sum.data_ptr(), ws.data_ptr(),
              torch.cuda.current_stream(depth.device).cuda_stream)


def _number(v, what, lo=0.0):
    if isinstance(v, bool) or not isinstance(v, (int, float, np.floating, np.integer)) or not math.isfinite(v) \
            or v < lo:
        raise ValueError(f"{what} must be a finite number >= {lo}, got {v!r}")
    return float(np.float32(v))


def _int(v, what, lo, hi):
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not lo <= v <= hi:
        raise ValueError(f"{what} must be an int in {lo}..{hi}, got {v!r}")
    return int(v)


def _params(tau=3.0, tau_rel=0.05, radius=1, gate=1.0, min_pixels=100):
    """The thresholds of motion(), checked (and the floats rounded to float32)."""
    return (_number(tau, "tau"), _number(tau_rel, "tau_rel"), _int(radius, "radius", 0, MAX_RADIUS),
            _number(gate, "gate"), _int(min_pixels, "min_pixels", 1, 2 ** 31 - 1))


def motion(depth, prev_depth, calib, cur_to_prev, *, window=None, tau=3.0, tau_rel=0.05, radius=1, gate=1.0,
           min_pixels=100):
    """Moving pixels and objects of B depth maps against their previous frames -> Motion on the same device, without a
    host sync.

    depth, prev_depth  fp32 [B,h,w] or [B,1,h,w] metric depth of the same window (PointCloud.depth of
                       geometry.reproject), 0 or NaN = no depth
    calib              the StereoCalib of both frames (fx, fy, cx, cy, focal_baseline, doffs)
    cur_to_prev        [B,4,4] or [B,3,4] (or one [4,4] / [3,4] when B = 1) float64 on the host: T(previous camera <-
                       current camera) = inv(prev_cam_to_world) @ cam_to_world; rounded once to float32
    window             the (y0, x0, h, w, v_origin) given to reproject: depth pixel (x, y) is image pixel
                       (x0 + x, v_origin + y).  None = (0, 0, h, w, 0)
    tau, tau_rel       a previous disparity d within max(tau, tau_rel e) px of the expected e holds the point (the D1
                       rule of evaluation.py)
    radius             the previous frame is searched over the (2 radius + 1)^2 pixels around the projection (0..4)
    gate               neighbouring moving pixels join one object when their disparities differ by at most gate px
    min_pixels         smaller components are not objects (their instance stays 0)
    The defaults were chosen on synthetic scenes; they are not tuned for DCANet or KITTI."""
    depth = geometry._bhw(depth, "depth", torch.float32)
    prev = geometry._bhw(prev_depth, "prev_depth", torch.float32)
    if prev.shape != depth.shape or prev.device != depth.device:
        raise ValueError(f"prev_depth {tuple(prev.shape)} on {prev.device}: expected {tuple(depth.shape)} on "
                         f"{depth.device}")
    B, h, w = depth.shape
    if B < 1 or h < 1 or w < 1:
        raise ValueError(f"depth {tuple(depth.shape)}: an empty batch or window")
    u0, v0 = _window_origin(window, h, w)
    with np.errstate(over="ignore"):
        A = _poses(cur_to_prev, B)[:, :3].reshape(B, 12).astype(np.float32)
    if not np.isfinite(A).all():
        raise ValueError("cur_to_prev overflows float32")
    tau, tau_rel, radius, gate, min_pixels = _params(tau, tau_rel, radius, gate, min_pixels)
    intr = (calib.fx, calib.fy, calib.cx, calib.cy)
    fB, doffs = float(calib.focal_baseline), float(calib.doffs)
    if not (all(math.isfinite(v) for v in intr + (fB, doffs)) and math.isfinite(float(np.float32(fB)))):
        raise ValueError(f"calib {calib!r}: not finite in float32")
    if depth.stride(2) != 1 or prev.stride() != depth.stride():
        depth, prev = depth.contiguous(), prev.contiguous()
    dev = depth.device
    label = torch.empty((B, h, w), dtype=torch.uint8, device=dev)
    residual = torch.empty((B, h, w), dtype=torch.float32, device=dev)
    instance = torch.empty((B, h, w), dtype=torch.int32, device=dev)
    objects = MovingObjects(torch.empty((B,), dtype=torch.int32, device=dev),
                            torch.empty((B,), dtype=torch.int32, device=dev),
                            torch.empty((B, MAX_OBJECTS, 8), dtype=torch.int32, device=dev),
                            torch.empty((B, MAX_OBJECTS, 6), dtype=torch.float32, device=dev),
                            torch.empty((B, MAX_OBJECTS), dtype=torch.int64, device=dev))
    for s in range(0, B, MAX_FRAMES):
        e = min(B, s + MAX_FRAMES)
        _labels_kernel(depth[s:e], prev[s:e], intr, fB, doffs, u0, v0, A[s:e], tau, tau_rel, radius, label[s:e],
                       residual[s:e])
    _components_kernel(depth, label, residual, intr, fB, doffs, u0, v0, gate, min_pixels, instance, objects)
    return Motion(label, residual, instance, objects)


def _options(motion_opt):
    """fuse_files / track_files' motion= -> the keyword arguments of motion(), or None (off)."""
    if motion_opt is None or motion_opt is False:
        return None
    if motion_opt is True:
        return {}
    if isinstance(motion_opt, dict):
        allowed = {"tau", "tau_rel", "radius", "gate", "min_pixels"}
        bad = set(motion_opt) - allowed
        if bad:
            raise ValueError(f"motion: unknown options {sorted(bad)}; allowed {sorted(allowed)}")
        _params(**motion_opt)
        return dict(motion_opt)
    raise ValueError(f"motion must be None, True or a dict of motion() options, got {motion_opt!r}")
