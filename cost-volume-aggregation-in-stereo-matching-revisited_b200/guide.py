"""LiDAR guidance of the stereo forward (include/dca_b200.h section 14): Guided Stereo Matching (Poggi et al., CVPR 2019).

  read_velodyne      KITTI velodyne .bin scan -> float32 [N, 4] (x, y, z, reflectance)
  lidar_hints        scans -> fp32 hint map [B,1,H,W] on the device: every point through calib.velo_to_rect into the left
                     (or right) view and the network frame, the nearest point per pixel (dca_lidar_hints, three launches,
                     no host sync)
  modulation_scale   validates the method's k and c and returns s = fp32(1 / (2 c^2))
  hint_map           a user's hint map checked and viewed as the contiguous fp32 [B,H,W] the kernels read

The forward takes the map as `GwcNet.forward(..., hints=)`: engine.guide_quarter pools it to 1/4 resolution and the guided
volume kernel multiplies every channel of volume plane d at a hinted pixel by k exp(-(d - hq)^2 / (2 c^2)).
"""
import math

import numpy as np
import torch

from . import _lib, engine

DEFAULT_K, DEFAULT_C = 10.0, 1.0       # Poggi et al.'s values; not tuned for DCANet


def read_velodyne(path):
    """KITTI velodyne scan (.bin: float32 x, y, z, reflectance per point) -> numpy float32 [N, 4]."""
    a = np.fromfile(path, dtype="<f4")
    if a.size % 4:
        raise ValueError(f"{path}: {a.size} floats, not a multiple of 4 (x, y, z, reflectance)")
    return a.reshape(-1, 4).astype(np.float32, copy=False)


def modulation_scale(k, c):
    """Validate the Gaussian's height k and width c (in volume planes, 4 full-res px each) -> s = fp32(1 / (2 c^2)),
    computed in float64."""
    k, c = float(k), float(c)
    if not (math.isfinite(k) and k > 0):
        raise ValueError(f"hint_k must be finite and > 0, got {k}")
    if not (math.isfinite(c) and c > 0):
        raise ValueError(f"hint_c must be finite and > 0, got {c}")
    with np.errstate(over="ignore"):
        s = float(np.float32(1.0 / (2.0 * c * c)))
    if not math.isfinite(s):
        raise ValueError(f"hint_c = {c} is too small: 1 / (2 c^2) overflows float32")
    return s


def hint_map(hints, B, H, W, what="hints"):
    """fp32 [B,1,H,W] or [B,H,W] CUDA tensor -> contiguous [B,H,W] (a view when it already is one)."""
    engine._require_cuda(hints)
    t = hints[:, 0] if hints.dim() == 4 and hints.shape[1] == 1 else hints
    if t.dim() != 3 or tuple(t.shape) != (B, H, W) or t.dtype != torch.float32:
        raise ValueError(f"{what}: expected float32 [{B},1,{H},{W}] or [{B},{H},{W}], got {hints.dtype} "
                         f"{tuple(hints.shape)}")
    return t.contiguous()


_ZBUF = {}


def _zbuf(dev, B, H, W):
    """Persistent z-buffer workspace per (device, calling stream, shape): no allocator traffic per call."""
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream, B, H, W)
    z = _ZBUF.get(key)
    if z is None:
        z = _ZBUF[key] = torch.empty((B, H, W), dtype=torch.int64, device=dev)
    return z


def _points_on_device(points, dev):
    if not points.is_cuda:
        src = points.contiguous()
        pinned = src.pin_memory()
        points = torch.empty(src.shape, dtype=src.dtype, device=dev)
        points.copy_(pinned, non_blocking=True)
    return points.contiguous()


def lidar_hints(points, calib, shape, *, window=None, view="left", min_depth=1.0, max_depth=80.0):
    """Velodyne scans -> fp32 hint map [B,1,H,W] on the device (0 = no hint).

    points     one [N, 3] or [N, 4] float32 tensor (B = 1) or a list of B of them (numpy arrays and CPU tensors are
               copied to the device through pinned memory; read_velodyne gives [N, 4])
    calib      a StereoCalib with velo_to_rect (read_kitti_calib)
    shape      (H, W) of the map: the network frame of the pair
    window     (y0, x0, h, w, v_origin), the framing `reproject` takes: image pixel (u, v) lands at map pixel
               (y0 + v - v_origin, u), and only pixels inside the window are written.  None = the whole map, (u, v) as is.
    view       "left" (camera 2) or "right" (camera 3: u - disp)
    min_depth, max_depth   points with camera Z outside this range (metres) are dropped; min_depth > 0
    The nearest point wins a pixel (ties: the first point); its disparity is fB / Z - doffs."""
    if calib.velo_to_rect is None:
        raise ValueError("lidar_hints needs a calibration with velo_to_rect (read_kitti_calib of an object / odometry "
                         "file, or of a raw calib_cam_to_cam.txt with velo_to_cam=)")
    if view not in ("left", "right"):
        raise ValueError(f"view must be 'left' or 'right', got {view!r}")
    min_depth, max_depth = float(min_depth), float(max_depth)
    if not (min_depth > 0 and math.isfinite(max_depth) and max_depth >= min_depth):
        raise ValueError(f"need 0 < min_depth <= max_depth < inf, got {min_depth}, {max_depth}")
    H, W = (int(v) for v in shape)
    y0, x0, h, w, v_origin = (0, 0, H, W, 0) if window is None else (int(v) for v in window)
    if not (0 <= y0 and 0 <= x0 and h > 0 and w > 0 and y0 + h <= H and x0 + w <= W):
        raise ValueError(f"window {tuple(window)} outside the {H}x{W} map")
    scans = list(points) if isinstance(points, (list, tuple)) else [points]
    if not scans:
        raise ValueError("points: no scan")
    dev = next((s.device for s in scans if torch.is_tensor(s) and s.is_cuda), None)
    dev = dev if dev is not None else torch.device("cuda", torch.cuda.current_device())
    scans = [torch.as_tensor(s) for s in scans]
    S = scans[0].shape[1] if scans[0].dim() == 2 else 0
    for s in scans:
        if s.dim() != 2 or s.shape[1] != S or S not in (3, 4) or s.dtype != torch.float32:
            raise ValueError(f"points: expected float32 [N, 3] or [N, 4] scans of one width, got {s.dtype} "
                             f"{tuple(s.shape)}")
    counts = [int(s.shape[0]) for s in scans]
    offsets = np.concatenate([[0], np.cumsum(counts)])
    if offsets[-1] >= 2 ** 31:
        raise ValueError(f"{offsets[-1]} points: at most 2^31 - 1 per call")
    B = len(scans)
    if B == 1:
        pts = scans[0]
    elif all(not s.is_cuda for s in scans):
        pts = torch.cat(scans)
    else:
        pts = torch.cat([s.to(dev) for s in scans])
    pts = _points_on_device(pts, dev)
    off = _points_on_device(torch.from_numpy(offsets.astype(np.int32)), dev)
    M = np.ascontiguousarray(calib.velo_to_rect, np.float32)
    out = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
    zbuf = _zbuf(dev, B, H, W)
    _lib.call("dca_lidar_hints", pts.data_ptr(), S, off.data_ptr(), B, int(offsets[-1]), M.ctypes.data,
              calib.fx, calib.fy, calib.cx, calib.cy, calib.focal_baseline, calib.doffs, int(view == "right"), y0, x0,
              h, w, v_origin, min_depth, max_depth, zbuf.data_ptr(), out.data_ptr(), H, W,
              torch.cuda.current_stream(dev).cuda_stream)
    return out
