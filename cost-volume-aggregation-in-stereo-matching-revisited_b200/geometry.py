"""Metric depth and 3-D point clouds from the disparity (include/dca_b200.h section 9).

  StereoCalib              focal lengths, principal point, baseline (metres) and doffs of a rectified pair; .Q() is the
                           4x4 reprojection matrix of OpenCV's reprojectImageTo3D convention
  read_kitti_calib         KITTI object / odometry calib files (P2, P3, R0_rect, Tr_velo_to_cam) and the stereo-2015 /
                           raw calib_cam_to_cam.txt (P_rect_02, P_rect_03; R_rect_00 with calib_velo_to_cam.txt)
  read_middlebury_calib    Middlebury calib.txt (cam0, doffs, baseline in mm)
  reproject                disparity (+ confidence / left-right labels as filters) -> PointCloud(xyz, index, count,
                           depth) on the device: one dca_reproject (two launches), no host sync
  save_ply, save_depth_png binary little-endian PLY, KITTI 16-bit depth PNG
  reproject_files          files in, point clouds out: ImagePipeline with the reprojection on the compute stream and
                           the PLY / depth PNG written by the writer thread
"""
import math
from typing import NamedTuple

import numpy as np
import torch

from . import _lib, engine
from .kitti_io import ImagePipeline

REPROJECT_TILE = 1024          # DCA_REPROJECT_TILE: pixels per tile of the workspace


# ---- calibration -------------------------------------------------------------------------------------------
class StereoCalib:
    """A rectified stereo pair: fx, fy, cx, cy in px, baseline in metres, doffs = the x-difference of the principal
    points (px; Middlebury), rect_to_velo = an optional 3x4 float32 transform from the rectified camera frame to
    another frame (KITTI's velodyne frame, see read_kitti_calib), velo_to_rect = the optional 3x4 float32 transform the
    other way (LiDAR points into the rectified camera frame: guide.lidar_hints)."""

    def __init__(self, fx, fy, cx, cy, baseline, doffs=0.0, rect_to_velo=None, velo_to_rect=None):
        self.fx, self.fy, self.cx, self.cy = float(fx), float(fy), float(cx), float(cy)
        self.baseline, self.doffs = float(baseline), float(doffs)
        if not (self.fx > 0 and self.fy > 0 and self.baseline > 0):
            raise ValueError(f"fx, fy and the baseline must be positive, got {fx}, {fy}, {baseline}")
        self.rect_to_velo = None if rect_to_velo is None else np.asarray(rect_to_velo, np.float32).reshape(3, 4)
        self.velo_to_rect = None if velo_to_rect is None else np.asarray(velo_to_rect, np.float32).reshape(3, 4)

    def Q(self):
        """float32 [4,4]: (X', Y', Z', W') = Q (u, v, d, 1) gives Z = fx B / (d + doffs), X = (u - cx) Z / fx,
        Y = (v - cy) Z / fy."""
        r = self.fx / self.fy
        return np.array([[1.0, 0.0, 0.0, -self.cx],
                         [0.0, r, 0.0, -self.cy * r],
                         [0.0, 0.0, 0.0, self.fx],
                         [0.0, 0.0, 1.0 / self.baseline, self.doffs / self.baseline]]).astype(np.float32)

    @property
    def focal_baseline(self):
        """fx * B (px x metres): depth = focal_baseline / (d + doffs)."""
        return self.fx * self.baseline

    def __repr__(self):
        return (f"StereoCalib(fx={self.fx}, fy={self.fy}, cx={self.cx}, cy={self.cy}, baseline={self.baseline}, "
                f"doffs={self.doffs}, rect_to_velo={'set' if self.rect_to_velo is not None else None}, "
                f"velo_to_rect={'set' if self.velo_to_rect is not None else None})")


def _read_kv(path, sep):
    out = {}
    with open(path) as f:
        for line in f:
            key, s, val = line.partition(sep)
            if s:
                out[key.strip()] = val.strip()
    return out


def _floats(text):
    return np.array([float(v) for v in text.replace("[", " ").replace("]", " ").replace(";", " ").split()])


def _h(m):
    """3x4 or 3x3 -> 4x4 homogeneous (float64)."""
    out = np.eye(4)
    m = np.asarray(m, np.float64)
    out[:3, :m.shape[1]] = m
    return out


def read_kitti_calib(path, velo_to_cam=None):
    """KITTI calibration -> StereoCalib of the colour pair (camera 2 = left, camera 3 = right).

    Object / odometry files: P2, P3 and, when present, R0_rect and Tr_velo_to_cam (odometry: Tr, already rectified).
    Stereo-2015 / raw calib_cam_to_cam.txt: P_rect_02, P_rect_03.  B = (P2[0,3] - P3[0,3]) / P2[0,0].  With a
    velodyne transform, rect_to_velo is the pseudo-LiDAR convention: the rectified cam-2 point shifted by camera 2's
    offset (-P2[0,3] / fx, -P2[1,3] / fy, 0), rotated by inv(R0_rect), then the inverse rigid transform of
    Tr_velo_to_cam; composed in float64, stored as float32.  velo_to_rect is its float64 inverse, Tr_velo_to_cam, then
    R0_rect, then the shift back: a velodyne point in the rectified cam-2 frame, where u = fx X / Z + cx.

    velo_to_cam = the path of a raw drive's calib_velo_to_cam.txt (R, T): with a raw calib_cam_to_cam.txt, the velodyne
    transform is [R | T] and the rectifying rotation R_rect_00 (the devkit's P_rect_02 R_rect_00 [R | T]), and both
    rect_to_velo and velo_to_rect are set."""
    kv = _read_kv(path, ":")
    k2, k3 = ("P2", "P3") if "P2" in kv else ("P_rect_02", "P_rect_03")
    if k2 not in kv or k3 not in kv:
        raise ValueError(f"{path}: no P2 / P3 (or P_rect_02 / P_rect_03) projection matrices")
    P2, P3 = _floats(kv[k2]).reshape(3, 4), _floats(kv[k3]).reshape(3, 4)
    fx, fy, cx, cy = P2[0, 0], P2[1, 1], P2[0, 2], P2[1, 2]
    baseline = (P2[0, 3] - P3[0, 3]) / fx
    V2C = R0 = None
    if velo_to_cam is not None:
        vk = _read_kv(velo_to_cam, ":")
        if "R" not in vk or "T" not in vk:
            raise ValueError(f"{velo_to_cam}: no R / T (a KITTI raw calib_velo_to_cam.txt)")
        V2C = np.hstack([_floats(vk["R"]).reshape(3, 3), _floats(vk["T"]).reshape(3, 1)])
        r0 = kv.get("R0_rect", kv.get("R_rect_00"))
        if r0 is None:
            raise ValueError(f"{path}: velo_to_cam needs the rectifying rotation (R_rect_00 or R0_rect)")
        R0 = _floats(r0).reshape(3, 3)
    else:
        tr = kv.get("Tr_velo_to_cam", kv.get("Tr"))
        if tr is not None and ("R0_rect" in kv or "Tr_velo_to_cam" not in kv):
            V2C = _floats(tr).reshape(3, 4)
            R0 = _floats(kv["R0_rect"]).reshape(3, 3) if "R0_rect" in kv else np.eye(3)
    rect_to_velo = velo_to_rect = None
    if V2C is not None:
        C2V = np.eye(4)
        C2V[:3, :3] = V2C[:, :3].T
        C2V[:3, 3] = -V2C[:, :3].T @ V2C[:, 3]
        R0inv = np.eye(4)
        R0inv[:3, :3] = np.linalg.inv(R0)
        shift, unshift = np.eye(4), np.eye(4)
        shift[:3, 3] = (-P2[0, 3] / fx, -P2[1, 3] / fy, 0.0)
        unshift[:3, 3] = (P2[0, 3] / fx, P2[1, 3] / fy, 0.0)
        rect_to_velo = (C2V @ R0inv @ shift)[:3]
        velo_to_rect = (unshift @ _h(R0) @ _h(V2C))[:3]
    return StereoCalib(fx, fy, cx, cy, baseline, 0.0, rect_to_velo, velo_to_rect)


def read_middlebury_calib(path):
    """Middlebury calib.txt (cam0=[f 0 cx; 0 f cy; 0 0 1], doffs, baseline in mm) -> StereoCalib in metres."""
    kv = _read_kv(path, "=")
    K = _floats(kv["cam0"]).reshape(3, 3)
    return StereoCalib(K[0, 0], K[1, 1], K[0, 2], K[1, 2], float(kv["baseline"]) / 1000.0, float(kv.get("doffs", 0.0)))


# ---- reprojection ---------------------------------------------------------------------------------------------
class PointCloud(NamedTuple):
    """Device tensors of one reprojection: xyz fp32 [B, H*W, 3] (rows past count[b] unwritten), index int32 [B, H*W]
    (window pixel y*W + x of each point), count int64 [B], depth fp32 [B,H,W] (0 = no depth)."""
    xyz: torch.Tensor
    index: torch.Tensor
    count: torch.Tensor
    depth: torch.Tensor

    def numpy(self, b=0, rgb=None):
        """Read back image b (synchronises): (xyz float32 [n,3], colours uint8 [n,3] or None).  rgb = a host image
        [H, W, >=3] covering the same window as the depth map; the colours are gathered through `index`."""
        n = int(self.count[b])
        xyz = self.xyz[b, :n].cpu().numpy()
        if rgb is None:
            return xyz, None
        a = np.asarray(rgb)
        if a.shape[:2] != tuple(self.depth.shape[1:]) or a.ndim != 3 or a.shape[2] < 3:
            raise ValueError(f"rgb {a.shape}: expected [{self.depth.shape[1]}, {self.depth.shape[2]}, 3]")
        return xyz, np.ascontiguousarray(a[..., :3].reshape(-1, 3)[self.index[b, :n].cpu().numpy()], dtype=np.uint8)


def _reproject_kernel(disp, peak, label, u0, v0, Q, T, min_peak, min_depth, max_depth):
    """One dca_reproject over [B,H,W] views sharing one layout (unit column stride)."""
    engine._require_cuda(disp, peak, label)
    B, H, W = disp.shape
    pitch_row = disp.stride(1)
    pitch_img = disp.stride(0) if B > 1 else H * pitch_row
    dev = disp.device
    tiles = (H * W + REPROJECT_TILE - 1) // REPROJECT_TILE
    depth = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    xyz = torch.empty((B, H * W, 3), dtype=torch.float32, device=dev)
    index = torch.empty((B, H * W), dtype=torch.int32, device=dev)
    count = torch.empty((B,), dtype=torch.int64, device=dev)
    ws = torch.empty((B, tiles), dtype=torch.int32, device=dev)
    q = np.ascontiguousarray(Q, np.float32)
    t = None if T is None else np.ascontiguousarray(T, np.float32)
    _lib.call("dca_reproject", disp.data_ptr(), 0 if peak is None else peak.data_ptr(),
              0 if label is None else label.data_ptr(), pitch_row, pitch_img, B, H, W, u0, v0, q.ctypes.data,
              None if t is None else t.ctypes.data, float(min_peak), float(min_depth), float(max_depth),
              depth.data_ptr(), xyz.data_ptr(), index.data_ptr(), count.data_ptr(), ws.data_ptr(),
              torch.cuda.current_stream(dev).cuda_stream)
    return PointCloud(xyz, index, count, depth)


def _bhw(t, what, dtype):
    if not torch.is_tensor(t):
        raise ValueError(f"{what}: expected a torch tensor, got {type(t).__name__}")
    if t.dim() == 4 and t.shape[1] == 1:
        t = t[:, 0]
    if t.dim() != 3 or t.dtype != dtype:
        raise ValueError(f"{what}: expected {dtype} [B,H,W] or [B,1,H,W], got {t.dtype} {tuple(t.shape)}")
    return t


def _window_maps(disp, confidence, label, window):
    """The disp / confidence / label maps ([B,H,W] or [B,1,H,W]) as [B,h,w] views of the window that share one layout
    with a unit column stride (copied only when they do not), and the image pixel (u0, v0) of window pixel (0, 0)."""
    maps = [_bhw(disp, "disp", torch.float32)]
    maps.append(None if confidence is None else _bhw(confidence, "confidence", torch.float32))
    maps.append(None if label is None else _bhw(label, "label", torch.uint8))
    for m in maps[1:]:
        if m is not None and (m.shape != maps[0].shape or m.device != maps[0].device):
            raise ValueError(f"confidence / label {tuple(m.shape)} on {m.device}: expected {tuple(maps[0].shape)} "
                             f"on {maps[0].device}")
    u0 = v0 = 0
    if window is not None:
        y0, x0, h, w, v_origin = (int(v) for v in window)
        H, W = maps[0].shape[1:]
        if not (0 <= y0 and 0 <= x0 and h > 0 and w > 0 and y0 + h <= H and x0 + w <= W):
            raise ValueError(f"window {tuple(window)} outside the {H}x{W} map")
        maps = [None if m is None else m[:, y0:y0 + h, x0:x0 + w] for m in maps]
        u0, v0 = x0, v_origin
    live = [m for m in maps if m is not None]
    if any(m.stride() != live[0].stride() or m.stride(2) != 1 for m in live):
        maps = [None if m is None else m.contiguous() for m in maps]
    return maps, u0, v0


def reproject(disp, calib, *, confidence=None, min_confidence=0.0, label=None, frame="camera", min_depth=0.0,
              max_depth=math.inf, window=None):
    """disp fp32 [B,H,W] or [B,1,H,W] (pred4, or LRCheck.filled) -> PointCloud on the same device, without a host sync.

    confidence   a Confidence.peak map: pixels with peak < min_confidence are dropped
    label        LRCheck.label: only DCA_LR_CONSISTENT pixels are kept
    frame        "camera" (the rectified left camera; X right, Y down, Z forward) or "velodyne" (calib.rect_to_velo)
    min_depth, max_depth   pixels with Z outside [min_depth, max_depth] (metres) are dropped
    window       (y0, x0, h, w, v_origin): reproject only rows y0..y0+h and columns x0..x0+w of the maps, with window
                 pixel (y, x) at image pixel (u, v) = (x0 + x, v_origin + y).  It undoes the framing of a network
                 input without a copy: the network frame's columns are the image's, its rows are shifted (zero
                 padding on top, or a centre crop).  None = the whole map, (u, v) = (x, y).
    The calibration applies to every image of the batch."""
    if frame not in ("camera", "velodyne"):
        raise ValueError(f"frame must be 'camera' or 'velodyne', got {frame!r}")
    T = None
    if frame == "velodyne":
        if calib.rect_to_velo is None:
            raise ValueError("frame='velodyne' needs a calibration with rect_to_velo (read_kitti_calib of an object / "
                             "odometry calib file)")
        T = calib.rect_to_velo
    maps, u0, v0 = _window_maps(disp, confidence, label, window)
    return _reproject_kernel(maps[0], maps[1], maps[2], u0, v0, calib.Q(), T,
                             min_confidence if confidence is not None else 0.0, min_depth, max_depth)


# ---- writers --------------------------------------------------------------------------------------------------
def save_ply(path, xyz, rgb=None, normal=None):
    """Binary little-endian PLY: float x y z per vertex, plus float nx ny nz when normal [n,3] is given and uchar red
    green blue when rgb [n,3] is given."""
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    fields = [("x", "<f4"), ("y", "<f4"), ("z", "<f4")]
    if normal is not None:
        normal = np.asarray(normal, np.float32).reshape(-1, 3)
        if len(normal) != len(xyz):
            raise ValueError(f"{len(xyz)} points and {len(normal)} normals")
        fields += [("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4")]
    if rgb is not None:
        rgb = np.asarray(rgb, np.uint8).reshape(-1, 3)
        if len(rgb) != len(xyz):
            raise ValueError(f"{len(xyz)} points and {len(rgb)} colours")
        fields += [("red", "u1"), ("green", "u1"), ("blue", "u1")]
    v = np.empty(len(xyz), dtype=fields)
    v["x"], v["y"], v["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    if normal is not None:
        v["nx"], v["ny"], v["nz"] = normal[:, 0], normal[:, 1], normal[:, 2]
    if rgb is not None:
        v["red"], v["green"], v["blue"] = rgb[:, 0], rgb[:, 1], rgb[:, 2]
    props = "".join(f"property {'float' if t == '<f4' else 'uchar'} {n}\n" for n, t in fields)
    header = f"ply\nformat binary_little_endian 1.0\nelement vertex {len(xyz)}\n{props}end_header\n"
    with open(path, "wb") as f:
        f.write(header.encode("ascii"))
        f.write(v.tobytes())


def save_depth_png(path, depth):
    """KITTI depth format: 16-bit PNG of uint16(min(depth * 256, 65535)), 0 = no depth."""
    from PIL import Image
    a = np.nan_to_num(np.asarray(depth, np.float32) * np.float32(256.0), nan=0.0, posinf=65535.0)
    a = np.clip(a, 0.0, 65535.0).astype("uint16")
    Image.fromarray(a).save(path, format="PNG")
    return a


# ---- files in, point clouds out ---------------------------------------------------------------------------------
class ReprojectPipeline(ImagePipeline):
    """ImagePipeline whose compute stream runs the forward and `reproject` on the window that undoes the framing:

      loader threads   decode + standardise + frame the pair, and keep the left RGB of the window
      compute stream   forward (with confidence / the left-right check when a filter needs them), reproject, then
                       asynchronous D2H of xyz, index, count and the depth map into the slot's pinned buffers
      writer thread    gathers the colours through index, writes the PLY and the depth PNG

    mode "fit" / "pad16" frame the pair as EvalPipeline does; points carry the original image's pixel coordinates.

    With a rectifier (rectify.StereoRectifier) the pairs are raw: the loaders only decode, the slots carry the raw uint8
    pair, the compute stream runs rectify.rectify before the forward, and the colours come from the rectified left image
    (one asynchronous D2H of the window into a pinned slot).  Points then carry rectified-image pixel coordinates."""

    def __init__(self, model, calibs, mode="fit", crop_height=384, crop_width=1248, min_confidence=None,
                 lr_check=False, lr_threshold=1.0, frame="camera", min_depth=0.0, max_depth=math.inf, depth=3,
                 workers=2, rectifier=None):
        if mode not in ("fit", "pad16"):
            raise ValueError(f"mode must be 'fit' or 'pad16', got {mode!r}")
        super().__init__(model, crop_height, crop_width, depth, workers)
        self.calibs, self.mode = calibs, mode
        self.min_confidence, self.lr_check, self.lr_threshold = min_confidence, lr_check, lr_threshold
        self.frame, self.min_depth, self.max_depth = frame, min_depth, max_depth
        self.slot_out = [None] * self.depth          # (xyz, index, count, depth) host buffers per slot
        self.rectifier = rectifier
        if rectifier is not None:
            from .rectify import RawSlots, framing
            W, H = rectifier.rect_size
            self.rect_window = framing(H, W, mode, (crop_height, crop_width))[1]
            self.in_host = self.in_dev = None                  # the fp32 input slots are not used
            self.raw = RawSlots(self, rectifier)
            h, w = self.rect_window[2:4]
            self.rgb_out = [self._host((h, w, 3), torch.uint8) for _ in range(self.depth)]

    def _host(self, shape, dtype):
        t = torch.empty(shape, dtype=dtype)
        return t.pin_memory() if self.cuda else t

    def _ensure(self, slot, Hn, Wn, h, w):
        if tuple(self.in_host[slot].shape) != (6, Hn, Wn):
            self.in_host[slot] = self._host((6, Hn, Wn), torch.float32)
            self.in_dev[slot] = torch.empty((6, Hn, Wn), dtype=torch.float32, device=self.dev) if self.cuda \
                else self.in_host[slot]
        o = self.slot_out[slot]
        if o is None or tuple(o[3].shape) != (h, w):
            self.slot_out[slot] = (self._host((h * w, 3), torch.float32), self._host((h * w,), torch.int32),
                                   self._host((1,), torch.int64), self._host((h, w), torch.float32))

    def _load_item(self, left, right):
        fitted, rgb, window, _, _ = self._load_framed(left, right, self.mode)
        return fitted, np.ascontiguousarray(rgb), window

    def _reproject(self, slot, calib, window):
        if self.rectifier is not None:
            from .rectify import rectify
            raw = self.raw.dev[slot]
            x = rectify(raw[0:1], raw[1:2], self.rectifier, self.mode, (self.ch, self.cw))
            y0, x0, h, w, vo = x.window
            self.rgb_out[slot].copy_(x.rgb[0, 0, vo:vo + h, x0:x0 + w], non_blocking=self.cuda)
            return self._forward_reproject(x.left, x.right, calib, x.window)
        x = self.in_dev[slot]
        return self._forward_reproject(x[None, 0:3], x[None, 3:6], calib, window)

    def _forward_reproject(self, left, right, calib, window):
        conf = self.min_confidence is not None
        kw = {}
        if conf:
            kw["confidence"] = True
        if self.lr_check:
            kw.update(lr_check=True, lr_threshold=self.lr_threshold)
        out = self.model(left, right, **kw)
        pred = out[0] if isinstance(out, (tuple, list)) else out
        return reproject(pred, calib, confidence=out[2].peak if conf else None,
                         min_confidence=self.min_confidence if conf else 0.0,
                         label=out[-1].label if self.lr_check else None, frame=self.frame, min_depth=self.min_depth,
                         max_depth=self.max_depth, window=window)

    def run(self, items):
        """items: (left, right, ply_path or None, depth_png_path or None).  Returns [(xyz float32 [n,3], rgb uint8
        [n,3])] in input order."""
        import queue
        import threading
        from concurrent.futures import ThreadPoolExecutor
        items = list(items)
        if self.rectifier is not None:
            return self._run_raw(items)
        calibs = self.calibs if isinstance(self.calibs, (list, tuple)) else [self.calibs] * len(items)
        if len(calibs) != len(items):
            raise ValueError(f"{len(calibs)} calibrations for {len(items)} items")
        results = [None] * len(items)
        slot_sem = threading.Semaphore(self.depth)
        q = queue.Queue()
        err = []

        def writer():
            while True:
                item = q.get()
                if item is None:
                    return
                i, slot, rgb, ply, png = item
                try:
                    if self.cuda:
                        self.done[slot].synchronize()
                    xyz_h, idx_h, cnt_h, dep_h = self.slot_out[slot]
                    n = int(cnt_h[0])
                    xyz = xyz_h[:n].numpy().copy()
                    col = rgb.reshape(-1, 3)[idx_h[:n].numpy()]
                    if ply is not None:
                        save_ply(ply, xyz, col)
                    if png is not None:
                        save_depth_png(png, dep_h.numpy())
                    results[i] = (xyz, col)
                except Exception as e:          # surfaced by run()
                    err.append(e)
                finally:
                    slot_sem.release()

        wt = threading.Thread(target=writer, daemon=True)
        wt.start()
        was_training = getattr(self.model, "training", False)
        if hasattr(self.model, "eval"):
            self.model.eval()
        try:
            with ThreadPoolExecutor(self.workers) as pool, torch.no_grad():
                futs = [pool.submit(self._load_item, it[0], it[1]) for it in items]
                for i, (fut, it) in enumerate(zip(futs, items)):
                    fitted, rgb, window = fut.result()
                    slot_sem.acquire()
                    slot = i % self.depth
                    self._ensure(slot, fitted.shape[1], fitted.shape[2], window[2], window[3])
                    np.copyto(self.in_host[slot].numpy(), fitted)
                    outs = self.slot_out[slot]
                    if self.cuda:
                        with torch.cuda.stream(self.copy_stream):
                            if i >= self.depth:
                                self.copy_stream.wait_event(self.free[slot])     # kernels of the slot's previous pair
                            self.in_dev[slot].copy_(self.in_host[slot], non_blocking=True)
                            self.h2d[slot].record(self.copy_stream)
                        with torch.cuda.stream(self.compute_stream):
                            self.compute_stream.wait_event(self.h2d[slot])
                            pc = self._reproject(slot, calibs[i], window)
                            self.free[slot].record(self.compute_stream)
                            for h, dv in zip(outs, (pc.xyz[0], pc.index[0], pc.count, pc.depth[0])):
                                h.copy_(dv, non_blocking=True)
                            self.done[slot].record(self.compute_stream)
                    else:
                        pc = self._reproject(slot, calibs[i], window)
                        for h, dv in zip(outs, (pc.xyz[0], pc.index[0], pc.count, pc.depth[0])):
                            h.copy_(dv)
                    q.put((i, slot, rgb, it[2], it[3]))
        finally:
            q.put(None)
            wt.join()
            if was_training and hasattr(self.model, "train"):
                self.model.train()
        if err:
            raise err[0]
        return results

    def _run_raw(self, items):
        """run() on raw pairs (self.rectifier set): the same slot ring, with uint8 raw pairs in and the rectified left
        window's colours out."""
        import queue
        import threading
        from concurrent.futures import ThreadPoolExecutor
        calibs = self.calibs if self.calibs is not None else self.rectifier.calib
        calibs = calibs if isinstance(calibs, (list, tuple)) else [calibs] * len(items)
        if len(calibs) != len(items):
            raise ValueError(f"{len(calibs)} calibrations for {len(items)} items")
        _, _, h, w, _ = self.rect_window
        results = [None] * len(items)
        slot_sem = threading.Semaphore(self.depth)
        q = queue.Queue()
        err = []

        def writer():
            while True:
                item = q.get()
                if item is None:
                    return
                i, slot, ply, png = item
                try:
                    if self.cuda:
                        self.done[slot].synchronize()
                    xyz_h, idx_h, cnt_h, dep_h = self.slot_out[slot]
                    n = int(cnt_h[0])
                    xyz = xyz_h[:n].numpy().copy()
                    col = self.rgb_out[slot].numpy().reshape(-1, 3)[idx_h[:n].numpy()]
                    if ply is not None:
                        save_ply(ply, xyz, col)
                    if png is not None:
                        save_depth_png(png, dep_h.numpy())
                    results[i] = (xyz, col)
                except Exception as e:          # surfaced by run()
                    err.append(e)
                finally:
                    slot_sem.release()

        wt = threading.Thread(target=writer, daemon=True)
        wt.start()
        was_training = getattr(self.model, "training", False)
        if hasattr(self.model, "eval"):
            self.model.eval()
        try:
            with ThreadPoolExecutor(self.workers) as pool, torch.no_grad():
                futs = [pool.submit(self.raw.load, it[0], it[1]) for it in items]
                for i, (fut, it) in enumerate(zip(futs, items)):
                    raw = fut.result()
                    slot_sem.acquire()
                    slot = i % self.depth
                    self._ensure_out(slot, h, w)
                    self.raw.put(slot, raw)
                    outs = self.slot_out[slot]
                    if self.cuda:
                        with torch.cuda.stream(self.copy_stream):
                            if i >= self.depth:
                                self.copy_stream.wait_event(self.free[slot])     # kernels of the slot's previous pair
                            self.raw.h2d(slot)
                            self.h2d[slot].record(self.copy_stream)
                        with torch.cuda.stream(self.compute_stream):
                            self.compute_stream.wait_event(self.h2d[slot])
                            pc = self._reproject(slot, calibs[i], None)
                            self.free[slot].record(self.compute_stream)
                            for hb, dv in zip(outs, (pc.xyz[0], pc.index[0], pc.count, pc.depth[0])):
                                hb.copy_(dv, non_blocking=True)
                            self.done[slot].record(self.compute_stream)
                    else:
                        pc = self._reproject(slot, calibs[i], None)
                        for hb, dv in zip(outs, (pc.xyz[0], pc.index[0], pc.count, pc.depth[0])):
                            hb.copy_(dv)
                    q.put((i, slot, it[2], it[3]))
        finally:
            q.put(None)
            wt.join()
            if was_training and hasattr(self.model, "train"):
                self.model.train()
        if err:
            raise err[0]
        return results

    def _ensure_out(self, slot, h, w):
        o = self.slot_out[slot]
        if o is None or tuple(o[3].shape) != (h, w):
            self.slot_out[slot] = (self._host((h * w, 3), torch.float32), self._host((h * w,), torch.int32),
                                   self._host((1,), torch.int64), self._host((h, w), torch.float32))


def reproject_files(model, items, calib=None, mode="fit", crop=(384, 1248), min_confidence=None, lr_check=False,
                    lr_threshold=1.0, frame="camera", min_depth=0.0, max_depth=math.inf, depth=3, workers=2,
                    rectifier=None):
    """Stereo pairs on disk -> coloured point clouds.  items = (left, right, ply_path or None, depth_png_path or None);
    calib = one StereoCalib or a list aligned with items.  min_confidence drops pixels whose Confidence.peak is below
    it (the forward runs with confidence=True); lr_check=True keeps the left-right consistent pixels only.  Depth PNGs
    cover the image (fit with padding, pad16) or the centre crop (fit of a larger image).  Returns [(xyz float32 [n,3],
    rgb uint8 [n,3])] in input order; PLY and PNG files are written as results arrive.

    rectifier = a rectify.StereoRectifier: the items are RAW pairs of rectifier.raw_size, rectified and standardised on
    the device (rectify.rectify with this mode and crop); calib defaults to rectifier.calib, the colours come from the
    rectified left image and the points carry rectified-image pixel coordinates."""
    if calib is None and rectifier is None:
        raise ValueError("reproject_files needs a calibration (calib=) or a rectifier (rectifier=)")
    pipe = ReprojectPipeline(model, calib, mode, crop[0], crop[1], min_confidence, lr_check, lr_threshold, frame,
                             min_depth, max_depth, depth, workers, rectifier)
    return pipe.run(items)
