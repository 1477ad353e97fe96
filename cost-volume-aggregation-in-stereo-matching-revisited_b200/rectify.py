"""Rectification of raw stereo pairs on the GPU, straight into the network's standardised input (include/dca_b200.h
section 10).

  StereoRectifier            K / D / R / P of both cameras (OpenCV's initUndistortRectifyMap arguments) -> the two
                             rectification maps (float64 on the host, stored float32, uploaded once per device) and
                             `calib`, the StereoCalib of the rectified pair
  read_kitti_raw_rectifier   KITTI raw calib_cam_to_cam.txt (S, K, D, R_rect, P_rect, S_rect of two cameras)
  rectify                    raw uint8 [B, Hs, Ws, 3|4] pair on the device -> Rectified(left, right, rgb, window): one
                             zero-fill, dca_rectify and dca_standardise_frame on the current stream, no host sync
  rectify_files              raw image files in, rectified-frame disparity out: ImagePipeline whose loaders only decode
                             and whose slots carry the raw uint8 pair
The point-cloud side is geometry.reproject_files(..., rectifier=).
"""
from typing import NamedTuple

import numpy as np
import torch

from . import _lib, engine
from .geometry import StereoCalib, _floats, _read_kv
from .kitti_io import ImagePipeline, crop_prediction

RECTIFY_TILE = 1024            # DCA_RECTIFY_TILE


def _matrix(a, shape, what):
    m = np.asarray(a, np.float64)
    if m.size != shape[0] * shape[1]:
        raise ValueError(f"{what}: expected {shape[0]}x{shape[1]}, got shape {m.shape}")
    m = m.reshape(shape)
    if not np.isfinite(m).all():
        raise ValueError(f"{what} is not finite")
    return m


def _size(s, what):
    try:
        w, h = (int(v) for v in s)
    except (TypeError, ValueError):
        raise ValueError(f"{what}: expected (width, height), got {s!r}") from None
    if w <= 0 or h <= 0 or (w, h) != tuple(float(v) for v in s):
        raise ValueError(f"{what} must be two positive integers (width, height), got {s!r}")
    return w, h


def _distortion(d, what):
    d = np.asarray(d if d is not None else [], np.float64).ravel()
    if d.size not in (0, 4, 5):
        raise ValueError(f"{what}: 0, 4 or 5 Brown-Conrady coefficients (k1, k2, p1, p2, k3) expected, got {d.size}")
    if not np.isfinite(d).all():
        raise ValueError(f"{what} is not finite")
    return np.concatenate([d, np.zeros(5 - d.size)])


def rectify_map(K, D, R, P, rect_size):
    """float64 [H, W, 2]: the raw-image coordinate (x, y) that rectified pixel (row v, column u) samples, by OpenCV's
    initUndistortRectifyMap definition: (x, y, w) = inv(P[:, :3] R) (u, v, 1); NaN where w <= 0; x' = x / w, y' = y / w;
    radial (k1, k2, k3) and tangential (p1, p2) distortion; then (fx xd + skew yd + cx, fy yd + cy) with the raw K."""
    W, H = rect_size
    k1, k2, p1, p2, k3 = D
    iR = np.linalg.inv(P[:, :3] @ R)
    u, v = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    x = iR[0, 0] * u + iR[0, 1] * v + iR[0, 2]
    y = iR[1, 0] * u + iR[1, 1] * v + iR[1, 2]
    w = iR[2, 0] * u + iR[2, 1] * v + iR[2, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        xp, yp = x / w, y / w
    r2 = xp * xp + yp * yp
    kr = 1.0 + ((k3 * r2 + k2) * r2 + k1) * r2
    xd = xp * kr + 2.0 * p1 * xp * yp + p2 * (r2 + 2.0 * xp * xp)
    yd = yp * kr + p1 * (r2 + 2.0 * yp * yp) + 2.0 * p2 * xp * yp
    out = np.stack([K[0, 0] * xd + K[0, 1] * yd + K[0, 2], K[1, 1] * yd + K[1, 2]], -1)
    out[~(w > 0)] = np.nan
    return out


class StereoRectifier:
    """Rectification of a calibrated stereo rig.  Per camera the arguments of OpenCV's initUndistortRectifyMap: K the 3x3
    raw intrinsics, D 0, 4 or 5 distortion coefficients (k1, k2, p1, p2, k3), R the 3x3 rotation from the raw camera
    frame to the rectified frame, P the 3x4 rectified projection (R1, R2, P1, P2 of OpenCV's stereoRectify).  raw_size
    and rect_size are (width, height).

    maps      float32 [2, H, W, 2]: per view and rectified pixel, the raw-image (x, y) it samples (NaN: behind the camera)
    calib     StereoCalib of the rectified pair: fx, fy, cx, cy from P1, baseline (P1[0,3] - P2[0,3]) / fx,
              doffs P2[0,2] - P1[0,2]
    """

    def __init__(self, K1, D1, R1, P1, K2, D2, R2, P2, raw_size, rect_size):
        self.raw_size = _size(raw_size, "raw_size")
        self.rect_size = _size(rect_size, "rect_size")
        cams = []
        for i, (K, D, R, P) in enumerate(((K1, D1, R1, P1), (K2, D2, R2, P2)), 1):
            K, R, P = _matrix(K, (3, 3), f"K{i}"), _matrix(R, (3, 3), f"R{i}"), _matrix(P, (3, 4), f"P{i}")
            D = _distortion(D, f"D{i}")
            if not (K[0, 0] > 0 and K[1, 1] > 0 and P[0, 0] > 0 and P[1, 1] > 0):
                raise ValueError(f"camera {i}: the focal lengths of K and P must be positive")
            if abs(np.linalg.det(P[:, :3] @ R)) < 1e-12:
                raise ValueError(f"camera {i}: P[:, :3] R is singular")
            cams.append((K, D, R, P))
        self.cameras = cams
        self.maps = np.stack([rectify_map(*c, self.rect_size) for c in cams]).astype(np.float32)
        P1, P2 = cams[0][3], cams[1][3]
        self.calib = StereoCalib(P1[0, 0], P1[1, 1], P1[0, 2], P1[1, 2], (P1[0, 3] - P2[0, 3]) / P1[0, 0],
                                 P2[0, 2] - P1[0, 2])
        self._dev_maps = {}

    def device_maps(self, device):
        """The maps on `device`, uploaded on first use (a synchronous copy) and cached."""
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        m = self._dev_maps.get(device)
        if m is None:
            m = self._dev_maps[device] = torch.from_numpy(self.maps).to(device)
        return m

    def __repr__(self):
        return f"StereoRectifier(raw_size={self.raw_size}, rect_size={self.rect_size}, calib={self.calib})"


def read_kitti_raw_rectifier(path, left=2, right=3):
    """KITTI raw calib_cam_to_cam.txt -> StereoRectifier of cameras `left` and `right` (2, 3 = the colour pair), from
    S_0i (raw size), K_0i, D_0i, R_rect_0i, P_rect_0i and S_rect_0i (rectified size)."""
    kv = _read_kv(path, ":")

    def get(key):
        if key not in kv:
            raise ValueError(f"{path}: no {key}")
        return _floats(kv[key])

    args = []
    for i in (left, right):
        args.append([get(f"K_{i:02d}"), get(f"D_{i:02d}"), get(f"R_rect_{i:02d}"), get(f"P_rect_{i:02d}")])
    sizes = [get(f"S_{left:02d}"), get(f"S_rect_{left:02d}")]
    if not np.array_equal(get(f"S_{right:02d}"), sizes[0]) or not np.array_equal(get(f"S_rect_{right:02d}"), sizes[1]):
        raise ValueError(f"{path}: cameras {left} and {right} differ in raw or rectified size")
    return StereoRectifier(*args[0], *args[1], raw_size=sizes[0], rect_size=sizes[1])


# ---- the kernels ------------------------------------------------------------------------------------------------
class Rectified(NamedTuple):
    """Device tensors of one rectification: left, right fp32 [B,3,Hn,Wn] (the network input), rgb uint8 [B,2,H,W,3] (the
    rectified images, view 0 = left) and window = (y0, x0, h, w, v_origin), the geometry.reproject window that undoes
    the framing (points carry rectified-image pixel coordinates)."""
    left: torch.Tensor
    right: torch.Tensor
    rgb: torch.Tensor
    window: tuple


def _require_cuda(*tensors):
    try:
        engine._require_cuda(*tensors)
    except _lib.DcaError as e:
        raise ValueError(str(e)) from None


def _rectify_kernel(left, right, maps, H, W):
    """One dca_rectify over [B,Hs,Ws,C] views sharing one layout -> (rgb uint8 [B,2,H,W,3], moments int64 [B,2,3,2])."""
    _require_cuda(left, right, maps)
    B, Hs, Ws, C = left.shape
    pitch_row = left.stride(1)
    pitch_img = left.stride(0) if B > 1 else Hs * pitch_row
    rgb = torch.empty((B, 2, H, W, 3), dtype=torch.uint8, device=left.device)
    moments = torch.zeros((B, 2, 3, 2), dtype=torch.int64, device=left.device)
    _lib.call("dca_rectify", left.data_ptr(), right.data_ptr(), C, pitch_row, pitch_img, B, Hs, Ws, maps.data_ptr(), H,
              W, rgb.data_ptr(), moments.data_ptr(), torch.cuda.current_stream(left.device).cuda_stream)
    return rgb, moments


def _standardise_kernel(rgb, moments, frame):
    """One dca_standardise_frame -> (left, right) fp32 [B,3,Hn,Wn]."""
    _require_cuda(rgb, moments)
    B, _, H, W, _ = rgb.shape
    Hn, Wn, dst_y0, src_y0, h, w = frame
    left = torch.empty((B, 3, Hn, Wn), dtype=torch.float32, device=rgb.device)
    right = torch.empty((B, 3, Hn, Wn), dtype=torch.float32, device=rgb.device)
    _lib.call("dca_standardise_frame", rgb.data_ptr(), moments.data_ptr(), B, H, W, left.data_ptr(), right.data_ptr(),
              Hn, Wn, dst_y0, src_y0, h, w, torch.cuda.current_stream(rgb.device).cuda_stream)
    return left, right


def framing(H, W, mode="fit", crop=(384, 1248)):
    """(Hn, Wn, dst_y0, src_y0, win_h, win_w) of dca_standardise_frame and the reproject window (y0, x0, h, w, v_origin)
    that frame an H x W image as kitti_io does: "fit" = fit_to_crop (zero padding on top and right, or a centre crop of
    the rows and the columns from 0), "pad16" = pad_to_multiple(16)."""
    if mode == "pad16":
        top, right = (-H) % 16, (-W) % 16
        return (H + top, W + right, top, 0, H, W), (top, 0, H, W, 0)
    if mode != "fit":
        raise ValueError(f"mode must be 'fit' or 'pad16', got {mode!r}")
    ch, cw = (int(v) for v in crop)
    if ch <= 0 or cw <= 0:
        raise ValueError(f"crop must be positive, got {crop!r}")
    if H <= ch and W <= cw:
        return (ch, cw, ch - H, 0, H, W), (ch - H, 0, H, W, 0)
    if H < ch or W < cw:
        raise ValueError(f"fit: a {H}x{W} image is neither inside nor around the {ch}x{cw} crop")
    top = int((H - ch) / 2)
    return (ch, cw, 0, top, ch, cw), (0, 0, ch, cw, top)


def _check_raw(left, right, rectifier):
    Ws, Hs = rectifier.raw_size
    for name, t in (("left", left), ("right", right)):
        if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8 or t.dim() != 4 or t.shape[3] not in (3, 4) or \
                tuple(t.shape[1:3]) != (Hs, Ws):
            raise ValueError(f"{name}: expected uint8 [B, {Hs}, {Ws}, 3 or 4] (raw_size {rectifier.raw_size}), got "
                             f"{getattr(t, 'dtype', type(t))} {tuple(getattr(t, 'shape', ()))}")
        if t.stride(3) != 1 or t.stride(2) != t.shape[3]:
            raise ValueError(f"{name}: the channels of a pixel must be adjacent and the pixels of a row packed "
                             f"(strides {t.stride()})")
    if left.shape != right.shape or left.device != right.device:
        raise ValueError(f"left {tuple(left.shape)} on {left.device} and right {tuple(right.shape)} on {right.device} "
                         f"differ")
    if left.shape[0] > 65535:
        raise ValueError(f"at most 65535 pairs per call, got {left.shape[0]}")
    if left.shape[0] > 1 and left.stride() != right.stride():
        left, right = left.contiguous(), right.contiguous()
    elif left.stride(1) != right.stride(1):
        left, right = left.contiguous(), right.contiguous()
    return left, right


def rectify(left, right, rectifier, mode="fit", crop=(384, 1248)):
    """Raw uint8 pair [B, Hs, Ws, 3|4] (RGB or RGBA, unit channel stride, (Ws, Hs) = rectifier.raw_size) on a CUDA device
    -> Rectified(left, right, rgb, window) on the same device, without a host sync once the maps are on the device.

    Each image is remapped into the rectified frame (bilinear, 0 outside the raw image, rounded to uint8), standardised
    by its own per-channel mean and std like kitti_io.load_pair, and framed: mode "fit" = fit_to_crop(crop), "pad16" =
    pad_to_multiple(16).  `left` and `right` go to model(left, right); `window` to geometry.reproject."""
    left, right = _check_raw(left, right, rectifier)
    W, H = rectifier.rect_size
    frame, window = framing(H, W, mode, crop)
    rgb, moments = _rectify_kernel(left, right, rectifier.device_maps(left.device), H, W)
    l, r = _standardise_kernel(rgb, moments, frame)
    return Rectified(l, r, rgb, window)


# ---- raw files in, disparity out --------------------------------------------------------------------------------
def _decode(x):
    from PIL import Image
    a = np.asarray(Image.open(x) if isinstance(x, (str, bytes)) or hasattr(x, "__fspath__") else x)
    if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] not in (3, 4):
        raise ValueError(f"expected an 8-bit RGB or RGBA image, got {a.dtype} {a.shape}")
    return a


class RawSlots:
    """Pinned host and device slots of the raw uint8 pair [2, Hs, Ws, C], (re)allocated when the channel count changes;
    shared by RectifyPipeline and geometry.ReprojectPipeline."""

    def __init__(self, pipe, rectifier):
        self.pipe, self.rectifier = pipe, rectifier
        self.host = [None] * pipe.depth
        self.dev = [None] * pipe.depth

    def load(self, left, right):
        """Loader thread: decode the pair -> uint8 [2, Hs, Ws, C]."""
        a, b = _decode(left), _decode(right)
        Ws, Hs = self.rectifier.raw_size
        if a.shape != b.shape or a.shape[:2] != (Hs, Ws):
            raise ValueError(f"left {a.shape} and right {b.shape}: expected [{Hs}, {Ws}, 3 or 4] (raw_size "
                             f"{self.rectifier.raw_size})")
        return np.stack([a, b])

    def put(self, slot, raw):
        p = self.pipe
        if self.host[slot] is None or tuple(self.host[slot].shape) != raw.shape:
            h = torch.empty(raw.shape, dtype=torch.uint8)
            self.host[slot] = h.pin_memory() if p.cuda else h
            self.dev[slot] = torch.empty(raw.shape, dtype=torch.uint8, device=p.dev) if p.cuda else self.host[slot]
        np.copyto(self.host[slot].numpy(), raw)

    def h2d(self, slot):
        self.dev[slot].copy_(self.host[slot], non_blocking=True)


class RectifyPipeline(ImagePipeline):
    """ImagePipeline on raw (unrectified) pairs:

      loader threads   decode only
      slot ring        pinned uint8 raw pairs; the H2D copy moves uint8 on the copy stream
      compute stream   rectify (fit to the crop) and the forward
      writer thread    crops the prediction back and writes the KITTI 16-bit PNG

    The disparities are in the rectified frame (rectifier.rect_size)."""

    def __init__(self, model, rectifier, crop_height=384, crop_width=1248, depth=3, workers=2):
        super().__init__(model, crop_height, crop_width, depth, workers)
        self.rectifier = rectifier
        W, H = rectifier.rect_size
        framing(H, W, "fit", (crop_height, crop_width))         # a rectified size the crop cannot frame raises here
        self.in_host = self.in_dev = None                          # the fp32 input slots are not used
        self.raw = RawSlots(self, rectifier)

    def run(self, triples):
        """triples: iterable of (raw left, raw right, savename or None).  Returns the cropped disparity maps (float32
        numpy [h, w], rectified frame) in input order; PNGs are written by the writer thread as results arrive."""
        import queue
        import threading
        from concurrent.futures import ThreadPoolExecutor
        triples = list(triples)
        results = [None] * len(triples)
        W, H = self.rectifier.rect_size
        slot_sem = threading.Semaphore(self.depth)
        q = queue.Queue()
        err = []

        def writer():
            while True:
                item = q.get()
                if item is None:
                    return
                i, slot, savename = item
                try:
                    if self.cuda:
                        self.done[slot].synchronize()
                    disp = crop_prediction(self.out_host[slot].numpy(), H, W, self.ch, self.cw).copy()
                    if savename is not None:
                        from .kitti_io import save_disparity_png
                        save_disparity_png(savename, disp)
                    results[i] = disp
                except Exception as e:          # surfaced by run()
                    err.append(e)
                finally:
                    slot_sem.release()

        def forward(slot):
            x = rectify(self.raw.dev[slot][0:1], self.raw.dev[slot][1:2], self.rectifier, "fit", (self.ch, self.cw))
            out = self.model(x.left, x.right)
            pred = out[0] if isinstance(out, (tuple, list)) else out
            return pred.reshape(self.ch, self.cw).float()

        wt = threading.Thread(target=writer, daemon=True)
        wt.start()
        was_training = getattr(self.model, "training", False)
        if hasattr(self.model, "eval"):
            self.model.eval()
        try:
            with ThreadPoolExecutor(self.workers) as pool, torch.no_grad():
                futs = [pool.submit(self.raw.load, l, r) for l, r, _ in triples]
                for i, (fut, (_, _, savename)) in enumerate(zip(futs, triples)):
                    raw = fut.result()
                    slot_sem.acquire()
                    slot = i % self.depth
                    self.raw.put(slot, raw)
                    if self.cuda:
                        with torch.cuda.stream(self.copy_stream):
                            if i >= self.depth:
                                self.copy_stream.wait_event(self.free[slot])     # kernels of the slot's previous pair
                            self.raw.h2d(slot)
                            self.h2d[slot].record(self.copy_stream)
                        with torch.cuda.stream(self.compute_stream):
                            self.compute_stream.wait_event(self.h2d[slot])
                            pred = forward(slot)
                            self.free[slot].record(self.compute_stream)
                            self.out_host[slot].copy_(pred, non_blocking=True)
                            self.done[slot].record(self.compute_stream)
                    else:
                        self.out_host[slot].copy_(forward(slot))
                    q.put((i, slot, savename))
        finally:
            q.put(None)
            wt.join()
            if was_training and hasattr(self.model, "train"):
                self.model.train()
        if err:
            raise err[0]
        return results


def rectify_files(model, triples, rectifier, crop_height=384, crop_width=1248, depth=3, workers=2):
    """Raw stereo pairs on disk -> disparity maps in the rectified frame.  triples = (raw left, raw right, savename or
    None); the images are (Ws, Hs) = rectifier.raw_size, RGB or RGBA.  Each pair is rectified and standardised on the
    device (rectify, mode "fit"), run through the model, cropped back like predict_files and, with a savename, written
    as a KITTI 16-bit PNG.  Returns float32 numpy [h, w] maps in input order."""
    return RectifyPipeline(model, rectifier, crop_height, crop_width, depth, workers).run(triples)
