"""Edge-aware refinement of the disparity on the GPU: a confidence-weighted fast global smoother (Min et al., IEEE TIP
2014) guided by the left image (include/dca_b200.h section 11).

  wls_filter   disparity (+ Confidence.peak, + LRCheck.label) and the uint8 left image -> Refined(disp, support): the
               rejected pixels are filled and the accepted ones smoothed, with disparity edges following colour edges
               (what OpenCV's ximgproc DisparityWLSFilter does, not bit-compatible with it).  One dca_wls_filter call,
               at most 1 + 6 num_iter launches on the current stream, no host sync once the weight table of
               (device, sigma) is cached (the LUT_CACHE most recent ones are kept).  Each line is solved as segments of
               SEGMENT elements joined by a small system over the separators, so a pass has parallelism per line.
"""
import math
from typing import NamedTuple

import numpy as np
import torch

from . import _lib, engine

LUT_SIZE = 3 * 255 * 255 + 1        # DCA_WLS_LUT_SIZE: one weight per squared colour distance
MAX_ITER = 8                        # DCA_WLS_MAX_ITER
SEGMENT = 64                        # DCA_WLS_SEGMENT: separator spacing of the partitioned line solves

LUT_CACHE = 8                       # weight tables kept on the devices (780 KB each)

_LUTS = {}                          # (device, sigma) -> fp32 [LUT_SIZE] on the device, oldest first


class Refined(NamedTuple):
    """disp: the refined disparity, fp32 shaped like the window of the input; support: the smoothed confidence V, in
    [0, 1] up to the fp32 rounding of the solves (small far from any confident pixel; below min_support the input
    disparity is kept)."""
    disp: torch.Tensor
    support: torch.Tensor


def weight_table(sigma):
    """float32 [LUT_SIZE]: lut[k] = exp(-sqrt(k) / sigma) evaluated in float64, then rounded to fp32; k is the squared
    RGB distance of two neighbours."""
    k = np.arange(LUT_SIZE, dtype=np.float64)
    return np.exp(-np.sqrt(k) / float(sigma)).astype(np.float32)


def lambda_schedule(lam, num_iter):
    """The fp32 lambda_t, t = 1..num_iter, of the FGS schedule: fp32(((lam 1.5) 4^(T-t)) / (4^T - 1)) in float64 with
    lam rounded to fp32 first (the C entry point's arithmetic)."""
    lam64 = float(np.float32(lam))
    den = 4.0 ** num_iter - 1.0
    return [np.float32(((lam64 * 1.5) * 4.0 ** (num_iter - t)) / den) for t in range(1, num_iter + 1)]


def workspace_floats(B, H, W):
    """DCA_WLS_WORKSPACE_BYTES / 4: the two weight maps and 8 boundary values per segment of each pass."""
    seg = lambda n: (n - 1) // SEGMENT + 1
    return B * (2 * H * W + 8 * (H * seg(W) + W * seg(H)))


def _device_lut(device, sigma):
    key = (str(device), float(sigma))
    lut = _LUTS.get(key)
    if lut is None:
        lut = torch.from_numpy(weight_table(sigma)).to(device)
        while len(_LUTS) >= LUT_CACHE:
            del _LUTS[next(iter(_LUTS))]
        _LUTS[key] = lut
    return lut


def _wls_kernel(disp, peak, label, guide, lut, lam, num_iter, min_support):
    """One dca_wls_filter over [B,H,W] maps sharing one layout (unit column stride) and a [B,H,W,3|4] uint8 guide
    (unit channel stride, packed pixels)."""
    engine._require_cuda(disp, peak, label, guide, lut)
    B, H, W = disp.shape
    pitch_row = disp.stride(1)
    pitch_img = disp.stride(0) if B > 1 else H * pitch_row
    C = guide.shape[3]
    g_row = guide.stride(1)
    g_img = guide.stride(0) if B > 1 else H * g_row
    dev = disp.device
    refined = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    support = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    ws = torch.empty((workspace_floats(B, H, W),), dtype=torch.float32, device=dev)
    _lib.call("dca_wls_filter", disp.data_ptr(), 0 if peak is None else peak.data_ptr(),
              0 if label is None else label.data_ptr(), pitch_row, pitch_img, B, H, W, guide.data_ptr(), C, g_row,
              g_img, lut.data_ptr(), float(lam), int(num_iter), float(min_support), refined.data_ptr(),
              support.data_ptr(), ws.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    return refined, support


def _bhw(t, what, dtype):
    if not torch.is_tensor(t):
        raise ValueError(f"{what}: expected a torch tensor, got {type(t).__name__}")
    if t.dim() == 4 and t.shape[1] == 1:
        t = t[:, 0]
    if t.dim() != 3 or t.dtype != dtype:
        raise ValueError(f"{what}: expected {dtype} [B,H,W] or [B,1,H,W], got {t.dtype} {tuple(t.shape)}")
    return t


def wls_filter(disp, guide, *, confidence=None, label=None, lam=8000.0, sigma=1.5, num_iter=3, min_support=1e-3,
               window=None):
    """disp fp32 [B,H,W] or [B,1,H,W] (pred4, or LRCheck.filled) -> Refined(disp, support) shaped like the window of
    disp, on the same device, without a host sync (after the first call for a device and sigma).

    guide        uint8 [B,h,w,3|4] (or [h,w,3|4] when B = 1): the left image of the window, RGB or RGBA (channel 3
                 unused); a strided view such as Rectified.rgb[:, 0, vo:vo+h, x0:x0+w] needs no copy
    confidence   a Confidence.peak map (clamped to [0, 1]); None = every pixel fully confident
    label        LRCheck.label: only DCA_LR_CONSISTENT pixels are trusted
    lam, sigma   smoothness (lambda) and colour scale of the weights exp(-|g_p - g_q| / sigma) (grey levels); 8000 and
                 1.5 are the values of OpenCV's disparity-filter tutorial
    num_iter     1..8 row + column passes of the FGS schedule
    min_support  pixels whose support is below it keep the input disparity
    window       (y0, x0, h, w, v_origin) as in geometry.reproject: refine only rows y0..y0+h and columns x0..x0+w of
                 the maps, so the zero padding of a framed network input is never smoothed into the image
    The pixels that do not pass (low confidence, inconsistent, non-finite) are filled from their neighbours along
    paths that do not cross colour edges."""
    maps = [_bhw(disp, "disp", torch.float32)]
    maps.append(None if confidence is None else _bhw(confidence, "confidence", torch.float32))
    maps.append(None if label is None else _bhw(label, "label", torch.uint8))
    for m in maps[1:]:
        if m is not None and (m.shape != maps[0].shape or m.device != maps[0].device):
            raise ValueError(f"confidence / label {tuple(m.shape)} on {m.device}: expected {tuple(maps[0].shape)} "
                             f"on {maps[0].device}")
    if window is not None:
        y0, x0, h, w, _ = (int(v) for v in window)
        H, W = maps[0].shape[1:]
        if not (0 <= y0 and 0 <= x0 and h > 0 and w > 0 and y0 + h <= H and x0 + w <= W):
            raise ValueError(f"window {tuple(window)} outside the {H}x{W} map")
        maps = [None if m is None else m[:, y0:y0 + h, x0:x0 + w] for m in maps]
    B, h, w = maps[0].shape
    if not torch.is_tensor(guide):
        raise ValueError(f"guide: expected a torch tensor, got {type(guide).__name__}")
    if guide.dim() == 3 and B == 1:
        guide = guide[None]
    if guide.dim() != 4 or guide.dtype != torch.uint8 or tuple(guide.shape[:3]) != (B, h, w) \
            or guide.shape[3] not in (3, 4):
        raise ValueError(f"guide: expected uint8 [{B},{h},{w},3|4], got {guide.dtype} {tuple(guide.shape)}")
    if guide.device != maps[0].device:
        raise ValueError(f"guide on {guide.device}, disp on {maps[0].device}")
    if not (isinstance(num_iter, int) and 1 <= num_iter <= MAX_ITER):
        raise ValueError(f"num_iter must be an int in 1..{MAX_ITER}, got {num_iter!r}")
    if not (math.isfinite(lam) and lam >= 0):
        raise ValueError(f"lam must be finite and >= 0, got {lam!r}")
    if not (math.isfinite(sigma) and sigma > 0):
        raise ValueError(f"sigma must be finite and > 0, got {sigma!r}")
    if not min_support >= 0:
        raise ValueError(f"min_support must be >= 0, got {min_support!r}")
    if guide.stride(3) != 1 or guide.stride(2) != guide.shape[3]:
        guide = guide.contiguous()
    live = [m for m in maps if m is not None]
    if any(m.stride() != live[0].stride() or m.stride(2) != 1 for m in live):
        maps = [None if m is None else m.contiguous() for m in maps]
    engine._require_cuda(maps[0])
    lut = _device_lut(maps[0].device, sigma)
    refined, support = _wls_kernel(maps[0], maps[1], maps[2], guide, lut, lam, num_iter, min_support)
    if disp.dim() == 4:
        refined, support = refined[:, None], support[:, None]
    return Refined(refined, support)
