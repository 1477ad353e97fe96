"""Accuracy against ground-truth disparity: the reference's evaluation loop (main_dca.py `mytest` :143-232) on the GPU.

  read_pfm, read_kitti_disparity   ground-truth readers (SceneFlow / Middlebury PFM, KITTI uint16 PNG)
  DisparityMeter                   device-side accumulator: per-image counters of dca_disparity_metrics (EPE, >1/2/3 px,
                                   D1, utils/metrics.py:45-63) and the DCA class-map confusion matrix of
                                   dca_class_confusion (main_dca.py:66-120, 209-232), and with a confidence map the
                                   sparsification tables of dca_confidence_histograms; no host sync until read back
  summarize                        counters -> EPE / bad-N / D1 under both conventions, pixel accuracy / mPA / mIoU,
                                   sparsification curves and AUSE of the confidence, and with a calibration the depth
                                   errors of dca_depth_metrics (abs rel, sq rel, RMSE, RMSE log, delta < 1.25^k)
  evaluate_files                   the `mytest` loop as a streaming pipeline (ImagePipeline plus a GT slot per pair);
                                   with lr_check=True also the metrics of the left-right consistent pixels and of the
                                   background-filled disparity, with wls= those of the refined disparity (wls.py)

Per-rank meters of a distributed run combine by concatenating their `rows()` (and summing `confusion()` and the
`sparsification_histograms()`) before `summarize`.  There is no CPU path: the kernels need CUDA tensors.
"""
import math
import warnings

import numpy as np
import torch

from . import _lib
from .engine import _require_cuda
from .kitti_io import ImagePipeline, crop_prediction, fit_gt_to_crop, pad_gt_to_multiple, save_disparity_png
from .wls import wls_filter

# column order of the counter rows (DCA_METRIC_* of include/dca_b200.h)
VALID, SUM_ABS, GT1, GT2, GT3, D1, PRED_NONFINITE = range(7)
METRIC_COUNT = 7
SUM_ABS_UNIT = 2.0 ** -20          # SUM_ABS is fixed point: px = SUM_ABS * 2^-20
CONF_BINS = 256                    # DCA_CONF_BINS: confidence bins of width 1/256
ERR_BINS = 2048 + 1                # DCA_ERR_BINS: 1/32 px error bins over [0, 64) and one for E >= 64
ERR_BIN_PX = 1.0 / 32
# column order of the depth rows (DCA_DEPTH_* of include/dca_b200.h); the four sums are fixed point, unit 2^-20
DEPTH_VALID, DEPTH_ABS_REL, DEPTH_SQ_REL, DEPTH_SQ, DEPTH_LOG_SQ, DEPTH_A1, DEPTH_A2, DEPTH_A3 = range(8)
DEPTH_COUNT = 8
SPARSIFICATION_DENSITY = [k / 20 for k in range(20, 0, -1)]        # 1.00, 0.95, ..., 0.05


# ---- ground-truth readers (host) ---------------------------------------------------------------------------
def read_pfm(path):
    """Single-channel PFM ('Pf') -> float32 [H,W], top row first.  A negative scale means little-endian data, a
    positive one big-endian; rows are stored bottom-up.  inf (Middlebury's 'no ground truth') is kept."""
    with open(path, "rb") as f:
        header = f.readline().strip()
        if header == b"PF":
            raise ValueError(f"{path}: 3-channel PFM ('PF'), expected a single-channel disparity map ('Pf')")
        if header != b"Pf":
            raise ValueError(f"{path}: not a PFM file (header {header[:8]!r})")
        dims = f.readline().split()
        while len(dims) < 2:
            dims += f.readline().split()
        w, h = int(dims[0]), int(dims[1])
        scale = float(f.readline().strip())
        data = np.frombuffer(f.read(), dtype="<f4" if scale < 0 else ">f4")
    if data.size < w * h:
        raise ValueError(f"{path}: {data.size} values for a {h}x{w} image")
    return np.ascontiguousarray(data[:w * h].reshape(h, w)[::-1], dtype=np.float32)


def read_kitti_disparity(path):
    """KITTI disparity PNG (uint16, disp * 256) -> float32 [H,W] px; 0 = no ground truth."""
    from PIL import Image
    a = np.asarray(Image.open(path))
    if a.ndim != 2:
        raise ValueError(f"{path}: expected a single-channel 16-bit PNG")
    return a.astype(np.float32) / np.float32(256.0)


# ---- kernel calls ----------------------------------------------------------------------------------------
def _disparity_metrics(pred, gt, rows, max_valid):
    """rows int64 [B, METRIC_COUNT] += counters of pred / gt fp32 [B,H,W] (dca_disparity_metrics)."""
    _require_cuda(pred, gt, rows)
    B, H, W = pred.shape
    _lib.call("dca_disparity_metrics", pred.data_ptr(), gt.data_ptr(), rows.data_ptr(), B, H, W, max_valid,
              torch.cuda.current_stream(pred.device).cuda_stream)


def _class_confusion(logits, gt, conf, max_valid):
    """conf int64 [D8,D8] += confusion of logits [B,D8,H8,W8] against gt fp32 [B,8*H8,8*W8] (dca_class_confusion)."""
    _require_cuda(logits, gt, conf)
    B, D8, H8, W8 = logits.shape
    _lib.call("dca_class_confusion", logits.data_ptr(), gt.data_ptr(), conf.data_ptr(), B, D8, H8, W8, max_valid,
              torch.cuda.current_stream(logits.device).cuda_stream)


def _confidence_histograms(pred, gt, peak, conf_hist, err_hist, max_valid):
    """conf_hist int64 [CONF_BINS, 2], err_hist int64 [ERR_BINS, 2] += (count, SUM_ABS) per bin of pred / gt / peak fp32
    [B,H,W] (dca_confidence_histograms)."""
    _require_cuda(pred, gt, peak, conf_hist, err_hist)
    B, H, W = pred.shape
    _lib.call("dca_confidence_histograms", pred.data_ptr(), gt.data_ptr(), peak.data_ptr(), conf_hist.data_ptr(),
              err_hist.data_ptr(), B, H, W, max_valid, torch.cuda.current_stream(pred.device).cuda_stream)


def _depth_metrics(pred, gt, rows, max_valid, focal_baseline, doffs, min_depth, max_depth):
    """rows int64 [B, DEPTH_COUNT] += depth errors of pred / gt fp32 [B,H,W] under one calibration
    (dca_depth_metrics)."""
    _require_cuda(pred, gt, rows)
    B, H, W = pred.shape
    _lib.call("dca_depth_metrics", pred.data_ptr(), gt.data_ptr(), rows.data_ptr(), B, H, W, max_valid,
              focal_baseline, doffs, min_depth, max_depth, torch.cuda.current_stream(pred.device).cuda_stream)


def _as_bhw(t, what):
    if t.dim() == 4 and t.shape[1] == 1:
        t = t[:, 0]
    if t.dim() != 3:
        raise ValueError(f"{what}: expected [B,H,W] or [B,1,H,W], got {tuple(t.shape)}")
    if t.dtype != torch.float32:
        raise ValueError(f"{what}: expected float32, got {t.dtype}")
    return t.contiguous()


class DisparityMeter:
    """Accumulates evaluation counters on the device.

    maxdisp     the model's maxdisp; D8 = maxdisp // 8 disparity classes in the confusion matrix
    max_valid   GT upper bound of the valid mask: None = maxdisp (the (gt > 0) & (gt < maxdisp) mask of the GwcNet /
                PSMNet test loops), 0 = no upper bound (KITTI devkit)
    device      where the counter tables live; None = the device of the first prediction
    min_depth, max_depth   the depth range (metres) of the depth errors of updates with a calibration

    `update` launches the two kernels on the current stream and never synchronises; it allocates only when the row
    table doubles.  `rows()` / `confusion()` / `summary()` are the read-back points."""

    def __init__(self, maxdisp, max_valid=None, device=None, capacity=64, min_depth=1e-3, max_depth=80.0):
        self.maxdisp = int(maxdisp)
        self.D8 = self.maxdisp // 8
        self.max_valid = float(self.maxdisp if max_valid is None else max_valid)
        self.device = None if device is None else torch.device(device)
        if self.device is not None and self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._cap = max(1, int(capacity))
        self._rows = self._conf = None
        self._conf_hist = self._err_hist = None
        self._n = 0
        self._has_conf = False
        self._with_confidence = None      # set by the first update: every update carries a confidence map, or none does
        self.min_depth, self.max_depth = float(min_depth), float(max_depth)
        self._depth_rows = None
        self._with_calib = None           # the same rule for calibrations: depth rows cover the same images as the rows
        if self.device is not None:
            self._alloc()

    def _alloc(self):
        self._rows = torch.zeros((self._cap, METRIC_COUNT), dtype=torch.int64, device=self.device)
        self._conf = torch.zeros((self.D8, self.D8), dtype=torch.int64, device=self.device)

    def __len__(self):
        return self._n

    def update(self, pred4, disp_true, prob_volume=None, confidence=None, calib=None):
        """Score a batch: pred4 [B,1,H,W] (or [B,H,W]) against disp_true [B,H,W] (or [B,1,H,W]) in the same pixel
        frame, both fp32 on the same device; prob_volume [B,D8,H/8,W/8] (the model's second output) adds to the
        confusion matrix; confidence (the `peak` map of the model's Confidence output, in pred4's frame) adds to the
        sparsification tables.  Either every update of a meter passes a confidence map or none does (ValueError
        otherwise): the tables must cover the same pixels as the counter rows, so that the sparsification curves end
        at epe_pooled.  calib (a geometry.StereoCalib shared by the batch) adds one row of depth errors per image; the
        same rule applies: every update passes one or none does."""
        pred, gt = _as_bhw(pred4, "pred4"), _as_bhw(disp_true, "disp_true")
        if gt.shape != pred.shape:
            raise ValueError(f"disp_true {tuple(gt.shape)} and pred4 {tuple(pred.shape)} differ")
        if self.device is None:
            self.device = pred.device
            self._alloc()
        if pred.device != self.device or gt.device != self.device:
            raise ValueError(f"meter lives on {self.device}, tensors on {pred.device} / {gt.device}")
        pv = None
        if prob_volume is not None:
            pv = prob_volume.contiguous()
            B, H, W = pred.shape
            if pv.dim() != 4 or tuple(pv.shape) != (B, self.D8, H // 8, W // 8) or H % 8 or W % 8 \
                    or pv.dtype != torch.float32 or pv.device != self.device:
                raise ValueError(f"prob_volume {tuple(pv.shape)} {pv.dtype}: expected float32 "
                                 f"[{B}, {self.D8}, {H}/8, {W}/8] on {self.device}")
        if self._with_confidence is not None and (confidence is not None) != self._with_confidence:
            raise ValueError("confidence: every update of a meter passes a confidence map or none does (this meter has "
                             f"had updates {'with' if self._with_confidence else 'without'} one)")
        if self._with_calib is not None and (calib is not None) != self._with_calib:
            raise ValueError("calib: every update of a meter passes a calibration or none does (this meter has had "
                             f"updates {'with' if self._with_calib else 'without'} one)")
        pk = None
        if confidence is not None:
            pk = _as_bhw(confidence, "confidence")
            if pk.shape != pred.shape or pk.device != self.device:
                raise ValueError(f"confidence {tuple(pk.shape)} on {pk.device}: expected {tuple(pred.shape)} "
                                 f"on {self.device}")
        B = pred.shape[0]
        if self._n + B > self._cap:
            while self._n + B > self._cap:
                self._cap *= 2
            grown = torch.zeros((self._cap, METRIC_COUNT), dtype=torch.int64, device=self.device)
            grown[:self._n].copy_(self._rows[:self._n])
            self._rows = grown
            if self._depth_rows is not None:
                grown = torch.zeros((self._cap, DEPTH_COUNT), dtype=torch.int64, device=self.device)
                grown[:self._n].copy_(self._depth_rows[:self._n])
                self._depth_rows = grown
        _disparity_metrics(pred, gt, self._rows[self._n:self._n + B], self.max_valid)
        if pv is not None:
            _class_confusion(pv, gt, self._conf, self.max_valid)
            self._has_conf = True
        if pk is not None:
            if self._conf_hist is None:
                self._conf_hist = torch.zeros((CONF_BINS, 2), dtype=torch.int64, device=self.device)
                self._err_hist = torch.zeros((ERR_BINS, 2), dtype=torch.int64, device=self.device)
            _confidence_histograms(pred, gt, pk, self._conf_hist, self._err_hist, self.max_valid)
        if calib is not None:
            if self._depth_rows is None:
                self._depth_rows = torch.zeros((self._cap, DEPTH_COUNT), dtype=torch.int64, device=self.device)
            _depth_metrics(pred, gt, self._depth_rows[self._n:self._n + B], self.max_valid, calib.focal_baseline,
                           calib.doffs, self.min_depth, self.max_depth)
        self._with_confidence = confidence is not None
        self._with_calib = calib is not None
        self._n += B

    def _readback(self, t):
        if t.is_cuda:
            torch.cuda.synchronize(t.device)          # updates may have run on any stream of the device
        return t.cpu().numpy().astype(np.uint64)

    def rows(self):
        """numpy uint64 [N, METRIC_COUNT]: one counter row per image, in update order."""
        if self._rows is None:
            return np.zeros((0, METRIC_COUNT), np.uint64)
        return self._readback(self._rows[:self._n])

    def confusion(self):
        """numpy uint64 [D8, D8]: row = GT class, column = predicted class."""
        if self._conf is None:
            return np.zeros((self.D8, self.D8), np.uint64)
        return self._readback(self._conf)

    def sparsification_histograms(self):
        """(conf_hist [CONF_BINS, 2], err_hist [ERR_BINS, 2]) numpy uint64 of (count, SUM_ABS) per bin, or None before
        any update with a confidence map."""
        if self._conf_hist is None:
            return None
        return self._readback(self._conf_hist), self._readback(self._err_hist)

    def depth_rows(self):
        """numpy uint64 [N, DEPTH_COUNT]: one depth-error row per image, in update order, or None when the updates
        carried no calibration."""
        if self._depth_rows is None:
            return None
        return self._readback(self._depth_rows[:self._n])

    def summary(self):
        h = self.sparsification_histograms()
        return summarize(self.rows(), self.confusion() if self._has_conf else None, *(h or (None, None)),
                         depth_rows=self.depth_rows())


def _nanmean(a):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return float(np.nanmean(a)) if a.size else float("nan")


def _sparsification_curve(hist, order):
    """EPE (px) of the most trusted fraction q of the pixels for every q of SPARSIFICATION_DENSITY: bins are taken
    whole in `order`, the boundary bin with the same fraction of its count and of its sum."""
    h = np.asarray(hist, dtype=np.uint64).reshape(-1, 2)[order]
    n, s = [int(v) for v in h[:, 0]], [int(v) for v in h[:, 1]]      # Python ints: exact sums
    total = sum(n)
    out = []
    for q in SPARSIFICATION_DENSITY:
        if not total:
            out.append(float("nan"))
            continue
        target = total * q
        take_n = take_s = 0
        part = 0.0
        for k in range(len(n)):
            if take_n + n[k] > target:
                part = (target - take_n) / n[k] * s[k]
                break
            take_n += n[k]
            take_s += s[k]
        out.append((take_s + part) * SUM_ABS_UNIT / target)
    return out


def _auc(curve):
    """Trapezoid of a sparsification curve over the removed fraction x = 1 - q in [0, 0.95]."""
    x = [1.0 - q for q in SPARSIFICATION_DENSITY]
    return float(sum(0.5 * (curve[i] + curve[i + 1]) * (x[i + 1] - x[i]) for i in range(len(x) - 1)))


def summarize(rows, confusion=None, conf_hist=None, err_hist=None, depth_rows=None):
    """Counter rows [N, METRIC_COUNT] (+ confusion [D8,D8]) (+ the sparsification tables) -> dict of metrics.

    epe, bad1, bad2, bad3, d1            mean over images of the per-image values (GwcNet / PSMNet test loops); images
                                         without valid pixels are skipped and counted in n_images_skipped
    *_pooled                             the same over all valid pixels at once (KITTI devkit)
    bad-N and D1 are fractions of the valid pixels; a non-finite prediction counts as an error of every kind and is
    left out of the EPE sum (the EPE is over the valid pixels with a finite prediction; n_pred_nonfinite says how many
    were not).  From the confusion matrix, the segmentation Evaluator's formulas (main_dca.py:66-120):
    pixel_accuracy = trace / total, mpa = nanmean(diag / row sums), miou = nanmean(diag / (row + column sums - diag));
    classes with neither GT nor predictions are nan and left out of the means.

    With both sparsification tables (DisparityMeter.sparsification_histograms):
    sparsification_density       q = 1.00, 0.95, ..., 0.05
    sparsification_epe           EPE of the N*q most confident pixels (highest confidence bins first; the boundary bin
                                 contributes the same fraction of its count and of its sum |E|)
    sparsification_epe_ideal     the same with the lowest-error bins first: the best any ranking can do, to within one
                                 error bin (1/32 px) as long as the boundary bin is not the E >= 64 px one (the
                                 error-sorted curve of the sparsification literature; DESIGN.md section 4 on its name)
    auc_epe, ause_epe            trapezoid of the confidence curve over the removed fraction 1 - q in [0, 0.95], and
                                 that minus the same area of the ideal curve (px; 0 = a perfect ranking)
    At q = 1 both curves equal epe_pooled exactly (the same integer sums).

    With depth rows (DisparityMeter.depth_rows), `depth` = the Eigen et al. errors, each as the mean over images of the
    per-image value (images without valid pixels skipped) and as *_pooled over all pixels:
    abs_rel = mean |Zp-Zg|/Zg, sq_rel = mean (Zp-Zg)^2/Zg (m), rmse = sqrt(mean (Zp-Zg)^2) (m),
    rmse_log = sqrt(mean (ln Zp - ln Zg)^2), a1 / a2 / a3 = fraction with max(Zp/Zg, Zg/Zp) < 1.25 / 1.25^2 / 1.25^3;
    plus n_valid, the pixels scored."""
    r = np.asarray(rows, dtype=np.uint64).reshape(-1, METRIC_COUNT).astype(np.float64)
    valid, nonfinite = r[:, VALID], r[:, PRED_NONFINITE]
    finite = valid - nonfinite
    epe_sum = r[:, SUM_ABS] * SUM_ABS_UNIT
    has = valid > 0
    out = {"n_images": int(r.shape[0]), "n_images_skipped": int((~has).sum()), "n_valid": int(valid.sum()),
           "n_pred_nonfinite": int(nonfinite.sum())}
    with np.errstate(divide="ignore", invalid="ignore"):
        per = {"epe": epe_sum[has] / finite[has]}
        for name, col in (("bad1", GT1), ("bad2", GT2), ("bad3", GT3), ("d1", D1)):
            per[name] = r[has, col] / valid[has]
        for name, v in per.items():
            out[name] = float(v.mean()) if v.size else float("nan")
        n, nf = valid.sum(), finite.sum()
        out["epe_pooled"] = float(epe_sum.sum() / nf) if nf else float("nan")
        for name, col in (("bad1", GT1), ("bad2", GT2), ("bad3", GT3), ("d1", D1)):
            out[name + "_pooled"] = float(r[:, col].sum() / n) if n else float("nan")
        if confusion is not None:
            cm = np.asarray(confusion, dtype=np.float64)
            diag, gt_n, pred_n = np.diag(cm), cm.sum(axis=1), cm.sum(axis=0)
            total = cm.sum()
            out["pixel_accuracy"] = float(diag.sum() / total) if total else float("nan")
            out["mpa"] = _nanmean(diag / gt_n)
            out["miou"] = _nanmean(diag / (gt_n + pred_n - diag))
            out["n_class_pixels"] = int(total)
    if conf_hist is not None and err_hist is not None:
        curve = _sparsification_curve(conf_hist, slice(None, None, -1))
        ideal = _sparsification_curve(err_hist, slice(None))
        out["sparsification_density"] = list(SPARSIFICATION_DENSITY)
        out["sparsification_epe"] = curve
        out["sparsification_epe_ideal"] = ideal
        out["auc_epe"] = _auc(curve)
        out["ause_epe"] = out["auc_epe"] - _auc(ideal)
    if depth_rows is not None:
        out["depth"] = _depth_summary(depth_rows)
    return out


def _depth_summary(depth_rows):
    r = np.asarray(depth_rows, dtype=np.uint64).reshape(-1, DEPTH_COUNT).astype(np.float64)
    n = r[:, DEPTH_VALID]
    has = n > 0
    cols = {"abs_rel": (DEPTH_ABS_REL, SUM_ABS_UNIT, False), "sq_rel": (DEPTH_SQ_REL, SUM_ABS_UNIT, False),
            "rmse": (DEPTH_SQ, SUM_ABS_UNIT, True), "rmse_log": (DEPTH_LOG_SQ, SUM_ABS_UNIT, True),
            "a1": (DEPTH_A1, 1.0, False), "a2": (DEPTH_A2, 1.0, False), "a3": (DEPTH_A3, 1.0, False)}
    out = {"n_valid": int(n.sum())}
    total = n.sum()
    for name, (col, unit, root) in cols.items():
        per = r[has, col] * unit / n[has]
        pooled = r[:, col].sum() * unit / total if total else float("nan")
        if root:
            per, pooled = np.sqrt(per), math.sqrt(pooled) if total else float("nan")
        out[name] = float(per.mean()) if per.size else float("nan")
        out[name + "_pooled"] = float(pooled)
    return out


# ---- the evaluation loop -----------------------------------------------------------------------------------
class EvalPipeline(ImagePipeline):
    """ImagePipeline with a ground-truth slot per pair and a `DisparityMeter.update` after every forward.

      loader threads   decode + standardise + frame the pair AND its GT (same framing, padding = invalid)
      slot ring        pinned image and GT buffers; both go to the device on the copy stream
      compute stream   forward, then meter.update (pred4 and prob_volume2 against the framed GT), then the D2H of the
                       prediction when a PNG is wanted
      writer thread    crops the prediction back and writes the KITTI PNG, as ImagePipeline does

    mode "fit": fit_to_crop / fit_gt_to_crop into crop_height x crop_width (my_img.py); "pad16": top/right zero padding
    to multiples of 16 (main_dca.py:153-166), slot buffers follow each pair's padded size.

    wls (a dict of wls_filter's lam / sigma / num_iter / min_support, or None): the slots also carry the uint8 left
    image of the window, and after the forward wls_filter refines the window of pred (of LRCheck.filled, with
    LRCheck.label, when lr_check is set; with Confidence.peak when confidence is set) and `wls_meter` scores it against
    the GT of the window."""

    def __init__(self, model, meter, mode="fit", crop_height=384, crop_width=1248, depth=3, workers=2, confidence=False,
                 lr_check=False, lr_threshold=1.0, calib=None, wls=None):
        if mode not in ("fit", "pad16"):
            raise ValueError(f"mode must be 'fit' or 'pad16', got {mode!r}")
        super().__init__(model, crop_height, crop_width, depth, workers)
        self.meter, self.mode, self.confidence = meter, mode, confidence
        self.lr_check, self.lr_threshold = lr_check, lr_threshold
        self.calib = calib             # None, one StereoCalib, or one per pair: the meter's depth errors
        self._pair_calib = None
        # with lr_check: pred scored on the consistent pixels only, and the background-filled disparity on all of them
        self.lr_meters = {k: DisparityMeter(meter.maxdisp, meter.max_valid, meter.device)
                          for k in ("lr_consistent", "lr_filled")} if lr_check else {}
        self.gt_host = [self._host(crop_height, crop_width) for _ in range(self.depth)]
        self.gt_dev = [torch.empty((crop_height, crop_width), dtype=torch.float32, device=self.dev)
                       for _ in range(self.depth)] if self.cuda else self.gt_host
        self.wls = wls
        self.wls_meter = DisparityMeter(meter.maxdisp, meter.max_valid, meter.device) if wls is not None else None
        # with wls: the uint8 left image of the window per slot, flat buffers sized for the crop and grown only for
        # larger windows (pad16), so pairs of varying size reuse the pinned memory through contiguous views
        self.rgb_host = [None] * self.depth
        self.rgb_dev = [None] * self.depth
        self._pair_window = None

    def _host(self, *shape):
        t = torch.empty(shape, dtype=torch.float32)
        return t.pin_memory() if self.cuda else t

    def _ensure(self, slot, H, W):
        """(Re)size a slot's buffers to an H x W frame (only pad16 mode changes sizes; the slot is idle here)."""
        if tuple(self.gt_host[slot].shape) == (H, W):
            return
        self.in_host[slot], self.out_host[slot], self.gt_host[slot] = self._host(6, H, W), self._host(H, W), \
            self._host(H, W)
        if self.cuda:
            self.in_dev[slot] = torch.empty((6, H, W), dtype=torch.float32, device=self.dev)
            self.gt_dev[slot] = torch.empty((H, W), dtype=torch.float32, device=self.dev)
        else:
            self.in_dev[slot], self.gt_dev[slot] = self.in_host[slot], self.gt_host[slot]

    def _rgb_slot(self, slot, h, w):
        """(host, device) contiguous uint8 [h,w,3] views of the slot's flat left-image buffers (the slot is idle here)."""
        n = h * w * 3
        t = self.rgb_host[slot]
        if t is None or t.numel() < n:
            t = torch.empty((max(n, self.ch * self.cw * 3),), dtype=torch.uint8)
            self.rgb_host[slot] = t.pin_memory() if self.cuda else t
            self.rgb_dev[slot] = torch.empty(t.shape, dtype=torch.uint8, device=self.dev) if self.cuda \
                else self.rgb_host[slot]
        return self.rgb_host[slot][:n].view(h, w, 3), self.rgb_dev[slot][:n].view(h, w, 3)

    def _load_eval(self, left, right, gt_path):
        gt = read_pfm(gt_path) if str(gt_path).lower().endswith(".pfm") else read_kitti_disparity(gt_path)
        fitted, rgb, window, h, w = self._load_framed(left, right, self.mode)
        if gt.shape != (h, w):
            raise ValueError(f"{gt_path}: ground truth {gt.shape} does not match the images ({h}, {w})")
        if self.mode == "fit":
            return fitted, fit_gt_to_crop(gt, self.ch, self.cw), h, w, 0, rgb, window
        return fitted, pad_gt_to_multiple(gt, 16)[0], h, w, window[0], rgb, window

    def _wls_update(self, slot, pred, peak, lr):
        y0, x0, h, w, _ = self._pair_window
        src, label = (lr.filled, lr.label) if lr is not None else (pred, None)
        rgb = self.rgb_dev[slot][:h * w * 3].view(h, w, 3)
        ref = wls_filter(src, rgb, confidence=peak, label=label, window=self._pair_window, **self.wls)
        self.wls_meter.update(ref.disp, self.gt_dev[slot][None, y0:y0 + h, x0:x0 + w])

    def _forward_eval(self, slot):
        x = self.in_dev[slot]
        if self.lr_check:            # (pred, prob_volume, [Confidence,] LRCheck), checked in the network frame
            gt = self.gt_dev[slot][None]
            out = self.model(x[None, 0:3], x[None, 3:6], confidence=self.confidence, lr_check=True,
                             lr_threshold=self.lr_threshold)
            pred, pv, lr = out[0], out[1], out[-1]
            self.meter.update(pred, gt, pv if torch.is_tensor(pv) else None, out[2].peak if self.confidence else None,
                              calib=self._pair_calib)
            # zero GT = no GT: the inconsistent pixels leave this meter without a change to the metrics kernel
            self.lr_meters["lr_consistent"].update(pred, torch.where(lr.label.reshape(gt.shape) == 0, gt, 0.0))
            self.lr_meters["lr_filled"].update(lr.filled, gt)
            if self.wls is not None:
                self._wls_update(slot, pred, out[2].peak if self.confidence else None, lr)
            return pred.reshape(x.shape[1], x.shape[2])
        if self.confidence:          # (pred, prob_volume, Confidence(peak, std)): the peak map ranks the pixels
            pred, pv, conf = self.model(x[None, 0:3], x[None, 3:6], confidence=True)
            self.meter.update(pred, self.gt_dev[slot][None], pv if torch.is_tensor(pv) else None, conf.peak,
                              calib=self._pair_calib)
            if self.wls is not None:
                self._wls_update(slot, pred, conf.peak, None)
            return pred.reshape(x.shape[1], x.shape[2])
        out = self.model(x[None, 0:3], x[None, 3:6])
        pred, pv = (out[0], out[1]) if isinstance(out, (tuple, list)) else (out, None)
        self.meter.update(pred, self.gt_dev[slot][None], pv if torch.is_tensor(pv) else None, calib=self._pair_calib)
        if self.wls is not None:
            self._wls_update(slot, pred, None, None)
        return pred.reshape(x.shape[1], x.shape[2])

    def _crop_back(self, disp, h, w, top):
        if self.mode == "fit":
            return crop_prediction(disp, h, w, self.ch, self.cw)
        return disp[top:top + h, :w]

    def run(self, quads):
        """quads: iterable of (leftname, rightname, gt_path, savename or None).  Scores every pair into the meter in
        input order; writes the PNGs (cropped back to the image size) of the pairs with a savename."""
        import queue
        import threading
        from concurrent.futures import ThreadPoolExecutor
        quads = list(quads)
        calibs = self.calib if isinstance(self.calib, (list, tuple)) else [self.calib] * len(quads)
        if len(calibs) != len(quads):
            raise ValueError(f"{len(calibs)} calibrations for {len(quads)} pairs")
        slot_sem = threading.Semaphore(self.depth)          # a slot is reusable once the writer is done with it
        q = queue.Queue()
        err = []

        def writer():
            while True:
                item = q.get()
                if item is None:
                    return
                slot, h, w, top, savename = item
                try:
                    if self.cuda:
                        self.done[slot].synchronize()
                    if savename is not None:
                        save_disparity_png(savename, self._crop_back(self.out_host[slot].numpy(), h, w, top).copy())
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
                futs = [pool.submit(self._load_eval, l, r, g) for l, r, g, _ in quads]
                for i, (fut, quad) in enumerate(zip(futs, quads)):
                    fitted, gt, h, w, top, rgb, window = fut.result()
                    slot_sem.acquire()
                    slot = i % self.depth
                    self._ensure(slot, fitted.shape[1], fitted.shape[2])
                    np.copyto(self.in_host[slot].numpy(), fitted)
                    np.copyto(self.gt_host[slot].numpy(), gt)
                    if self.wls is not None:
                        rgb_h, rgb_d = self._rgb_slot(slot, rgb.shape[0], rgb.shape[1])
                        np.copyto(rgb_h.numpy(), rgb)
                        self._pair_window = window
                    savename = quad[3]
                    self._pair_calib = calibs[i]
                    if self.cuda:
                        with torch.cuda.stream(self.copy_stream):
                            if i >= self.depth:
                                self.copy_stream.wait_event(self.free[slot])     # kernels of the slot's previous pair
                            self.in_dev[slot].copy_(self.in_host[slot], non_blocking=True)
                            self.gt_dev[slot].copy_(self.gt_host[slot], non_blocking=True)
                            if self.wls is not None:
                                rgb_d.copy_(rgb_h, non_blocking=True)
                            self.h2d[slot].record(self.copy_stream)
                        with torch.cuda.stream(self.compute_stream):
                            self.compute_stream.wait_event(self.h2d[slot])
                            pred = self._forward_eval(slot)
                            self.free[slot].record(self.compute_stream)
                            if savename is not None:
                                self.out_host[slot].copy_(pred, non_blocking=True)
                            self.done[slot].record(self.compute_stream)
                    else:
                        pred = self._forward_eval(slot)
                        if savename is not None:
                            self.out_host[slot].copy_(pred)
                    q.put((slot, h, w, top, savename))
        finally:
            q.put(None)
            wt.join()
            if was_training and hasattr(self.model, "train"):
                self.model.train()
        if err:
            raise err[0]


WLS_KEYS = ("lam", "sigma", "num_iter", "min_support")


def evaluate_files(model, quads, mode="fit", crop=(384, 1248), depth=3, workers=2, maxdisp=None, max_valid=None,
                   confidence=False, lr_check=False, lr_threshold=1.0, calib=None, min_depth=1e-3, max_depth=80.0,
                   wls=None):
    """main_dca.py `mytest` over files: quads = (left, right, gt_path, savename or None); GT is a KITTI PNG or a PFM
    (by extension).  maxdisp defaults to model.maxdisp, max_valid as in DisparityMeter.  Returns (summary dict,
    per-image counter rows [N, METRIC_COUNT] in input order); synchronises once, at the end.  confidence=True runs
    model(left, right, confidence=True) and adds the sparsification curves of its `peak` map to the summary.

    lr_check=True runs model(left, right, lr_check=True, lr_threshold=...) (the check in the network frame, before the
    crop back); the summary keeps every key of the run without the flag and adds
      lr_consistent   summarize() of pred against the GT of the pixels labelled consistent only
      lr_filled       summarize() of the background-filled disparity against the whole GT
      lr_density      lr_consistent's n_valid / n_valid: the fraction of the valid GT pixels that pass the check
    The per-image rows returned are those of pred against the whole GT, as without the flag.

    calib (one geometry.StereoCalib, or a list aligned with quads) adds `depth`: the depth errors of summarize() with
    the GT depth fB / (gt + doffs) in [min_depth, max_depth] metres (80 m: the KITTI convention).

    wls=True (the defaults of wls.wls_filter) or a dict of its lam / sigma / num_iter / min_support adds `wls`:
    summarize() of the refined disparity of the image window against the GT of the window.  The refinement uses the
    left image, Confidence.peak when confidence=True, and LRCheck.filled with LRCheck.label when lr_check=True."""
    if wls is not None and wls is not False:
        wls = {} if wls is True else dict(wls)
        bad = set(wls) - set(WLS_KEYS)
        if bad:
            raise ValueError(f"wls: unknown keys {sorted(bad)}, expected a subset of {WLS_KEYS}")
    else:
        wls = None
    if maxdisp is None:
        maxdisp = getattr(model, "maxdisp", 192)
    try:
        dev = next(model.parameters()).device
    except (StopIteration, AttributeError):
        dev = torch.device("cpu")
    meter = DisparityMeter(maxdisp, max_valid, dev, min_depth=min_depth, max_depth=max_depth)
    pipe = EvalPipeline(model, meter, mode, crop[0], crop[1], depth, workers, confidence, lr_check, lr_threshold,
                        calib, wls)
    pipe.run(quads)
    rows = meter.rows()
    h = meter.sparsification_histograms()
    summary = summarize(rows, meter.confusion() if meter._has_conf else None, *(h or (None, None)),
                        depth_rows=meter.depth_rows())
    if lr_check:
        for k, m in pipe.lr_meters.items():
            summary[k] = summarize(m.rows())
        n = summary["n_valid"]
        summary["lr_density"] = summary["lr_consistent"]["n_valid"] / n if n else float("nan")
    if wls is not None:
        summary["wls"] = summarize(pipe.wls_meter.rows())
    return summary, rows
