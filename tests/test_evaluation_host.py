"""CPU: evaluation against ground truth (evaluation.py): GT readers, GT framing, summary formulas, the metric definitions
against the GwcNet formulas, and the evaluate_files pipeline with the kernel calls replaced by their CPU restatements
(tests/_eval_restatement.py)."""
import importlib
import math

import numpy as np
import pytest
import torch
from PIL import Image

import _eval_restatement as O
from test_kitti_io import _FakeStereo, _rgb

ev = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.evaluation")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")


def _write_pfm(path, a, little=True, header=b"Pf"):
    a = np.asarray(a, np.float32)
    with open(path, "wb") as f:
        f.write(header + b"\n%d %d\n%s\n" % (a.shape[1], a.shape[0], b"-1.0" if little else b"1.0"))
        f.write(np.ascontiguousarray(a[::-1]).astype("<f4" if little else ">f4").tobytes())


# ---- readers -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("little", [True, False])
def test_read_pfm_round_trips_both_byte_orders_bottom_up_rows_and_inf(tmp_path, little):
    a = np.random.default_rng(1).uniform(0, 200, (7, 11)).astype(np.float32)
    a[0, 0], a[3, 4], a[6, 10] = np.inf, 0.0, 1e-3
    _write_pfm(tmp_path / "d.pfm", a, little)
    back = ev.read_pfm(str(tmp_path / "d.pfm"))
    assert back.dtype == np.float32 and back.shape == (7, 11)
    assert np.array_equal(back, a)                          # row 0 of the result = top row (stored last)
    assert np.isinf(back[0, 0])


def test_read_pfm_rejects_three_channel_and_garbage(tmp_path):
    _write_pfm(tmp_path / "c.pfm", np.zeros((2, 3)), header=b"PF")
    with pytest.raises(ValueError, match="3-channel"):
        ev.read_pfm(str(tmp_path / "c.pfm"))
    (tmp_path / "x.pfm").write_bytes(b"P6\n1 1\n255\n\0\0\0")
    with pytest.raises(ValueError):
        ev.read_pfm(str(tmp_path / "x.pfm"))


def test_read_kitti_disparity_round_trips_save_disparity_png(tmp_path):
    disp = np.random.default_rng(2).uniform(0, 250, (13, 29)).astype(np.float32)
    disp[2, 3] = 0.0
    stored = io.save_disparity_png(str(tmp_path / "d.png"), disp)
    back = ev.read_kitti_disparity(str(tmp_path / "d.png"))
    assert back.dtype == np.float32 and back[2, 3] == 0.0
    assert np.array_equal(back, stored.astype(np.float32) / 256.0)
    assert float(np.abs(back - disp).max()) < 1.0 / 256.0


# ---- framing -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h,w", [(37, 53), (48, 64), (60, 70)])
def test_fit_mode_gt_marker_lands_under_its_image_pixel(h, w):
    y, x = h - 20, w // 2                     # inside the crop window in every case
    pair = np.zeros((6, h, w), np.float32)
    pair[:, y, x] = 1.0
    gt = np.full((h, w), 5.0, np.float32)
    gt[y, x] = 77.0
    left, _, _, _ = io.fit_to_crop(pair, 48, 64)
    g = io.fit_gt_to_crop(gt, 48, 64)
    assert g.shape == (48, 64) and g.dtype == np.float32
    assert np.argwhere(left[0, 0].numpy() == 1.0).tolist() == np.argwhere(g == 77.0).tolist()
    if h <= 48 and w <= 64:                    # padded: everything outside the image reads as invalid (0)
        inside = np.zeros((48, 64), bool)
        inside[48 - h:, :w] = True
        assert (g[~inside] == 0).all() and not O.gt_valid_mask(g[~inside], 0).any()
        assert (g[inside] > 0).all()


@pytest.mark.parametrize("h,w", [(37, 53), (48, 64), (17, 80)])
def test_pad16_mode_gt_marker_lands_under_its_image_pixel(h, w):
    y, x = h // 3, w - 2
    pair = np.zeros((6, h, w), np.float32)
    pair[:, y, x] = 1.0
    gt = np.full((h, w), 5.0, np.float32)
    gt[y, x] = 77.0
    img, top, right = io.pad_to_multiple(torch.from_numpy(pair)[None], 16)
    g, gtop, gright = io.pad_gt_to_multiple(gt, 16)
    assert (gtop, gright) == (top, right) and g.shape == tuple(img.shape[2:]) and g.shape[0] % 16 == g.shape[1] % 16 == 0
    assert np.argwhere(img[0, 0].numpy() == 1.0).tolist() == np.argwhere(g == 77.0).tolist()
    assert (g[:top] == 0).all() and (g[:, w:] == 0).all() and (g[top:, :w] > 0).all()


# ---- summary -------------------------------------------------------------------------------------------
def _row(valid, epe_px_sum, gt1, gt2, gt3, d1, nonfinite=0):
    return [valid, int(round(epe_px_sum * 2 ** 20)), gt1, gt2, gt3, d1, nonfinite]


def test_summary_image_mean_and_pixel_pooled():
    rows = np.array([_row(100, 50.0, 10, 5, 2, 1),       # EPE 0.5, bad1 0.10, bad3 0.02, d1 0.01
                     _row(0, 0.0, 0, 0, 0, 0),           # no valid pixels: skipped, counted
                     _row(300, 300.0, 60, 30, 30, 3)],   # EPE 1.0, bad1 0.20, bad3 0.10, d1 0.01
                    np.uint64)
    s = ev.summarize(rows)
    assert s["n_images"] == 3 and s["n_images_skipped"] == 1 and s["n_valid"] == 400 and s["n_pred_nonfinite"] == 0
    assert s["epe"] == pytest.approx(0.75) and s["bad1"] == pytest.approx(0.15)
    assert s["bad2"] == pytest.approx((0.05 + 0.1) / 2) and s["bad3"] == pytest.approx(0.06)
    assert s["d1"] == pytest.approx(0.01)
    assert s["epe_pooled"] == pytest.approx(350.0 / 400) and s["bad1_pooled"] == pytest.approx(70 / 400)
    assert s["bad3_pooled"] == pytest.approx(32 / 400) and s["d1_pooled"] == pytest.approx(4 / 400)
    assert "miou" not in s


def test_summary_non_finite_predictions_are_errors_and_leave_the_epe():
    s = ev.summarize(np.array([_row(10, 4.0, 3, 2, 2, 2, nonfinite=2)], np.uint64))
    assert s["n_pred_nonfinite"] == 2 and s["epe"] == pytest.approx(4.0 / 8) and s["bad1"] == pytest.approx(0.3)
    empty = ev.summarize(np.zeros((0, ev.METRIC_COUNT), np.uint64))
    assert empty["n_images"] == 0 and math.isnan(empty["epe"]) and math.isnan(empty["d1_pooled"])


def test_summary_confusion_matrix_evaluator_formulas():
    cm = np.array([[5, 1, 0, 0],
                   [2, 2, 0, 0],
                   [0, 0, 0, 0],     # class 2: neither GT nor predictions -> nan, left out of both means
                   [0, 3, 0, 0]],    # class 3: GT only, never predicted -> Acc 0, IoU 0
                  np.uint64)
    s = ev.summarize(np.array([_row(1, 0.0, 0, 0, 0, 0)], np.uint64), cm)
    assert s["pixel_accuracy"] == pytest.approx(7 / 13) and s["n_class_pixels"] == 13
    assert s["mpa"] == pytest.approx((5 / 6 + 2 / 4 + 0.0) / 3)
    iou = [5 / (6 + 7 - 5), 2 / (4 + 6 - 2), 0.0]
    assert s["miou"] == pytest.approx(sum(iou) / 3)


def test_meter_rejects_cpu_tensors_without_a_kernel():
    m = ev.DisparityMeter(48, device="cpu")
    with pytest.raises(_lib.DcaError):
        m.update(torch.zeros(1, 1, 16, 16), torch.ones(1, 16, 16))


# ---- the metric definitions against the GwcNet formulas --------------------------------------------------
def test_restatement_agrees_with_the_gwcnet_formulas():
    g = torch.Generator().manual_seed(3)
    B, H, W, maxdisp = 3, 20, 33, 48
    gt = torch.rand(B, H, W, generator=g) * 60 - 5              # negatives, zeros after rounding, >= maxdisp
    gt[0, :4] = 0.0
    pred = gt + torch.randn(B, H, W, generator=g) * 3
    pred[1, 2, :5] = gt[1, 2, :5] + torch.tensor([1.0, 2.0, 3.0, -3.0, 0.5])   # exactly on the thresholds
    rows = O.disparity_metric_counts(pred, gt, maxdisp)
    for b in range(B):
        mask = (gt[b] > 0) & (gt[b] < maxdisp)                     # GwcNet test loop
        E = (gt[b] - pred[b]).abs()[mask]
        assert rows[b, ev.VALID] == int(mask.sum())
        epe = torch.nn.functional.l1_loss(pred[b][mask], gt[b][mask]).item()          # EPE_metric
        assert rows[b, ev.SUM_ABS] * 2.0 ** -20 / rows[b, ev.VALID] == pytest.approx(epe, rel=1e-5)
        for t, col in ((1, ev.GT1), (2, ev.GT2), (3, ev.GT3)):                        # Thres_metric
            assert rows[b, col] == int((E > t).sum())
        d1 = (E > 3) & (E / gt[b][mask].abs() > 0.05)                                  # D1_metric
        assert rows[b, ev.D1] == int(d1.sum())
        assert rows[b, ev.PRED_NONFINITE] == 0


# ---- evaluate_files on the CPU with the kernels replaced by their restatements ----------------------------
class _FakeStereoLogits(_FakeStereo):
    """_FakeStereo with a 6-class 1/8-res 'prob_volume': logits[k] = -|d - 8k| at every 8th pixel."""

    def forward(self, left, right, disp_true=None):
        d, d8 = super().forward(left, right)
        k = torch.arange(6.0).view(1, 6, 1, 1)
        return d, -(d8 * 10.0 - 8.0 * k).abs()


def _patch_kernels(monkeypatch):
    monkeypatch.setattr(ev, "_disparity_metrics", lambda pred, gt, rows, mv: rows.add_(
        torch.from_numpy(O.disparity_metric_counts(pred, gt, mv))))
    monkeypatch.setattr(ev, "_class_confusion", lambda lg, gt, conf, mv: conf.add_(
        torch.from_numpy(O.class_confusion(lg, gt, lg.shape[1], mv))))


def _gt_file(tmp_path, i, h, w):
    gt = np.random.default_rng(100 + i).uniform(0, 60, (h, w)).astype(np.float32)
    gt[: h // 5] = 0.0
    if i % 2:
        _write_pfm(tmp_path / f"g{i}.pfm", gt, little=bool(i % 4 == 1))
        return str(tmp_path / f"g{i}.pfm")
    io.save_disparity_png(str(tmp_path / f"g{i}.png"), gt)
    return str(tmp_path / f"g{i}.png")


@pytest.mark.parametrize("mode", ["fit", "pad16"])
def test_evaluate_files_equals_a_serial_loop(tmp_path, monkeypatch, mode):
    """More pairs than slots, mixed sizes (padded, exact, cropped), PNG and PFM ground truth: per-pair rows, the
    confusion matrix and the written PNGs equal a plain serial loop."""
    _patch_kernels(monkeypatch)
    sizes = [(37, 53), (48, 64), (60, 70), (20, 64), (48, 30), (37, 53), (52, 80)]
    model = _FakeStereoLogits().eval()
    quads, ref_rows, ref_conf = [], [], np.zeros((6, 6), np.int64)
    for i, (h, w) in enumerate(sizes):
        Image.fromarray(_rgb(10 + i, h, w)).save(tmp_path / f"l{i}.png")
        Image.fromarray(_rgb(50 + i, h, w)).save(tmp_path / f"r{i}.png")
        quads.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"), _gt_file(tmp_path, i, h, w),
                      str(tmp_path / f"p{i}.png") if i % 3 else None))
        gt = ev.read_pfm(quads[-1][2]) if quads[-1][2].endswith(".pfm") else ev.read_kitti_disparity(quads[-1][2])
        pair = io.load_pair(quads[-1][0], quads[-1][1])
        if mode == "fit":
            left, right, _, _ = io.fit_to_crop(pair, 48, 64)
            gt = io.fit_gt_to_crop(gt, 48, 64)
        else:
            x, top, _ = io.pad_to_multiple(torch.from_numpy(pair)[None], 16)
            left, right = x[:, 0:3], x[:, 3:6]
            gt = io.pad_gt_to_multiple(gt, 16)[0]
        with torch.no_grad():
            pred, logits = model(left, right)
        ref_rows.append(O.disparity_metric_counts(pred, gt[None], 48)[0])
        ref_conf += O.class_confusion(logits, gt[None], 6, 48)
        if quads[-1][3]:
            disp = pred[0, 0].numpy()
            disp = io.crop_prediction(disp, h, w, 48, 64) if mode == "fit" else disp[top:top + h, :w]
            io.save_disparity_png(str(tmp_path / f"q{i}.png"), disp)
    summary, rows = ev.evaluate_files(model, quads, mode=mode, crop=(48, 64), depth=2, workers=3, maxdisp=48)
    assert rows.dtype == np.uint64 and rows.shape == (len(sizes), ev.METRIC_COUNT)
    assert np.array_equal(rows.astype(np.int64), np.stack(ref_rows))
    assert summary == ev.summarize(np.stack(ref_rows).astype(np.uint64), ref_conf)
    assert summary["n_images"] == len(sizes) and summary["n_valid"] > 0 and summary["n_class_pixels"] > 0
    for i, q in enumerate(quads):
        if q[3]:
            assert np.array_equal(np.asarray(Image.open(q[3])), np.asarray(Image.open(tmp_path / f"q{i}.png")))


def test_evaluate_files_rejects_ground_truth_of_another_size(tmp_path, monkeypatch):
    _patch_kernels(monkeypatch)
    Image.fromarray(_rgb(1, 20, 30)).save(tmp_path / "l.png")
    Image.fromarray(_rgb(2, 20, 30)).save(tmp_path / "r.png")
    io.save_disparity_png(str(tmp_path / "g.png"), np.ones((21, 30), np.float32))
    with pytest.raises(ValueError, match="ground truth"):
        ev.evaluate_files(_FakeStereoLogits(), [(str(tmp_path / "l.png"), str(tmp_path / "r.png"),
                                                 str(tmp_path / "g.png"), None)], crop=(32, 32), maxdisp=48)


def test_entry_points_reject_bad_arguments_without_a_device():
    """DCA_ERR_ARG for NULL pointers / empty shapes / NaN bound, DCA_ERR_UNSUPPORTED for D8 > 64: returned before any CUDA
    call, so this runs without a GPU."""
    import os
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    assert lib.dca_disparity_metrics(None, p, p, 1, 4, 4, 0.0, None) == -1
    assert lib.dca_disparity_metrics(p, p, p, 0, 4, 4, 0.0, None) == -1
    assert lib.dca_disparity_metrics(p, p, p, 1, 4, 4, float("nan"), None) == -1
    assert lib.dca_class_confusion(p, None, p, 1, 6, 2, 2, 0.0, None) == -1
    assert lib.dca_class_confusion(p, p, p, 1, 6, 0, 2, 0.0, None) == -1
    assert lib.dca_class_confusion(p, p, p, 1, 65, 2, 2, 0.0, None) == -3
