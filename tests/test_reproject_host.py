"""CPU: metric depth and point clouds (geometry.py).  The calibration readers on synthetic KITTI (both key styles) and
Middlebury files, a velodyne point through P2 / P3 and back through the float32 restatement
(tests/_reproject_restatement.py), the restatement against a float64 closed form, the PLY and depth-PNG writers, the depth
errors of summarize() against numpy, the calib-or-none rule of the meter, reproject_files and evaluate_files(calib=...)
with the kernels replaced by their restatements, the dry-run launch sequence, and the entry points' argument checks."""
import importlib
import math
import os

import numpy as np
import pytest
import torch
from PIL import Image

import _dryrun
import _eval_restatement as O
import _reproject_restatement as R
from test_evaluation_host import _FakeStereoLogits, _gt_file, _patch_kernels
from test_kitti_io import _rgb

geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
ev = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.evaluation")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")


# ---- calibration -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("style", ["object", "cam_to_cam"])
def test_read_kitti_calib_q_baseline_and_rect_to_velo(tmp_path, style):
    s = R.kitti_scene()
    R.write_kitti_calib(tmp_path / "calib.txt", s, style)
    c = geo.read_kitti_calib(str(tmp_path / "calib.txt"))
    B = s["t2"][0] - s["t3"][0]
    assert (c.fx, c.fy, c.cx, c.cy, c.doffs) == pytest.approx((s["fx"], s["fy"], s["cx"], s["cy"], 0.0), rel=1e-12)
    assert c.baseline == pytest.approx(B, rel=1e-9) and c.focal_baseline == pytest.approx(s["fx"] * B, rel=1e-9)
    want_q = np.array([[1, 0, 0, -s["cx"]], [0, 1, 0, -s["cy"]], [0, 0, 0, s["fx"]], [0, 0, 1 / B, 0]], np.float32)
    assert c.Q().dtype == np.float32 and np.allclose(c.Q(), want_q, rtol=1e-6, atol=0)
    if style == "cam_to_cam":
        assert c.rect_to_velo is None
        return
    # by hand: velo = Rv^T (R0^T (x - (t2x, t2y, 0)) - tv)
    Rv, tv, R0, t2 = s["Rv"], s["tv"], s["R0_rect"], s["t2"]
    M = Rv.T @ R0.T
    want = np.hstack([M, (-M @ np.array([t2[0], t2[1], 0.0]) - Rv.T @ tv)[:, None]])
    assert c.rect_to_velo.dtype == np.float32 and c.rect_to_velo.shape == (3, 4)
    np.testing.assert_allclose(c.rect_to_velo, want, rtol=0, atol=1e-6)


def test_read_middlebury_calib(tmp_path):
    (tmp_path / "calib.txt").write_text(
        "cam0=[3979.911 0 1244.772; 0 3979.911 1019.507; 0 0 1]\ncam1=[3979.911 0 1369.115; 0 3979.911 1019.507; 0 0 1]\n"
        "doffs=124.343\nbaseline=193.001\nwidth=2964\nheight=1988\nndisp=270\nisint=0\nvmin=23\nvmax=245\n")
    c = geo.read_middlebury_calib(str(tmp_path / "calib.txt"))
    assert (c.fx, c.fy, c.cx, c.cy) == (3979.911, 3979.911, 1244.772, 1019.507)
    assert c.baseline == pytest.approx(0.193001) and c.doffs == 124.343 and c.rect_to_velo is None
    # Z = f B / (d + doffs): the Middlebury depth formula in metres
    d = np.float32(150.0)
    _, P, Z = R.keep_and_points(np.full((1, 1, 1), d, np.float32), None, None, 1244, 1019, c.Q(), None, 0, 0, np.inf)
    assert float(Z[0, 0, 0]) == pytest.approx(3979.911 * 0.193001 / (150.0 + 124.343), rel=1e-6)


@pytest.mark.parametrize("frame", ["camera", "velodyne"])
def test_a_velodyne_point_through_p2_p3_comes_back(tmp_path, frame):
    """Integer pixels (u, v) of camera 2 at depths z: the velodyne point behind each (float64), its P2 / P3 projections
    (the disparity), then the restatement from the disparity map back to the camera / velodyne frame."""
    s = R.kitti_scene()
    R.write_kitti_calib(tmp_path / "calib.txt", s)
    c = geo.read_kitti_calib(str(tmp_path / "calib.txt"))
    rng = np.random.default_rng(5)
    H, W = 40, 96
    disp = np.full((1, H, W), np.nan, np.float32)
    pts = {}
    for _ in range(60):
        v, u, z = int(rng.integers(0, H)), int(rng.integers(0, W)), float(rng.uniform(2.0, 60.0))
        u_img, v_img = u + 500, v + 150                                  # a window inside a KITTI-size image
        rect = np.array([(u_img - s["cx"]) * z / s["fx"] - s["t2"][0], (v_img - s["cy"]) * z / s["fy"] - s["t2"][1], z])
        velo = s["Rv"].T @ (s["R0_rect"].T @ rect - s["tv"])
        cam0 = s["R0_rect"] @ (s["Tr_velo_to_cam"] @ np.append(velo, 1.0))
        p2, p3 = s["P2"] @ np.append(cam0, 1.0), s["P3"] @ np.append(cam0, 1.0)
        assert abs(p2[0] / p2[2] - u_img) < 1e-9 and abs(p2[1] / p2[2] - v_img) < 1e-9
        disp[0, v, u] = p2[0] / p2[2] - p3[0] / p3[2]
        pts[v * W + u] = (rect + np.array([s["t2"][0], s["t2"][1], 0.0]), velo)
    T = c.rect_to_velo if frame == "velodyne" else None
    xyz, index, count, depth = R.reproject(disp, u0=500, v0=150, Q=c.Q(), T=T)
    assert count[0] == len(pts) and np.array_equal(index[0], sorted(pts))
    for i, p in zip(index[0], xyz[0]):
        want = pts[int(i)][1 if frame == "velodyne" else 0]
        np.testing.assert_allclose(p, want, rtol=2e-6, atol=2e-5)
        assert depth[0].ravel()[i] == pytest.approx(pts[int(i)][0][2], rel=2e-6)
    assert (depth[0].ravel()[np.setdiff1d(np.arange(H * W), index[0])] == 0).all()


# ---- the restatement ---------------------------------------------------------------------------------------------
def test_restatement_against_the_float64_closed_form():
    rng = np.random.default_rng(0)
    c = geo.StereoCalib(1000.0, 980.0, 60.5, 20.25, 0.3, doffs=2.5)
    B, H, W = 2, 23, 61
    d = rng.uniform(-5, 120, (B, H, W)).astype(np.float32)
    d[0, 0, :6] = [np.nan, np.inf, -np.inf, 0.0, -2.5, -3.0]                  # -2.5: W' = 0
    peak = rng.uniform(0, 1, (B, H, W)).astype(np.float32)
    label = rng.integers(0, 4, (B, H, W)).astype(np.uint8)
    xyz, index, count, depth = R.reproject(d, peak, label, 7, 3, c.Q(), None, 0.3, 2.0, 90.0)
    d64 = d.astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        Z = 1000.0 * 0.3 / (d64 + 2.5)
        X = (np.arange(W) + 7 - 60.5) * Z / 1000.0
        Y = (np.arange(H)[:, None] + 3 - 20.25) * Z / 980.0
        keep = np.isfinite(d64) & (d64 + 2.5 > 0) & (Z >= 2.0) & (Z <= 90.0) & (peak >= np.float32(0.3)) & (label == 0)
    near = np.abs(Z - 2.0) < 1e-4 * 2.0
    near |= np.abs(Z - 90.0) < 1e-4 * 90.0
    for b in range(B):
        kb = keep[b] & ~near[b]
        got = np.zeros(H * W, bool)
        got[index[b]] = True
        assert np.array_equal(got[~near[b].ravel()], kb[~near[b]].ravel())
        assert np.array_equal(index[b], np.flatnonzero(got))                  # row-major order
        want = np.stack([X[b].ravel(), Y[b].ravel(), Z[b].ravel()], -1)[index[b]]
        np.testing.assert_allclose(xyz[b], want, rtol=3e-6, atol=1e-6)
        assert count[b] == len(index[b]) > 0
        assert np.array_equal(depth[b].ravel() != 0, got)
    assert not np.isin(np.arange(6), index[0]).any()


# ---- writers ---------------------------------------------------------------------------------------------------
def _read_ply(path):
    raw = open(path, "rb").read()
    head, _, body = raw.partition(b"end_header\n")
    lines = head.decode().splitlines()
    n = int([l for l in lines if l.startswith("element vertex")][0].split()[-1])
    props = [(l.split()[2], "<f4" if l.split()[1] == "float" else "u1") for l in lines if l.startswith("property")]
    assert "format binary_little_endian 1.0" in lines
    return np.frombuffer(body, dtype=props, count=n), props


@pytest.mark.parametrize("with_rgb", [True, False])
def test_ply_reads_back(tmp_path, with_rgb):
    rng = np.random.default_rng(1)
    xyz = rng.normal(0, 10, (57, 3)).astype(np.float32)
    rgb = rng.integers(0, 256, (57, 3), dtype=np.uint8) if with_rgb else None
    geo.save_ply(str(tmp_path / "p.ply"), xyz, rgb)
    v, props = _read_ply(str(tmp_path / "p.ply"))
    assert [p[0] for p in props] == ["x", "y", "z"] + (["red", "green", "blue"] if with_rgb else [])
    assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], -1), xyz)
    if with_rgb:
        assert np.array_equal(np.stack([v["red"], v["green"], v["blue"]], -1), rgb)
    geo.save_ply(str(tmp_path / "e.ply"), np.zeros((0, 3), np.float32))
    assert len(_read_ply(str(tmp_path / "e.ply"))[0]) == 0


def test_depth_png_reads_back(tmp_path):
    depth = np.array([[0.0, 1.0, 80.0], [255.99, 300.0, np.inf]], np.float32)
    stored = geo.save_depth_png(str(tmp_path / "d.png"), depth)
    back = np.asarray(Image.open(tmp_path / "d.png"))
    assert back.dtype == np.uint16 and np.array_equal(back, stored)
    assert back.tolist() == [[0, 256, 20480], [65533, 65535, 65535]]


# ---- depth errors ----------------------------------------------------------------------------------------------
def _depth_case(seed, B=3, H=17, W=29):
    rng = np.random.default_rng(seed)
    gt = rng.uniform(-2, 200, (B, H, W)).astype(np.float32)
    gt[0, 0, :3] = [0.0, np.nan, np.inf]
    pred = (gt * rng.uniform(0.7, 1.4, gt.shape)).astype(np.float32)
    pred[1, 0, :4] = [np.nan, np.inf, -5.0, 0.0]
    return pred, gt


def test_depth_summary_against_numpy():
    pred, gt = _depth_case(2)
    fb, doffs, lo, hi = 721.5 * 0.54, 0.0, 1e-3, 80.0
    rows, _ = R.depth_metrics(pred, gt, 192.0, fb, doffs, lo, hi)
    s = ev.summarize(O.disparity_metric_counts(pred, gt, 192.0).astype(np.uint64), depth_rows=rows.astype(np.uint64))
    dep = s["depth"]
    per = {k: [] for k in ("abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3")}
    allz = []
    for b in range(gt.shape[0]):
        g, p = gt[b].astype(np.float64), pred[b].astype(np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            zg = fb / (g + doffs)
            m = np.isfinite(g) & (g > 0) & (g < 192) & (zg >= lo) & (zg <= hi)
            zp = np.where(np.isfinite(p + doffs) & (p + doffs > 0), fb / (p + doffs), hi)
        zp, zg = np.clip(zp[m], lo, hi), zg[m]
        allz.append((zp, zg))
        t = np.maximum(zp / zg, zg / zp)
        per["abs_rel"].append(np.mean(np.abs(zp - zg) / zg))
        per["sq_rel"].append(np.mean((zp - zg) ** 2 / zg))
        per["rmse"].append(np.sqrt(np.mean((zp - zg) ** 2)))
        per["rmse_log"].append(np.sqrt(np.mean((np.log(zp) - np.log(zg)) ** 2)))
        for k, thr in (("a1", 1.25), ("a2", 1.25 ** 2), ("a3", 1.25 ** 3)):
            per[k].append(np.mean(t < thr))
    zp, zg = (np.concatenate([a[i] for a in allz]) for i in (0, 1))
    pooled = {"abs_rel": np.mean(np.abs(zp - zg) / zg), "sq_rel": np.mean((zp - zg) ** 2 / zg),
              "rmse": np.sqrt(np.mean((zp - zg) ** 2)), "rmse_log": np.sqrt(np.mean((np.log(zp) - np.log(zg)) ** 2)),
              "a1": np.mean(np.maximum(zp / zg, zg / zp) < 1.25)}
    assert dep["n_valid"] == len(zp) > 0
    for k, v in per.items():
        assert dep[k] == pytest.approx(np.mean(v), rel=1e-5, abs=1e-6), k
    for k, v in pooled.items():
        assert dep[k + "_pooled"] == pytest.approx(v, rel=1e-5, abs=1e-6), k
    assert 0 < dep["a1"] <= dep["a2"] <= dep["a3"] <= 1
    assert set(s) - set(ev.summarize(O.disparity_metric_counts(pred, gt, 192.0).astype(np.uint64))) == {"depth"}


def _patch_depth(monkeypatch):
    monkeypatch.setattr(ev, "_depth_metrics", lambda pred, gt, rows, mv, fb, doffs, lo, hi: rows.add_(
        torch.from_numpy(R.depth_metrics(pred, gt, mv, fb, doffs, lo, hi)[0])))


def test_meter_takes_a_calibration_with_every_update_or_none(monkeypatch):
    _patch_kernels(monkeypatch)
    _patch_depth(monkeypatch)
    c = geo.StereoCalib(700.0, 700.0, 10.0, 10.0, 0.5)
    pred, gt = (torch.from_numpy(a) for a in _depth_case(3, B=2))
    m = ev.DisparityMeter(192, device="cpu", capacity=1)
    m.update(pred, gt, calib=c)
    m.update(pred, gt, calib=c)                       # the row tables grow together
    with pytest.raises(ValueError, match="calib"):
        m.update(pred, gt)
    assert len(m) == 4 and m.depth_rows().shape == (4, ev.DEPTH_COUNT)
    want = R.depth_metrics(pred, gt, 192.0, c.focal_baseline, 0.0, 1e-3, 80.0)[0]
    assert np.array_equal(m.depth_rows().astype(np.int64), np.concatenate([want, want]))
    assert m.summary()["depth"] == ev.summarize(m.rows(), depth_rows=m.depth_rows())["depth"]
    plain = ev.DisparityMeter(192, device="cpu")
    plain.update(pred, gt)
    with pytest.raises(ValueError, match="calib"):
        plain.update(pred, gt, calib=c)
    assert plain.depth_rows() is None and "depth" not in plain.summary()


# ---- files in, point clouds out, with the kernel replaced by its restatement ---------------------------------------
def _restated_kernel(disp, peak, label, u0, v0, Q, T, min_peak, min_depth, max_depth):
    xyz, index, count, depth = R.reproject(disp, None if peak is None else peak.numpy(),
                                           None if label is None else label.numpy(), u0, v0, Q, T, min_peak,
                                           min_depth, max_depth)
    B, H, W = disp.shape
    X, I = torch.zeros(B, H * W, 3), torch.zeros(B, H * W, dtype=torch.int32)
    for b in range(B):
        X[b, :count[b]] = torch.from_numpy(xyz[b])
        I[b, :count[b]] = torch.from_numpy(index[b])
    return geo.PointCloud(X, I, torch.from_numpy(count), torch.from_numpy(depth))


class _FakeStereoFilters(_FakeStereoLogits):
    """_FakeStereoLogits with GwcNet's confidence and lr_check outputs (fixed functions of the disparity)."""

    def forward(self, left, right, disp_true=None, confidence=False, lr_check=False, lr_threshold=1.0):
        import dcanet_b200 as d
        disp, lg = super().forward(left, right)
        out = [disp, lg]
        if confidence:
            peak = torch.sigmoid(torch.sin(disp * 3.0) * 4.0)
            out.append(d.Confidence(peak, 1.0 - peak))
        if lr_check:
            label = (((disp * 10).long() % 3) != 0).to(torch.uint8)
            out.append(d.LRCheck(disp, label, disp))
        return tuple(out)


def _frame(pair, mode, ch, cw):
    """(left, right [1,3,..], window) as the pipeline frames a pair."""
    _, h, w = pair.shape
    if mode == "pad16":
        x, top, _ = io.pad_to_multiple(torch.from_numpy(pair)[None], 16)
        return x[:, 0:3], x[:, 3:6], (top, 0, h, w, 0)
    left, right, _, _ = io.fit_to_crop(pair, ch, cw)
    if h <= ch and w <= cw:
        return left, right, (ch - h, 0, h, w, 0)
    return left, right, (0, 0, ch, cw, int((h - ch) / 2))


@pytest.mark.parametrize("mode", ["fit", "pad16"])
@pytest.mark.parametrize("filters", [False, True])
def test_reproject_files_equals_a_serial_loop(tmp_path, monkeypatch, mode, filters):
    monkeypatch.setattr(geo, "_reproject_kernel", _restated_kernel)
    sizes = [(37, 53), (48, 64), (60, 70), (20, 64), (37, 53)]
    model = _FakeStereoFilters().eval()
    calibs = [geo.StereoCalib(50.0 + i, 52.0, 30.0, 20.0, 0.5, doffs=0.25 * i) for i in range(len(sizes))]
    items, ref = [], []
    kw = dict(min_confidence=0.4, lr_check=True) if filters else {}
    for i, (h, w) in enumerate(sizes):
        rgb = _rgb(10 + i, h, w)
        Image.fromarray(rgb).save(tmp_path / f"l{i}.png")
        Image.fromarray(_rgb(50 + i, h, w)).save(tmp_path / f"r{i}.png")
        items.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"),
                      str(tmp_path / f"p{i}.ply") if i % 2 == 0 else None, str(tmp_path / f"d{i}.png") if i else None))
        left, right, (y0, x0, hh, ww, vo) = _frame(io.load_pair(items[-1][0], items[-1][1]), mode, 48, 64)
        with torch.no_grad():
            out = model(left, right, confidence=filters, lr_check=filters)
        win = lambda t: t[:, 0, y0:y0 + hh, x0:x0 + ww].numpy()
        xyz, index, count, depth = R.reproject(win(out[0]), win(out[2].peak) if filters else None,
                                               win(out[3].label) if filters else None, x0, vo, calibs[i].Q(), None,
                                               0.4 if filters else 0.0, 0.0, np.inf)
        col = rgb[vo:vo + hh, x0:x0 + ww].reshape(-1, 3)[index[0]]
        ref.append((xyz[0], col, depth[0]))
    got = geo.reproject_files(model, items, calibs, mode=mode, crop=(48, 64), depth=2, workers=3, **kw)
    assert len(got) == len(items)
    for i, ((gx, gc), (rx, rc, rd)) in enumerate(zip(got, ref)):
        assert np.array_equal(gx, rx) and np.array_equal(gc, rc) and len(gx) > 0, i
        if items[i][2]:
            v, _ = _read_ply(items[i][2])
            assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], -1), rx)
            assert np.array_equal(np.stack([v["red"], v["green"], v["blue"]], -1), rc)
        if items[i][3]:
            assert np.array_equal(np.asarray(Image.open(items[i][3])), geo.save_depth_png(str(tmp_path / "x.png"), rd))
    if filters:
        plain = geo.reproject_files(model, items[:2], calibs[:2], mode=mode, crop=(48, 64), depth=2)
        assert all(len(p[0]) > len(g[0]) for p, g in zip(plain, got[:2]))


@pytest.mark.parametrize("mode", ["fit", "pad16"])
def test_evaluate_files_with_a_calibration_equals_a_serial_loop(tmp_path, monkeypatch, mode):
    _patch_kernels(monkeypatch)
    _patch_depth(monkeypatch)
    sizes = [(37, 53), (48, 64), (60, 70)]
    model = _FakeStereoLogits().eval()
    calibs = [geo.StereoCalib(700.0 + 10 * i, 700.0, 30.0, 20.0, 0.54, doffs=0.5 * i) for i in range(len(sizes))]
    quads, rows, drows = [], [], []
    for i, (h, w) in enumerate(sizes):
        Image.fromarray(_rgb(10 + i, h, w)).save(tmp_path / f"l{i}.png")
        Image.fromarray(_rgb(50 + i, h, w)).save(tmp_path / f"r{i}.png")
        quads.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"), _gt_file(tmp_path, i, h, w), None))
        gt = ev.read_pfm(quads[-1][2]) if quads[-1][2].endswith(".pfm") else ev.read_kitti_disparity(quads[-1][2])
        pair = io.load_pair(quads[-1][0], quads[-1][1])
        left, right, _ = _frame(pair, mode, 48, 64)
        gt = io.fit_gt_to_crop(gt, 48, 64) if mode == "fit" else io.pad_gt_to_multiple(gt, 16)[0]
        with torch.no_grad():
            pred, _ = model(left, right)
        rows.append(O.disparity_metric_counts(pred, gt[None], 48)[0])
        drows.append(R.depth_metrics(pred, gt[None], 48.0, calibs[i].focal_baseline, calibs[i].doffs, 1e-3, 50.0)[0][0])
    kw = dict(mode=mode, crop=(48, 64), depth=2, workers=2, maxdisp=48)
    summary, got = ev.evaluate_files(model, quads, calib=calibs, max_depth=50.0, **kw)
    plain, plain_rows = ev.evaluate_files(model, quads, **kw)
    assert np.array_equal(got, plain_rows) and np.array_equal(got.astype(np.int64), np.stack(rows))
    assert {k: v for k, v in summary.items() if k != "depth"} == plain
    assert summary["depth"] == ev.summarize(got, depth_rows=np.stack(drows).astype(np.uint64))["depth"]
    assert summary["depth"]["n_valid"] > 0
    one, _ = ev.evaluate_files(model, quads, calib=calibs[0], **kw)          # one calibration for every pair
    assert one["depth"]["n_valid"] > 0


# ---- launch sequence -------------------------------------------------------------------------------------------
def test_reproject_is_one_entry_point_call_after_an_unchanged_forward():
    """The default forward's recorded sequence is unchanged; reproject on its pred4, windowed, adds exactly one
    dca_reproject (its count and scatter launches) with the window's pitches, shape and origin."""
    import dcanet_b200 as d
    from test_host_sequence import _gold
    from test_lr_check_host import _forward_trace
    net = d.GwcNet(48).eval()
    one, _, (pred, pv) = _forward_trace(net, 1)
    assert one == _gold("kernel_sequence_tiny.json")
    c = geo.StereoCalib(700.0, 700.0, 60.0, 30.0, 0.5)
    peak = torch.zeros(1, 1, 64, 128)
    label = torch.zeros(1, 1, 64, 128, dtype=torch.uint8)
    with _dryrun.recording() as trace:
        pc = geo.reproject(pred, c, confidence=peak, min_confidence=0.5, label=label, window=(10, 4, 50, 120, 7),
                           min_depth=1.0, max_depth=80.0)
    assert len(trace) == 1 and trace[0][0] == "dca_reproject"
    full = trace.full[0]
    assert full[1] == pred.data_ptr() + 4 * (10 * 128 + 4) and full[2] == peak.data_ptr() + 4 * (10 * 128 + 4)
    assert full[3] == label.data_ptr() + 10 * 128 + 4
    assert full[4:11] == (128, 50 * 128, 1, 50, 120, 4, 7)           # B = 1: the image pitch is not read
    assert full[13:16] == (0.5, 1.0, 80.0) and full[12] is None
    assert pc.xyz.shape == (1, 50 * 120, 3) and pc.index.shape == (1, 6000) and pc.depth.shape == (1, 50, 120)
    assert full[-2] != 0 and pc.count.shape == (1,)
    with _dryrun.recording() as trace:
        geo.reproject(pred, c, frame="camera")
    assert [t[0] for t in trace] == ["dca_reproject"] and trace.full[0][10] == 0 and trace.full[0][2] == 0


def test_reproject_rejects_bad_arguments_on_the_host():
    c = geo.StereoCalib(700.0, 700.0, 60.0, 30.0, 0.5)
    d = torch.zeros(1, 1, 8, 8)
    with pytest.raises(ValueError, match="rect_to_velo"):
        geo.reproject(d, c, frame="velodyne")
    with pytest.raises(ValueError, match="frame"):
        geo.reproject(d, c, frame="world")
    with pytest.raises(ValueError, match="window"):
        geo.reproject(d, c, window=(4, 0, 5, 8, 0))
    with pytest.raises(ValueError):
        geo.reproject(d, c, confidence=torch.zeros(1, 1, 8, 7))
    with pytest.raises(ValueError):
        geo.reproject(d.double(), c)
    with pytest.raises(_lib.DcaError):                  # no CPU path
        geo.reproject(d, c)


def test_entry_points_reject_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    q = np.eye(4, dtype=np.float32)
    ok = [p, 0, 0, 8, 64, 1, 8, 8, 0, 0, q.ctypes.data, None, 0.0, 0.0, math.inf, 0, p, p, p, p, None]

    def call(**kw):
        args = list(ok)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_reproject(*args)

    for i in (0, 10, 16, 17, 18, 19):
        assert call(**{f"a{i}": None}) == -1, i
    assert call(a5=0) == call(a6=0) == call(a7=-1) == call(a5=65536) == -1
    assert call(a6=65536, a7=32768, a3=32768, a4=2 ** 31) == -1                # H W = 2^31
    assert call(a3=7) == call(a4=63) == -1                                      # pitches smaller than the window
    nan = float("nan")
    assert call(a12=nan) == call(a13=nan) == call(a14=nan) == call(a13=2.0, a14=1.0) == -1
    dm = [p, p, p, 1, 4, 4, 0.0, 100.0, 0.0, 1e-3, 80.0, None]

    def dcall(**kw):
        args = list(dm)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_depth_metrics(*args)

    assert dcall(a0=None) == dcall(a2=None) == dcall(a3=0) == dcall(a6=nan) == -1
    assert dcall(a7=0.0) == dcall(a7=math.inf) == dcall(a8=nan) == dcall(a9=0.0) == dcall(a10=math.inf) == -1
    assert dcall(a10=1e-4) == -1
