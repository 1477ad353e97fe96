"""CPU: LiDAR guidance host logic (guide.py, geometry.read_kitti_calib, evaluate_files(hints=)): the velodyne-to-camera
transform of every KITTI calibration style, the projection restated in tests/_guide_restatement.py against the KITTI
projection matrices and the reprojection, argument validation, and the hint-file dispatch of evaluate_files with the
kernels replaced by their restatements."""
import importlib
import math

import numpy as np
import pytest
import torch
from PIL import Image

import _eval_restatement as EO
import _guide_restatement as G
from _reproject_restatement import keep_and_points, kitti_scene, write_kitti_calib
from test_evaluation_host import _FakeStereoLogits, _patch_kernels
from test_kitti_io import _rgb

pkg = "cost-volume-aggregation-in-stereo-matching-revisited_b200"
geo = importlib.import_module(pkg + ".geometry")
guide = importlib.import_module(pkg + ".guide")
ev = importlib.import_module(pkg + ".evaluation")
io = importlib.import_module(pkg + ".kitti_io")
gw = importlib.import_module(pkg + ".gwcnet_dca_g")


def _h(m):
    out = np.eye(4)
    out[:3] = np.asarray(m, np.float64).reshape(3, 4)
    return out


def _write_raw(tmp_path, s):
    fmt = lambda a: " ".join("%.12e" % v for v in np.asarray(a).ravel())
    (tmp_path / "calib_cam_to_cam.txt").write_text("\n".join([
        "calib_time: 09-Jan-2012 13:57:47", "R_rect_00: " + fmt(s["R0_rect"]), "P_rect_00: " + fmt(s["P2"]),
        "R_rect_02: " + fmt(np.eye(3)), "P_rect_02: " + fmt(s["P2"]), "P_rect_03: " + fmt(s["P3"])]) + "\n")
    (tmp_path / "calib_velo_to_cam.txt").write_text("calib_time: 15-Mar-2012 11:37:16\nR: " + fmt(s["Rv"]) + "\nT: "
                                                   + fmt(s["tv"]) + "\ndelta_f: 0 0\ndelta_c: 0 0\n")
    return str(tmp_path / "calib_cam_to_cam.txt"), str(tmp_path / "calib_velo_to_cam.txt")


def _calibs(tmp_path):
    s = kitti_scene()
    write_kitti_calib(tmp_path / "obj.txt", s, "object")
    fmt = lambda a: " ".join("%.12e" % v for v in np.asarray(a).ravel())
    Tr = (np.hstack([s["R0_rect"], np.zeros((3, 1))]) @ _h(s["Tr_velo_to_cam"]))           # odometry: Tr is rectified
    (tmp_path / "odo.txt").write_text("\n".join(["P0: " + fmt(s["P2"]), "P1: " + fmt(s["P3"]), "P2: " + fmt(s["P2"]),
                                                 "P3: " + fmt(s["P3"]), "Tr: " + fmt(Tr)]) + "\n")
    cam, velo = _write_raw(tmp_path, s)
    return s, {"object": geo.read_kitti_calib(str(tmp_path / "obj.txt")),
               "odometry": geo.read_kitti_calib(str(tmp_path / "odo.txt")),
               "raw": geo.read_kitti_calib(cam, velo_to_cam=velo)}


# ---- calibration -----------------------------------------------------------------------------------------------
def test_velo_to_rect_is_the_inverse_of_rect_to_velo_for_every_calibration_style(tmp_path):
    s, calibs = _calibs(tmp_path)
    ref = calibs["object"]
    for style, c in calibs.items():
        assert c.velo_to_rect is not None and c.rect_to_velo is not None, style
        prod = _h(c.velo_to_rect) @ _h(c.rect_to_velo)
        assert np.abs(prod - np.eye(4)).max() < 1e-5, style
        # every style describes the same rig
        assert np.abs(c.velo_to_rect - ref.velo_to_rect).max() < 1e-5, style
    # the float64 composition: unshift R0 Tr_velo_to_cam, stored as float32
    sh = np.eye(4)
    sh[:3, 3] = (s["P2"][0, 3] / s["fx"], s["P2"][1, 3] / s["fy"], 0.0)
    R0 = np.eye(4)
    R0[:3, :3] = s["R0_rect"]
    want = (sh @ R0 @ _h(s["Tr_velo_to_cam"]))[:3].astype(np.float32)
    assert np.abs(ref.velo_to_rect - want).max() <= 1e-6 * np.abs(want).max()


def test_raw_calib_without_velo_to_cam_is_unchanged(tmp_path):
    s = kitti_scene()
    cam, _ = _write_raw(tmp_path, s)
    c = geo.read_kitti_calib(cam)
    assert c.rect_to_velo is None and c.velo_to_rect is None
    write_kitti_calib(tmp_path / "raw2.txt", s, "raw")
    (tmp_path / "v.txt").write_text("R: " + " ".join(["1", "0", "0", "0", "1", "0", "0", "0", "1"]) + "\nT: 0 0 0\n")
    with pytest.raises(ValueError, match="R_rect_00"):
        geo.read_kitti_calib(str(tmp_path / "raw2.txt"), velo_to_cam=str(tmp_path / "v.txt"))


def test_a_velodyne_point_lands_on_its_p2_and_p3_pixel_with_disparity_fb_over_z(tmp_path):
    s, calibs = _calibs(tmp_path)
    c = calibs["object"]
    rng = np.random.default_rng(3)
    for _ in range(20):
        Xc = np.array([rng.uniform(-8, 8), rng.uniform(-1, 2), rng.uniform(5, 50)])       # rectified cam-0 frame
        x0 = np.linalg.solve(s["R0_rect"], Xc)                                            # unrectified cam 0
        pv = np.linalg.solve(s["Rv"], x0 - s["tv"])                                       # velodyne
        p2 = s["P2"] @ np.append(Xc, 1.0)
        p3 = s["P3"] @ np.append(Xc, 1.0)
        u2, v2, u3 = p2[0] / p2[2], p2[1] / p2[2], p3[0] / p3[2]
        pts = np.append(pv, 0.5)[None].astype(np.float32)
        for view, u in (("left", u2), ("right", u3)):
            m = G.lidar_hints([pts], c.velo_to_rect, c.fx, c.fy, c.cx, c.cy, c.focal_baseline, c.doffs, 400, 1300,
                              view=view)[0]
            ys, xs = np.nonzero(m)
            assert (int(ys[0]), int(xs[0])) == (math.floor(v2 + 0.5), math.floor(u + 0.5)), view
            assert abs(float(m[ys[0], xs[0]]) - c.focal_baseline / Xc[2]) < 1e-3
            assert abs(float(m[ys[0], xs[0]]) - (u2 - u3)) < 1e-3


@pytest.mark.parametrize("window", [None, (9, 0, 375, 1242, 0), (0, 0, 352, 1216, 11)])
def test_round_trip_through_the_reprojection(tmp_path, window):
    """reproject(lidar_hints(points), frame="velodyne") gives the points back, up to the pixel quantisation."""
    _, calibs = _calibs(tmp_path)
    c = calibs["object"]
    H, W = (384, 1248) if window is not None and window[0] == 9 else (375, 1242) if window is None else (352, 1216)
    pts = G.camera_points(5, 4000, c.fx, c.fy, c.cx, c.cy, 1242, 375, c.rect_to_velo, zmin=4.0, zmax=40.0)
    m = G.lidar_hints([pts], c.velo_to_rect, c.fx, c.fy, c.cx, c.cy, c.focal_baseline, c.doffs, H, W, window=window)
    y0, x0, h, w, vo = window or (0, 0, H, W, 0)
    keep, P, Z = keep_and_points(m[:, y0:y0 + h, x0:x0 + w], None, None, x0, vo, c.Q(), c.rect_to_velo, 0.0, 0.0,
                                 np.inf)
    keep &= m[:, y0:y0 + h, x0:x0 + w] > 0
    got = P[keep]
    assert len(got) > 1000
    # every reprojected point has a scan point within the quantisation (half a pixel at its depth, plus rounding)
    from scipy.spatial import cKDTree
    dist, _ = cKDTree(pts[:, :3]).query(got)
    zq = Z[keep]
    assert np.all(dist <= 0.75 * zq / c.fx * math.sqrt(2) + 1e-3)


def test_z_buffer_ties_points_behind_the_camera_and_window_placement(tmp_path):
    _, calibs = _calibs(tmp_path)
    c = calibs["object"]
    T = _h(c.rect_to_velo)
    cam = lambda u, v, Z: (T @ np.array([(u - c.cx) * Z / c.fx, (v - c.cy) * Z / c.fy, Z, 1.0]))[:3]
    near, far = cam(100.2, 50.1, 10.0), cam(100.3, 50.2, 20.0)
    behind = (T @ np.array([1.0, 0.2, -15.0, 1.0]))[:3]                                   # Z < 0: dropped
    pts = np.array([np.append(p, 0.0) for p in (far, near, near, behind)], np.float32)
    args = (c.velo_to_rect, c.fx, c.fy, c.cx, c.cy, c.focal_baseline, c.doffs)
    m = G.lidar_hints([pts], *args, 200, 400)[0]
    assert np.count_nonzero(m) == 1
    M = np.asarray(c.velo_to_rect, np.float32)
    Zn = G.transform(M, pts[1:2])[0, 2]
    assert m[50, 100] == np.float32(c.focal_baseline) / Zn - np.float32(0.0)
    # fit mode, image smaller than the crop: rows move down by the top padding; pad16 the same; a centre crop moves them up
    for window, row in (((34, 0, 166, 400, 0), 34 + 50), ((0, 0, 100, 400, 20), 30)):
        mw = G.lidar_hints([pts], *args, 200, 400, window=window)[0]
        assert np.count_nonzero(mw) == 1 and mw[row, 100] == m[50, 100]
    # outside the window's columns: nothing
    assert not G.lidar_hints([pts], *args, 200, 400, window=(0, 200, 200, 200, 0))[0].any()


def test_quarter_takes_the_nearest_valid_hint_of_each_block():
    h = np.zeros((1, 8, 8), np.float32)
    h[0, 0, 0], h[0, 3, 3], h[0, 1, 2] = 10.0, 30.0, np.nan
    h[0, 4, 4], h[0, 5, 5] = 200.0, -3.0            # >= maxdisp, negative: no hint
    h[0, 6, 7] = np.inf
    h[0, 0, 4] = 17.0
    q = G.quarter(h, 192)
    assert q.tolist() == [[[7.5, 4.25], [0.0, 0.0]]]


# ---- argument validation ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,c", [(0.0, 1.0), (-1.0, 1.0), (math.inf, 1.0), (math.nan, 1.0), (10.0, 0.0),
                                 (10.0, -2.0), (10.0, math.inf), (10.0, math.nan), (10.0, 1e-30)])
def test_modulation_parameters_are_validated(k, c):
    with pytest.raises(ValueError):
        guide.modulation_scale(k, c)


def test_modulation_scale_is_float32_of_the_float64_value():
    assert guide.modulation_scale(10.0, 1.0) == 0.5
    assert guide.modulation_scale(3.0, 0.7) == float(np.float32(1.0 / (2 * 0.7 * 0.7)))


def test_forward_and_hot_path_validate_hint_arguments():
    net = gw.GwcNet(48).eval()
    x = torch.zeros(1, 3, 32, 64)
    with pytest.raises(ValueError, match="lr_check"):
        net(x, x, hints_right=torch.zeros(1, 1, 32, 64))
    f = torch.zeros(1, 320, 8, 16)
    with pytest.raises(ValueError, match="hint_k"):
        net.hot_path(f, f, None, None, None, hints=torch.zeros(1, 1, 32, 64), hint_k=0.0)
    with pytest.raises(ValueError, match="hint_c"):
        net.hot_path(f, f, None, None, None, hints=torch.zeros(1, 1, 32, 64), hint_c=-1.0)


def test_lidar_hints_validates_before_touching_a_device(tmp_path):
    _, calibs = _calibs(tmp_path)
    pts = np.zeros((4, 4), np.float32)
    no_velo = geo.StereoCalib(700, 700, 600, 180, 0.5)
    with pytest.raises(ValueError, match="velo_to_rect"):
        guide.lidar_hints(pts, no_velo, (32, 64))
    with pytest.raises(ValueError, match="view"):
        guide.lidar_hints(pts, calibs["object"], (32, 64), view="centre")
    with pytest.raises(ValueError, match="window"):
        guide.lidar_hints(pts, calibs["object"], (32, 64), window=(0, 0, 40, 64, 0))
    with pytest.raises(ValueError, match="min_depth"):
        guide.lidar_hints(pts, calibs["object"], (32, 64), min_depth=0.0)


def test_read_velodyne_reads_kitti_bin_scans(tmp_path):
    a = np.random.default_rng(0).normal(size=(17, 4)).astype(np.float32)
    a.tofile(tmp_path / "s.bin")
    assert np.array_equal(guide.read_velodyne(str(tmp_path / "s.bin")), a)
    np.zeros(5, np.float32).tofile(tmp_path / "bad.bin")
    with pytest.raises(ValueError, match="multiple of 4"):
        guide.read_velodyne(str(tmp_path / "bad.bin"))


# ---- evaluate_files(hints=) ---------------------------------------------------------------------------------------
class _HintedFake(_FakeStereoLogits):
    """Records the hint arguments of every call; the prediction does not depend on them."""

    def __init__(self):
        super().__init__()
        self.calls = []

    def forward(self, left, right, disp_true=None, **kw):
        self.calls.append({k: (v.clone() if torch.is_tensor(v) else v) for k, v in kw.items()})
        return super().forward(left, right)


def test_evaluate_files_requires_calib_with_hints(tmp_path):
    with pytest.raises(ValueError, match="calib"):
        ev.evaluate_files(_HintedFake(), [], hints=[])
    with pytest.raises(ValueError, match="hint_c"):
        ev.evaluate_files(_HintedFake(), [], hints=[], calib=geo.StereoCalib(700, 700, 30, 20, 0.5), hint_c=0.0)


@pytest.mark.parametrize("mode", ["fit", "pad16"])
def test_evaluate_files_dispatches_hint_files_and_scores_the_unhinted_pixels(tmp_path, monkeypatch, mode):
    """A .bin is projected with the pair's calib and window, a sparse-depth PNG becomes fB / depth - doffs framed like the
    GT; the model gets them as hints=; `unhinted` scores pred on the GT pixels without a valid hint."""
    _patch_kernels(monkeypatch)
    monkeypatch.setattr(ev, "_depth_metrics", lambda *a: None)      # a calibration adds depth rows: not scored here
    _, calibs = _calibs(tmp_path)
    cal = calibs["object"]
    calib = geo.StereoCalib(cal.fx / 20, cal.fy / 20, 30.0, 20.0, cal.baseline, 0.0, cal.rect_to_velo,
                            cal.velo_to_rect)

    def fake_lidar(points, c, shape, window, view):
        m = G.lidar_hints([points], c.velo_to_rect, c.fx, c.fy, c.cx, c.cy, c.focal_baseline, c.doffs, *shape,
                          window=window, view=view)
        return torch.from_numpy(m)[:, None]
    monkeypatch.setattr(ev, "_lidar_hints", fake_lidar)
    sizes = [(37, 53), (48, 64), (40, 60)]
    quads, hints, expect = [], [], []
    for i, (h, w) in enumerate(sizes):
        Image.fromarray(_rgb(10 + i, h, w)).save(tmp_path / f"l{i}.png")
        Image.fromarray(_rgb(50 + i, h, w)).save(tmp_path / f"r{i}.png")
        gt = np.random.default_rng(100 + i).uniform(1, 40, (h, w)).astype(np.float32)
        io.save_disparity_png(str(tmp_path / f"g{i}.png"), gt)
        quads.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png"), str(tmp_path / f"g{i}.png"), None))
        if i == 1:                                       # sparse depth PNG
            depth = np.zeros((h, w), np.float32)
            depth[::3, ::4] = np.random.default_rng(7).uniform(3, 30, depth[::3, ::4].shape)
            io.save_disparity_png(str(tmp_path / "d1.png"), depth)
            hints.append(str(tmp_path / "d1.png"))
        else:                                            # velodyne scan
            pts = G.camera_points(20 + i, 300, calib.fx, calib.fy, calib.cx, calib.cy, w, h, calib.rect_to_velo)
            pts.tofile(tmp_path / f"v{i}.bin")
            hints.append(str(tmp_path / f"v{i}.bin"))
    model = _HintedFake().eval()
    summary, rows = ev.evaluate_files(model, quads, mode=mode, crop=(48, 64), depth=2, workers=2, maxdisp=48,
                                      calib=calib, hints=hints, hint_k=5.0, hint_c=2.0)
    assert len(model.calls) == len(quads)
    un_rows, n_hinted, n_valid = [], 0, 0
    for i, ((h, w), call) in enumerate(zip(sizes, model.calls)):
        assert call["hint_k"] == 5.0 and call["hint_c"] == 2.0 and "hints_right" not in call
        gt = ev.read_kitti_disparity(quads[i][2])
        if mode == "fit":
            gtf = io.fit_gt_to_crop(gt, 48, 64)
            window = (48 - h, 0, h, w, 0)
        else:
            gtf, top, _ = io.pad_gt_to_multiple(gt, 16)
            window = (top, 0, h, w, 0)
        if i == 1:
            depth = ev.read_kitti_disparity(hints[1])
            with np.errstate(divide="ignore"):
                disp = np.where(depth > 0, np.float32(calib.focal_baseline) / depth, np.float32(0)).astype(np.float32)
            want = io.fit_gt_to_crop(disp, 48, 64) if mode == "fit" else io.pad_gt_to_multiple(disp, 16)[0]
        else:
            want = G.lidar_hints([guide.read_velodyne(hints[i])], calib.velo_to_rect, calib.fx, calib.fy, calib.cx,
                                 calib.cy, calib.focal_baseline, calib.doffs, *gtf.shape, window=window)[0]
        got = call["hints"].reshape(gtf.shape).numpy()
        assert np.array_equal(got, want), i
        assert np.count_nonzero(got) > 10
        hinted = np.isfinite(got) & (got > 0) & (got < 48)
        valid = (gtf > 0) & (gtf < 48)
        n_hinted += int((hinted & valid).sum())
        n_valid += int(valid.sum())
        pair = io.load_pair(quads[i][0], quads[i][1])
        if mode == "fit":
            left, right, _, _ = io.fit_to_crop(pair, 48, 64)
        else:
            xx, _, _ = io.pad_to_multiple(torch.from_numpy(pair)[None], 16)
            left, right = xx[:, 0:3], xx[:, 3:6]
        with torch.no_grad():
            pred, _ = _FakeStereoLogits()(left, right)
        un_rows.append(EO.disparity_metric_counts(pred, np.where(hinted, 0, gtf)[None].astype(np.float32), 48)[0])
    assert summary["unhinted"] == ev.summarize(np.stack(un_rows).astype(np.uint64))
    assert summary["hint_density"] == pytest.approx(n_hinted / n_valid, rel=1e-12)
    assert 0 < summary["hint_density"] < 1
    assert "epe" in summary and rows.shape == (3, ev.METRIC_COUNT)
