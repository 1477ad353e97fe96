"""CPU: rectification of raw stereo pairs (rectify.py).  The maps against the identity rig and an independent float64
projection, the KITTI raw calib_cam_to_cam.txt reader, an end-to-end render of a textured plane through distorted raw
cameras against its direct rectified render, the float32 restatement (tests/_rectify_restatement.py) of the
standardised input against kitti_io.load_pair + fit_to_crop / pad_to_multiple, rectify_files and
reproject_files(rectifier=) with the kernels replaced by the restatement, the dry-run launch sequence, and the argument
checks on the host and in the entry points."""
import importlib
import math
import os

import numpy as np
import pytest
import torch
from PIL import Image

import _dryrun
import _rectify_restatement as Rs
import _reproject_restatement as R
from test_evaluation_host import _FakeStereoLogits
from test_reproject_host import _FakeStereoFilters, _read_ply, _restated_kernel

rect = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.rectify")
geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")


def _rig_args(cams, i):
    c = cams[i]
    return c["K"], c["D"], c["R_rect"], c["P_rect"]


def _kitti_rectifier(cams=None):
    cams = cams or Rs.kitti_raw_rig()
    return rect.StereoRectifier(*_rig_args(cams, 2), *_rig_args(cams, 3), raw_size=(1392, 512), rect_size=(1242, 375))


def _small_rectifier(raw=(56, 40), rect_size=(52, 36)):
    """A small distorted rig for the pipeline tests, its focal lengths and principal points scaled with the sizes."""
    s, sr = raw[0] / 56.0, rect_size[0] / 52.0
    K = np.array([[50.0 * s, 0.0, raw[0] / 2 + 0.3], [0.0, 49.0 * s, raw[1] / 2 - 0.4], [0.0, 0.0, 1.0]])
    Kr = np.array([[47.0 * sr, 0.0, rect_size[0] / 2], [0.0, 47.0 * sr, rect_size[1] / 2], [0.0, 0.0, 1.0]])
    R1, R2 = Rs._rot(0.01, -0.02, 0.005), Rs._rot(-0.01, 0.015, -0.004)
    P1 = Kr @ np.hstack([np.eye(3), [[0.0], [0.0], [0.0]]])
    P2 = Kr @ np.hstack([np.eye(3), [[-0.3], [0.0], [0.0]]])
    return rect.StereoRectifier(K, [-0.08, 0.02, 0.001, -0.002, 0.0], R1, P1, K, [-0.07, 0.015, 0.0, 0.001], R2, P2,
                                raw, rect_size)


# ---- maps ------------------------------------------------------------------------------------------------------
def test_identity_rig_maps_to_the_integer_pixel_grid():
    K = np.array([[500.0, 0.0, 31.5], [0.0, 480.0, 20.25], [0.0, 0.0, 1.0]])
    P = np.hstack([K, np.zeros((3, 1))])
    P2 = P.copy()
    P2[0, 3] = -500.0 * 0.2
    r = rect.StereoRectifier(K, [], np.eye(3), P, K, np.zeros(5), np.eye(3), P2, (64, 40), (64, 40))
    assert r.maps.shape == (2, 40, 64, 2) and r.maps.dtype == np.float32
    gx, gy = np.meshgrid(np.arange(64, dtype=np.float32), np.arange(40, dtype=np.float32))
    for v in range(2):
        assert np.array_equal(r.maps[v, ..., 0], gx) and np.array_equal(r.maps[v, ..., 1], gy)
    c = r.calib
    assert (c.fx, c.fy, c.cx, c.cy, c.doffs) == (500.0, 480.0, 31.5, 20.25, 0.0) and c.baseline == pytest.approx(0.2)


def _distort(xp, yp, D):
    k1, k2, p1, p2, k3 = D
    r2 = xp * xp + yp * yp
    kr = 1 + k1 * r2 + k2 * r2 ** 2 + k3 * r2 ** 3
    return xp * kr + 2 * p1 * xp * yp + p2 * (r2 + 2 * xp * xp), yp * kr + p1 * (r2 + 2 * yp * yp) + 2 * p2 * xp * yp


def test_maps_against_an_independent_projection():
    """A 3-D point in camera i's rectified frame, seen at integer rectified pixel (u, v) through P[:, :3], is the point
    R^T X in the raw frame; the raw camera (forward distortion, then K) sees it where the map says."""
    cams = Rs.kitti_raw_rig()
    r = _kitti_rectifier(cams)
    rng = np.random.default_rng(0)
    for view, i in enumerate((2, 3)):
        c = cams[i]
        K, D, Rr, P = c["K"], c["D"], c["R_rect"], c["P_rect"]
        for _ in range(300):
            u, v, z = int(rng.integers(0, 1242)), int(rng.integers(0, 375)), rng.uniform(2.0, 80.0)
            X = z * np.linalg.solve(P[:, :3], [u, v, 1.0])
            assert np.allclose(P[:, :3] @ X / X[2], [u, v, 1.0])
            Xr = Rr.T @ X
            xd, yd = _distort(Xr[0] / Xr[2], Xr[1] / Xr[2], D)
            want = (K[0, 0] * xd + K[0, 1] * yd + K[0, 2], K[1, 1] * yd + K[1, 2])
            assert np.abs(r.maps[view, v, u] - want).max() < 1e-3, (view, u, v)
    # the conventions matter: R instead of R^T, or the distortion undone instead of applied, land pixels away
    c = cams[2]
    X = 10.0 * np.linalg.solve(c["P_rect"][:, :3], [1200.0, 20.0, 1.0])
    for Xr, D in ((c["R_rect"] @ X, c["D"]), (c["R_rect"].T @ X, -c["D"])):
        xd, yd = _distort(Xr[0] / Xr[2], Xr[1] / Xr[2], D)
        wrong = (c["K"][0, 0] * xd + c["K"][0, 2], c["K"][1, 1] * yd + c["K"][1, 2])
        assert np.abs(r.maps[0, 20, 1200] - wrong).max() > 5.0


def test_points_behind_the_camera_map_to_nan():
    K = np.array([[100.0, 0.0, 50.0], [0.0, 100.0, 30.0], [0.0, 0.0, 1.0]])
    P = np.hstack([K, np.zeros((3, 1))])
    P2 = P.copy()
    P2[0, 3] = -10.0
    Rt = Rs._rot(0.0, np.pi / 2 - 0.05, 0.0)              # the rectified frame looks almost sideways
    r = rect.StereoRectifier(K, [], Rt, P, K, [], np.eye(3), P2, (100, 60), (100, 60))
    x, y, w = np.linalg.inv(P[:, :3] @ Rt) @ np.stack([*np.meshgrid(np.arange(100.0), np.arange(60.0)),
                                                         np.ones((60, 100))]).reshape(3, -1)
    behind = (w <= 0).reshape(60, 100)
    assert behind.any() and not behind.all()
    assert np.isnan(r.maps[0][behind]).all() and np.isfinite(r.maps[0][~behind]).all()


def test_constructor_rejects_bad_calibrations():
    K, P = np.eye(3) * [100, 100, 1], np.hstack([np.eye(3) * [100, 100, 1], np.zeros((3, 1))])
    ok = dict(K1=K, D1=[], R1=np.eye(3), P1=P, K2=K, D2=[], R2=np.eye(3), P2=P, raw_size=(8, 6), rect_size=(8, 6))
    rect.StereoRectifier(**dict(ok, P2=P - [[0, 0, 0, 10], [0, 0, 0, 0], [0, 0, 0, 0]]))
    bad = [dict(D1=[0.1, 0.2, 0.3]), dict(D2=np.zeros(6)), dict(K1=np.eye(2)), dict(R2=np.eye(4)), dict(P1=K),
           dict(K1=K * [[-1], [1], [1]]), dict(P2=P * [[1], [0], [1]]), dict(K2=K + np.nan), dict(D1=[np.inf, 0, 0, 0]),
           dict(raw_size=(0, 6)), dict(rect_size=(8, -1)), dict(raw_size=(8.5, 6)), dict(rect_size=8)]
    for kw in bad:
        with pytest.raises(ValueError):
            rect.StereoRectifier(**dict(ok, **kw))


# ---- KITTI raw calibration -----------------------------------------------------------------------------------------
def test_kitti_raw_reader(tmp_path):
    cams = Rs.kitti_raw_rig()
    path = str(tmp_path / "calib_cam_to_cam.txt")
    Rs.write_kitti_raw_calib(path, cams)
    r = rect.read_kitti_raw_rectifier(path)
    assert r.raw_size == (1392, 512) and r.rect_size == (1242, 375) and r.maps.shape == (2, 375, 1242, 2)
    want = _kitti_rectifier(cams)
    assert np.allclose(r.maps, want.maps, rtol=0, atol=2e-3, equal_nan=True)
    k = geo.read_kitti_calib(path)
    c = r.calib
    assert (c.fx, c.fy, c.cx, c.cy, c.baseline, c.doffs) == (k.fx, k.fy, k.cx, k.cy, k.baseline, k.doffs)
    assert c.baseline == pytest.approx(0.0598 + 0.4731, rel=1e-9)
    r01 = rect.read_kitti_raw_rectifier(path, left=0, right=1)
    assert r01.calib.baseline == pytest.approx(0.537, rel=1e-9)
    for key in ("S_02", "K_03", "D_02", "R_rect_03", "P_rect_02", "S_rect_03"):
        Rs.write_kitti_raw_calib(path, cams, drop=key)
        with pytest.raises(ValueError, match=key):
            rect.read_kitti_raw_rectifier(path)
    Rs.write_kitti_raw_calib(path, cams, d_len=3)
    with pytest.raises(ValueError, match="0, 4 or 5"):
        rect.read_kitti_raw_rectifier(path)
    Rs.write_kitti_raw_calib(path, cams, d_len=4)
    assert rect.read_kitti_raw_rectifier(path).raw_size == (1392, 512)


# ---- the geometry, end to end ----------------------------------------------------------------------------------------
def _texture(X, Y):
    """Grey level of the plane at (X, Y) metres: smooth, periods of about 40 px at the plane's depth."""
    return 127.5 + 55.0 * np.sin(X * 9.0 + 0.3) * np.cos(Y * 7.0) + 40.0 * np.sin(X * 4.0 - Y * 11.0)


def _undistort(xd, yd, D):
    xp, yp = xd.copy(), yd.copy()
    for _ in range(60):
        ex, ey = _distort(xp, yp, D)
        xp, yp = xp - (ex - xd), yp - (ey - yd)
    ex, ey = _distort(xp, yp, D)
    assert max(np.abs(ex - xd).max(), np.abs(ey - yd).max()) < 1e-9
    return xp, yp


def test_rectified_render_of_a_plane_matches_the_direct_render():
    """A textured plane Z = 8 m (fronto-parallel in the rectified frame), rendered in float64 through each distorted raw
    camera (undistort the raw pixel's ray, rotate it into the rectified frame, intersect) and rounded to uint8, then
    rectified by the restatement of dca_rectify; against the plane rendered directly in the rectified views.  Inside,
    the two differ by the raw rounding (0.5), the bilinear interpolation of the texture (< 0.6 for its curvature at one
    pixel) and the output rounding (0.5): at most 2 grey levels."""
    cams = Rs.kitti_raw_rig()
    r = _kitti_rectifier(cams)
    z0 = 8.0
    raws, direct = [], []
    for i in (2, 3):
        c = cams[i]
        K, D, Rr, P = c["K"], c["D"], c["R_rect"], c["P_rect"]
        t = np.linalg.solve(P[:, :3], P[:, 3])                     # camera i's offset: X_i = X_0 + t
        xs, ys = np.meshgrid(np.arange(1392.0), np.arange(512.0))
        yd = (ys - K[1, 2]) / K[1, 1]
        xd = (xs - K[0, 2] - K[0, 1] * yd) / K[0, 0]
        xp, yp = _undistort(xd, yd, D)
        ray = np.einsum("ij,jhw->ihw", Rr, np.stack([xp, yp, np.ones_like(xp)]))
        Xi = ray * (z0 / ray[2])
        raws.append(np.clip(np.rint(_texture(Xi[0] - t[0], Xi[1] - t[1])), 0, 255).astype(np.uint8))
        us, vs = np.meshgrid(np.arange(1242.0), np.arange(375.0))
        Xr = z0 * np.einsum("ij,jhw->ihw", np.linalg.inv(P[:, :3]), np.stack([us, vs, np.ones_like(us)]))
        direct.append(_texture(Xr[0] - t[0], Xr[1] - t[1]))
    rgb_l = np.repeat(raws[0][None, ..., None], 3, -1)
    rgb_r = np.repeat(raws[1][None, ..., None], 4, -1)            # an RGBA source: channel 3 is ignored
    rgb_r[..., 3] = 7
    rgb, moments = Rs.remap(rgb_l, rgb_r, r.maps)
    for v in range(2):
        m = r.maps[v]
        inside = (m[..., 0] >= 2) & (m[..., 0] <= 1392 - 3) & (m[..., 1] >= 2) & (m[..., 1] <= 512 - 3)
        assert inside.mean() > 0.9
        err = np.abs(rgb[0, v, ..., 0].astype(np.float64) - direct[v])[inside]
        assert err.max() <= 2.0, (v, err.max())
        assert np.array_equal(rgb[0, v, ..., 0], rgb[0, v, ..., 2])
        q = rgb[0, v].astype(np.int64)
        assert moments[0, v].tolist() == [[int(q[..., c].sum()), int((q[..., c] ** 2).sum())] for c in range(3)]
        print("plane render view %d: max |rectified - direct| %.3f, mean %.3f grey levels" % (v, err.max(),
                                                                                               err.mean()))


# ---- the restatement of the standardised input -----------------------------------------------------------------------
def _ulp_close(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    both_nan = np.isnan(a) & np.isnan(b)
    diff = np.abs(a.astype(np.float64) - b.astype(np.float64))
    tol = np.spacing(np.maximum(np.abs(a), np.abs(b))).astype(np.float64)
    return bool((both_nan | (diff <= tol)).all())


@pytest.mark.parametrize("H,W,mode", [(37, 53, "fit"), (48, 64, "fit"), (60, 70, "fit"), (37, 53, "pad16"),
                                      (48, 64, "pad16")])
def test_standardised_input_equals_load_pair_and_the_framing(H, W, mode):
    rng = np.random.default_rng(H * W)
    rgb = rng.integers(0, 256, (1, 2, H, W, 3), dtype=np.uint8)
    rgb[0, 1, ..., 1] = 77                                           # a constant channel: NaN, as load_pair gives
    q = rgb.astype(np.int64)
    moments = np.stack([q.sum(axis=(2, 3)), (q * q).sum(axis=(2, 3))], -1)
    frame, window = Rs.framing(H, W, mode, 48, 64)
    assert rect.framing(H, W, mode, (48, 64)) == (frame, window)
    left, right = Rs.standardise_frame(rgb, moments, frame)
    with np.errstate(invalid="ignore", divide="ignore"):
        pair = io.load_pair(rgb[0, 0], rgb[0, 1])
    if mode == "fit":
        wl, wr, _, _ = io.fit_to_crop(pair, 48, 64)
    else:
        x, _, _ = io.pad_to_multiple(torch.from_numpy(pair)[None], 16)
        wl, wr = x[:, 0:3], x[:, 3:6]
    assert left.shape == tuple(wl.shape) and right.shape == tuple(wr.shape)
    assert _ulp_close(left, wl.numpy()) and _ulp_close(right, wr.numpy())
    assert np.isnan(right[0, 1][window[0]:window[0] + window[2], :window[3]]).all()
    exact = (left == wl.numpy()).mean()
    print("standardised %dx%d %s: %.4f of the left values bit-equal to load_pair" % (H, W, mode, exact))
    # the window is ReprojectPipeline's for this size
    pipe = geo.ReprojectPipeline(_FakeStereoLogits(), geo.StereoCalib(1, 1, 0, 0, 1), mode, 48, 64)
    with np.errstate(invalid="ignore", divide="ignore"):
        assert pipe._load_item(rgb[0, 0], rgb[0, 1])[2] == window


def test_channel_statistics_agree_with_numpy():
    rng = np.random.default_rng(3)
    for H, W in ((1, 1), (3, 5), (375, 1242)):
        ch = rng.integers(0, 256, (H, W), dtype=np.uint8)
        mean, std = Rs.channel_stats(int(ch.sum(dtype=np.int64)), int((ch.astype(np.int64) ** 2).sum()), H * W)
        assert mean == np.mean(ch)
        assert std == pytest.approx(float(np.std(ch)), rel=1e-13, abs=1e-300)


# ---- pipelines with the kernels replaced by the restatement -----------------------------------------------------------
def _patch_rectify(monkeypatch):
    def rk(left, right, maps, H, W):
        rgb, m = Rs.remap(left.numpy(), right.numpy(), maps.numpy())
        return torch.from_numpy(rgb), torch.from_numpy(m)

    def sk(rgb, moments, frame):
        left, right = Rs.standardise_frame(rgb.numpy(), moments.numpy(), frame)
        return torch.from_numpy(left), torch.from_numpy(right)

    monkeypatch.setattr(rect, "_rectify_kernel", rk)
    monkeypatch.setattr(rect, "_standardise_kernel", sk)


def _raw_pngs(tmp_path, r, n, rgba_at=()):
    Ws, Hs = r.raw_size
    rng = np.random.default_rng(11)
    items = []
    for i in range(n):
        c = 4 if i in rgba_at else 3
        base = rng.integers(0, 256, (Hs, Ws + 4, c), dtype=np.uint8)
        Image.fromarray(np.ascontiguousarray(base[:, :Ws])).save(tmp_path / f"rl{i}.png")
        Image.fromarray(np.ascontiguousarray(base[:, 4:])).save(tmp_path / f"rr{i}.png")
        items.append((str(tmp_path / f"rl{i}.png"), str(tmp_path / f"rr{i}.png")))
    return items


@pytest.mark.parametrize("crop", [(48, 64), (32, 48)])
def test_rectify_files_equals_a_serial_loop(tmp_path, monkeypatch, crop):
    _patch_rectify(monkeypatch)
    r = _small_rectifier()
    pairs = _raw_pngs(tmp_path, r, 5, rgba_at=(2,))
    model = _FakeStereoLogits().eval()
    triples = [(l, rr, str(tmp_path / f"o{i}.png") if i % 2 else None) for i, (l, rr) in enumerate(pairs)]
    W, H = r.rect_size
    frame, _ = Rs.framing(H, W, "fit", *crop)
    ref = []
    for l, rr, _ in triples:
        a, b = np.asarray(Image.open(l))[None], np.asarray(Image.open(rr))[None]
        rgb, m = Rs.remap(a, b, r.maps)
        left, right = Rs.standardise_frame(rgb, m, frame)
        with torch.no_grad():
            pred, _ = model(torch.from_numpy(left), torch.from_numpy(right))
        ref.append(io.crop_prediction(pred[0, 0].numpy(), H, W, *crop))
    got = rect.rectify_files(model, triples, r, *crop, depth=2, workers=3)
    assert len(got) == len(ref)
    for i, (g, w) in enumerate(zip(got, ref)):
        assert g.shape == w.shape and np.array_equal(g, w), i
        if triples[i][2]:
            assert np.array_equal(np.asarray(Image.open(triples[i][2])),
                                  io.save_disparity_png(str(tmp_path / "x.png"), w))


@pytest.mark.parametrize("mode", ["fit", "pad16"])
def test_reproject_files_with_a_rectifier_equals_a_serial_loop(tmp_path, monkeypatch, mode):
    _patch_rectify(monkeypatch)
    monkeypatch.setattr(geo, "_reproject_kernel", _restated_kernel)
    r = _small_rectifier()
    pairs = _raw_pngs(tmp_path, r, 4, rgba_at=(1,))
    model = _FakeStereoFilters().eval()
    items = [(l, rr, str(tmp_path / f"p{i}.ply") if i % 2 == 0 else None, str(tmp_path / f"d{i}.png") if i else None)
             for i, (l, rr) in enumerate(pairs)]
    W, H = r.rect_size
    frame, (y0, x0, h, w, vo) = Rs.framing(H, W, mode, 48, 64)
    c = r.calib
    ref = []
    for l, rr, _, _ in items:
        rgb, m = Rs.remap(np.asarray(Image.open(l))[None], np.asarray(Image.open(rr))[None], r.maps)
        left, right = Rs.standardise_frame(rgb, m, frame)
        with torch.no_grad():
            out = model(torch.from_numpy(left), torch.from_numpy(right), confidence=True, lr_check=True)
        win = lambda t: t[:, 0, y0:y0 + h, x0:x0 + w].numpy()
        xyz, index, _, depth = R.reproject(win(out[0]), win(out[2].peak), win(out[3].label), x0, vo, c.Q(), None, 0.4,
                                           0.0, np.inf)
        ref.append((xyz[0], rgb[0, 0, vo:vo + h, x0:x0 + w].reshape(-1, 3)[index[0]], depth[0]))
    got = geo.reproject_files(model, items, mode=mode, crop=(48, 64), min_confidence=0.4, lr_check=True, depth=2,
                              workers=2, rectifier=r)
    for i, ((gx, gc), (rx, rc, rd)) in enumerate(zip(got, ref)):
        assert np.array_equal(gx, rx) and np.array_equal(gc, rc) and len(gx) > 0, i
        if items[i][2]:
            v, _ = _read_ply(items[i][2])
            assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], -1), rx)
            assert np.array_equal(np.stack([v["red"], v["green"], v["blue"]], -1), rc)
        if items[i][3]:
            assert np.array_equal(np.asarray(Image.open(items[i][3])), geo.save_depth_png(str(tmp_path / "x.png"), rd))
    other = geo.StereoCalib(c.fx, c.fy, c.cx, c.cy, 2 * c.baseline)           # an explicit calib wins over r.calib
    twice = geo.reproject_files(model, items[:1], other, mode=mode, crop=(48, 64), min_confidence=0.4, lr_check=True,
                                rectifier=r)
    assert np.allclose(twice[0][0][:, 2], 2 * ref[0][0][:, 2], rtol=1e-6)
    with pytest.raises(ValueError, match="calib"):
        geo.reproject_files(model, items, mode=mode)


def test_raw_pipelines_reject_images_of_another_size(tmp_path, monkeypatch):
    _patch_rectify(monkeypatch)
    r = _small_rectifier()
    Image.fromarray(np.zeros((40, 50, 3), np.uint8)).save(tmp_path / "s.png")
    Image.fromarray(np.zeros((40, 56), np.uint8)).save(tmp_path / "g.png")
    for name in ("s.png", "g.png"):
        with pytest.raises(ValueError):
            rect.rectify_files(_FakeStereoLogits(), [(str(tmp_path / name), str(tmp_path / name), None)], r, 48, 64)
    with pytest.raises(ValueError, match="neither inside nor around"):
        rect.RectifyPipeline(_FakeStereoLogits(), r, 32, 64)


# ---- launch sequence and argument checks ----------------------------------------------------------------------------
def test_rectify_is_two_entry_point_calls():
    r = _small_rectifier()
    big = torch.zeros(3, 40, 70, 4, dtype=torch.uint8)                     # a strided RGBA view: rows of 70 pixels
    left, right = big[:2, :, :56], big[1:, :, 3:59]
    for mode, crop in (("fit", (48, 64)), ("fit", (32, 48)), ("pad16", (384, 1248))):
        with _dryrun.recording() as trace:
            x = rect.rectify(left, right, r, mode, crop)
        assert [t[0] for t in trace] == ["dca_rectify", "dca_standardise_frame"]
        f0, f1 = trace.full
        assert f0[1] == left.data_ptr() and f0[2] == right.data_ptr() == big.data_ptr() + 40 * 70 * 4 + 12
        assert f0[3:9] == (4, 70 * 4, 40 * 70 * 4, 2, 40, 56)
        assert f0[9] == r.device_maps("cpu").data_ptr() and f0[10:12] == (36, 52)
        assert f0[12] == x.rgb.data_ptr() and x.rgb.shape == (2, 2, 36, 52, 3) and x.rgb.dtype == torch.uint8
        frame, window = Rs.framing(36, 52, mode, *crop)
        assert f1[1:3] == f0[12:14] and f1[3:6] == (2, 36, 52) and f1[6:8] == (x.left.data_ptr(), x.right.data_ptr())
        assert f1[8:14] == frame and x.window == window
        assert x.left.shape == x.right.shape == (2, 3, frame[0], frame[1]) and x.left.dtype == torch.float32
    one = torch.zeros(1, 40, 56, 3, dtype=torch.uint8)
    with _dryrun.recording() as trace:
        rect.rectify(one, one.clone(), r)
    assert trace.full[0][3:9] == (3, 56 * 3, 40 * 56 * 3, 1, 40, 56)        # B = 1: the image pitch is Hs pitch_row


def test_rectify_rejects_bad_arguments_on_the_host():
    r = _small_rectifier()
    ok = torch.zeros(1, 40, 56, 3, dtype=torch.uint8)
    bad = [torch.zeros(1, 40, 56, 3), torch.zeros(1, 40, 55, 3, dtype=torch.uint8),
           torch.zeros(1, 40, 56, 1, dtype=torch.uint8), torch.zeros(40, 56, 3, dtype=torch.uint8),
           torch.zeros(1, 3, 40, 56, dtype=torch.uint8).permute(0, 2, 3, 1),
           torch.zeros(1, 40, 112, 3, dtype=torch.uint8)[:, :, ::2], np.zeros((1, 40, 56, 3), np.uint8)]
    for t in bad:
        with pytest.raises(ValueError):
            rect.rectify(t, ok, r)
        with pytest.raises(ValueError):
            rect.rectify(ok, t, r)
    with pytest.raises(ValueError):
        rect.rectify(ok, torch.zeros(2, 40, 56, 3, dtype=torch.uint8), r)
    with pytest.raises(ValueError, match="mode"):
        rect.rectify(ok, ok, r, mode="pad32")
    with pytest.raises(ValueError, match="neither inside nor around"):
        rect.rectify(ok, ok, r, crop=(30, 64))
    with pytest.raises(ValueError, match="CUDA"):                           # no CPU path
        rect.rectify(ok, ok, r)


def test_entry_points_reject_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    ok = [p, p, 3, 30, 300, 2, 10, 10, p, 7, 5, p, p, None]

    def call(**kw):
        args = list(ok)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_rectify(*args)

    for i in (0, 1, 8, 11, 12):
        assert call(**{f"a{i}": None}) == -1, i
    for i in (5, 6, 7, 9, 10):
        assert call(**{f"a{i}": 0}) == -1 and call(**{f"a{i}": -3}) == -1, i
    assert call(a5=65536) == call(a2=2) == call(a2=5) == call(a2=1) == -1
    assert call(a3=29) == call(a4=299) == call(a2=4, a3=39) == -1                # pitches smaller than a row / an image
    assert call(a9=65536, a10=32768) == -3                                      # H W = 2^31
    assert call(a6=65536, a7=32768, a3=32768 * 3, a4=2 ** 31 * 3) == -3         # Hs Ws = 2^31
    assert call(a7=(1 << 24) + 1, a6=1, a3=3 * ((1 << 24) + 1), a4=3 * ((1 << 24) + 1)) == -3
    sf = [p, p, 2, 7, 5, p, p, 16, 16, 9, 0, 7, 5, None]

    def scall(**kw):
        args = list(sf)
        for k, v in kw.items():
            args[int(k[1:])] = v
        return lib.dca_standardise_frame(*args)

    for i in (0, 1, 5, 6):
        assert scall(**{f"a{i}": None}) == -1, i
    for i in (2, 3, 4, 7, 8, 11, 12):
        assert scall(**{f"a{i}": 0}) == -1, i
    assert scall(a2=65536) == scall(a9=-1) == scall(a10=-1) == scall(a9=10) == scall(a10=1) == -1
    assert scall(a12=6) == scall(a8=4) == scall(a11=8, a3=9, a9=9) == -1       # windows outside the image / frame
    assert scall(a7=65536, a8=32768) == -3
