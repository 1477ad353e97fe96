"""CPU: the occupancy grid of include/dca_b200.h section 17 through its numpy restatement
(tests/_occupancy_restatement.py) on the analytic scene of tests/test_motion_host.py (a road 1.65 m below the camera, a
wall at 60 m and a box, the camera moving 1 m forward per frame at KITTI intrinsics); OccupancyGrid and
fuse_files(volume=grid) with the kernels replaced by their restatements; save_map, agreement, and the argument checks
of the Python API and of the C entry point.

The scene bounds are measured values with a margin; they say nothing about KITTI or any real camera."""
import importlib
import math
import os

import numpy as np
import pytest
import torch

import _occupancy_restatement as R
import _reproject_restatement as RP
import dcanet_b200 as d
from test_motion_host import BOX, CALIB, FWIN, INTR, N_FRAMES, _box_at, _items, _NoModel, _patch, pose, render

oc = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.occupancy")
fu = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.fusion")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")

F32 = np.float32
W2G = oc.KITTI_WORLD_TO_GRID
# 0.2 m cells with edges on multiples of 0.2 m: grid x = world X in [-20, 20], grid y = world Z in [-2, 60]
GRID = dict(origin=(-19.9, -1.9), cell_size=0.2, dims=(200, 310))
STATIC = np.array([2.0, 0.0, 16.05])        # the box: X 1.1..2.9, Z 16.05..17.05 (cells i 105..114, j 90..95)
FOOT = (slice(90, 96), slice(105, 115))     # [j, i] of its footprint
FRAMES = 10


def mats(c2w):
    """grid <- camera and camera <- grid, float32 [B,12], from camera-to-world [B,4,4]."""
    M = W2G @ c2w
    return M[:, :3].reshape(-1, 12).astype(F32), np.linalg.inv(M)[:, :3].reshape(-1, 12).astype(F32)


def classes(L, U, occupied=0.65, free=0.2):
    p = 1 / (1 + np.exp(-L.astype(np.float64)))
    c = np.full(L.shape, d.UNKNOWN, np.uint8)
    c[(U > 0) & (p <= free)] = d.FREE
    c[(U > 0) & (p >= occupied)] = d.OCCUPIED
    return c


def restated(frames, at=STATIC, **kw):
    """The restatement over `frames` (one call per frame) -> (log_odds, updates)."""
    L = np.zeros(GRID["dims"][::-1], F32)
    U = np.zeros(GRID["dims"][::-1], np.int32)
    for i in frames:
        M, Mi = mats(pose(i)[None])
        R.integrate(L, U, GRID["origin"], GRID["cell_size"], render(pose(i), at)[None], M, Mi, INTR, **kw)
    return L, U


@pytest.fixture(scope="module")
def static_map():
    return restated(range(FRAMES))


def test_the_box_footprint_is_occupied_and_nothing_else(static_map):
    c = classes(*static_map)
    foot = c[FOOT]
    assert (foot[0] == d.OCCUPIED).all()                     # the front face
    assert (foot[:5, 0] == d.OCCUPIED).all()                 # the side seen from the left (the last 5 cm: j = 95)
    grown = np.zeros(c.shape, bool)
    grown[89:97, 104:116] = True
    assert not ((c == d.OCCUPIED) & ~grown).any()


def test_the_road_in_front_of_the_box_is_free(static_map):
    c = classes(*static_map)
    # Z 10..15.5 m: seen from at least five cameras beyond their 5.9 m blind zone
    assert (c[60:88, 105:115] == d.FREE).all()
    assert (c[60:88, 90:105] == d.FREE).all()                # and beside it


def test_the_shadow_the_blind_zone_and_the_outside_of_the_view_stay_unknown(static_map):
    L, U = static_map
    c = classes(L, U)
    assert (U[97:106, 108:112] == 0).all()                   # behind the box
    assert (U[:9, :] == 0).all()                             # Z < -0.1: behind every camera
    assert (U[14, 95:105] == 0).all()                        # Z = 0.9: under the first camera's 5.9 m blind zone
    assert (U[10:40, :20] == 0).all() and (U[10:40, -20:] == 0).all()      # |X| > 16 m within 8 m: outside the view
    assert (c[U == 0] == d.UNKNOWN).all()
    assert (U[258:, :] == 0).all() and (U[250, 95:105] > 0).all()    # the last camera (Z = 9) sees to 49.1 m


def test_one_call_of_b_frames_equals_b_calls():
    frames = [0, 2, 3, 5]
    z = np.stack([render(pose(i), STATIC) for i in frames])
    M, Mi = mats(np.stack([pose(i) for i in frames]))
    L = np.zeros(GRID["dims"][::-1], F32)
    U = np.zeros(GRID["dims"][::-1], np.int32)
    R.integrate(L, U, GRID["origin"], GRID["cell_size"], z, M, Mi, INTR)
    L1, U1 = restated(frames)
    assert np.array_equal(L, L1) and np.array_equal(U, U1)


# ---- the Python API with the restated kernel ------------------------------------------------------------------------
def _restated_kernel(calls=None):
    def kernel(grid, box, depth, weight, intr, u0, v0, M, Minv, max_depth):
        if calls is not None:
            calls.append((box, depth.shape[0], None if weight is None else weight.clone()))
        R.integrate(grid.log_odds.numpy(), grid.updates.numpy(), grid.origin, grid.cell_size, depth.numpy(), M, Minv,
                    intr, u0, v0, weight=None if weight is None else weight.numpy(), camera_height=grid.camera_height,
                    band=grid.band, col_width=grid.col_width, range_res=grid.range_res, max_depth=max_depth,
                    min_hits=grid.min_hits, l_hit=grid.l_hit, l_miss=grid.l_miss, l_min=grid.l_min, l_max=grid.l_max,
                    box=box)
    return kernel


def test_integrate_splits_batches_and_its_box_equals_the_whole_grid(monkeypatch):
    calls = []
    monkeypatch.setattr(oc, "_integrate_kernel", _restated_kernel(calls))
    frames = list(range(FRAMES)) + list(range(FRAMES))[::-1]                 # 20 frames: 16 + 4
    z = torch.from_numpy(np.stack([render(pose(i), STATIC) for i in frames]))
    c2w = np.stack([pose(i) for i in frames])
    g = d.OccupancyGrid(**GRID, device="cpu")
    g.integrate(z[:, None], CALIB, c2w)
    assert [c[1] for c in calls] == [16, 4]
    for box, _, _ in calls:
        assert box[1] > 0 and box[1] + box[3] < GRID["dims"][1]             # only the rows the cameras reach
    L = np.zeros(GRID["dims"][::-1], F32)
    U = np.zeros(GRID["dims"][::-1], np.int32)
    M, Mi = mats(c2w)
    for s in (0, 16):
        R.integrate(L, U, GRID["origin"], GRID["cell_size"], z[s:s + 16].numpy(), M[s:s + 16], Mi[s:s + 16], INTR)
    assert np.array_equal(g.log_odds.numpy(), L) and np.array_equal(g.updates.numpy(), U)
    assert int((U > 0).sum()) > 5000
    assert torch.equal(g.classes(), torch.from_numpy(classes(L, U)))


def test_a_lower_max_depth_and_a_window(monkeypatch):
    """max_depth lowers the grid's, a window is (y0, x0, h, w, v_origin), and a frame looking away from the grid makes
    no call."""
    calls = []
    monkeypatch.setattr(oc, "_integrate_kernel", _restated_kernel(calls))
    u0, v0, w, h = FWIN
    z = torch.from_numpy(render(pose(0), STATIC, FWIN))[None]
    g = d.OccupancyGrid(**GRID, device="cpu")
    g.integrate(z, CALIB, pose(0), window=(0, u0, h, w, v0), max_depth=20.0)
    M, Mi = mats(pose(0)[None])
    L = np.zeros(GRID["dims"][::-1], F32)
    U = np.zeros(GRID["dims"][::-1], np.int32)
    R.integrate(L, U, GRID["origin"], GRID["cell_size"], z.numpy(), M, Mi, INTR, u0, v0, max_depth=20.0)
    assert np.array_equal(g.log_odds.numpy(), L) and np.array_equal(g.updates.numpy(), U)
    assert (U[115:, :] == 0).all() and (U > 0).sum() > 500                  # nothing beyond Z = 21.1
    away = pose(0)
    away[:3, :3] = np.diag([-1.0, 1.0, -1.0])                               # looking backwards from Z = -30
    away[2, 3] = -30.0
    n = len(calls)
    g.integrate(z, CALIB, away, window=(0, u0, h, w, v0))
    assert len(calls) == n


def test_weights_and_masks_reach_the_grid(monkeypatch):
    """Weight 0 hides a pixel from the grid entirely; weight 0.5 halves its hits."""
    monkeypatch.setattr(oc, "_integrate_kernel", _restated_kernel())
    z = torch.from_numpy(render(pose(0), STATIC))[None]
    a = d.OccupancyGrid(**GRID, device="cpu").integrate(z, CALIB, pose(0), weight=torch.zeros_like(z))
    assert int(a.updates.sum()) == 0
    b = d.OccupancyGrid(**GRID, device="cpu", min_hits=200).integrate(z, CALIB, pose(0))
    c = d.OccupancyGrid(**GRID, device="cpu", min_hits=200).integrate(z, CALIB, pose(0), weight=torch.full_like(z, 0.5))
    nb = int((b.classes() == d.OCCUPIED).sum())
    nc = int((c.classes() == d.OCCUPIED).sum())
    assert nb > nc and nb > 0


def _grid_pipeline(monkeypatch, calls):
    """FusePipeline with the analytic depth of each pair in order (the moving box of tests/test_motion_host.py) and the
    grid's kernel by its restatement."""
    state = {"i": 0}

    def observe(self, slot, calib, window):
        i = state["i"]
        state["i"] += 1
        u0, v0, w, h = FWIN
        return torch.from_numpy(render(pose(i), _box_at(i), FWIN))[None], None, None, (0, u0, h, w, v0)
    monkeypatch.setattr(fu.FusePipeline, "_observe", observe)
    monkeypatch.setattr(oc, "_integrate_kernel", _restated_kernel(calls))
    _patch(monkeypatch)


MOVING = dict(origin=(-9.9, -1.9), cell_size=0.2, dims=(100, 210))


def _footprints(c, frames):
    """OCCUPIED cells of each frame's box footprint, grown by one cell."""
    out = []
    for i in frames:
        lo, hi = BOX[0] + _box_at(i), BOX[1] + _box_at(i)
        i0, i1 = (int(math.floor((v + 9.9) / 0.2 + 0.5)) for v in (lo[0], hi[0]))
        j0, j1 = (int(math.floor((v + 1.9) / 0.2 + 0.5)) for v in (lo[2], hi[2]))
        out.append(int((c[j0 - 1:j1 + 2, i0 - 1:i1 + 2] == d.OCCUPIED).sum()))
    return out


def _fuse_grid(tmp_path, monkeypatch, motion):
    calls = []
    _grid_pipeline(monkeypatch, calls)
    g = d.OccupancyGrid(**MOVING, device="cpu", l_hit=3.5)            # one hit makes a cell occupied
    d.fuse_files(_NoModel(), _items(tmp_path), np.stack([pose(i) for i in range(N_FRAMES)]), g, CALIB, crop=(16, 16),
                 weight=None, motion=motion)
    return g, calls


def test_fuse_files_with_motion_leaves_no_occupied_cells_on_the_movers_path(tmp_path, monkeypatch):
    g, calls = _fuse_grid(tmp_path, monkeypatch, True)
    c = g.classes().numpy()
    assert _footprints(c, range(1, N_FRAMES)) == [0] * (N_FRAMES - 1)
    assert _footprints(c, [0])[0] > 5                                        # frame 0 has no reference
    assert len(calls) == N_FRAMES and calls[0][2] is None and all(k[2] is not None for k in calls[1:])
    ghost, _ = _fuse_grid(tmp_path, monkeypatch, None)
    cg = ghost.classes().numpy()
    assert min(_footprints(cg, range(N_FRAMES))) > 5
    assert int((c == d.FREE).sum()) > 1000


def test_fuse_files_with_a_grid_refuses_ply(tmp_path):
    g = d.OccupancyGrid(**GRID, device="cpu")
    before = _lib.LAUNCHES
    with pytest.raises(ValueError, match="save_map"):
        d.fuse_files(_NoModel(), [], [], g, CALIB, ply=str(tmp_path / "x.ply"))
    assert _lib.LAUNCHES == before


def test_lidar_hint_free_pixels_are_no_depth(monkeypatch):
    """lidar_hints -> reproject -> integrate: a pixel without a hint (disparity 0) has W' = 0 in reproject, so its depth
    is 0, which the grid does not count; the hints alone give the map."""
    monkeypatch.setattr(oc, "_integrate_kernel", _restated_kernel())
    z = render(pose(0), STATIC)
    disp = np.zeros_like(z)
    disp[::6, ::2] = (F32(CALIB.focal_baseline) / z[::6, ::2]).astype(F32)     # a sparse "scan": every 6th row
    _, _, _, depth = RP.reproject(disp[None], Q=CALIB.Q())
    assert (depth[0][disp == 0] == 0).all() and (depth[0][::6, ::2] > 0).all()
    g = d.OccupancyGrid(**GRID, device="cpu", min_hits=1)
    g.integrate(torch.from_numpy(depth), CALIB, pose(0))
    c = g.classes(free=0.45).numpy()                   # one frame: one miss, p = sigmoid(-0.4)
    assert (c[FOOT][0] == d.OCCUPIED).all() and (c[60:80, 105:115] == d.FREE).all()
    grown = np.zeros(c.shape, bool)
    grown[89:97, 104:116] = True
    assert not ((c == d.OCCUPIED) & ~grown).any()


# ---- maps out -------------------------------------------------------------------------------------------------------
def test_save_map_orientation_and_yaml(tmp_path):
    g = d.OccupancyGrid((1.0, -2.0), 0.5, (3, 4), device="cpu")
    g.updates[3, 2] = 1
    g.log_odds[3, 2] = 2.0                  # cell (i=2, j=3): the largest y, so image row 0, column 2
    g.updates[0, 0] = 1
    g.log_odds[0, 0] = -2.0                 # cell (0, 0): the last image row, column 0
    g.updates[1, 1] = 1                     # updated but at p = 0.5: unknown
    pgm, yml = g.save_map(tmp_path / "m")
    data = open(pgm, "rb").read()
    assert data.startswith(b"P5\n3 4\n255\n")
    img = np.frombuffer(data[len(b"P5\n3 4\n255\n"):], np.uint8).reshape(4, 3)
    want = np.full((4, 3), 205, np.uint8)
    want[0, 2] = 0
    want[3, 0] = 254
    assert np.array_equal(img, want)
    y = dict(line.split(": ", 1) for line in open(yml).read().splitlines())
    assert y["image"] == "m.pgm" and y["mode"] == "trinary" and float(y["resolution"]) == 0.5
    assert [float(v) for v in y["origin"].strip("[]").split(",")] == [0.75, -2.25, 0.0]
    assert y["negate"] == "0" and float(y["occupied_thresh"]) == 0.65 and float(y["free_thresh"]) == 0.196


def test_agreement_on_hand_built_grids():
    a = d.OccupancyGrid((0.0, 0.0), 1.0, (4, 2), device="cpu")
    b = d.OccupancyGrid((0.0, 0.0), 1.0, (4, 2), device="cpu")
    #          a: O O F F / F ? O F      b: O F F ? / F O O O
    for g, rows in ((a, ["OOFF", "F?OF"]), (b, ["OFF?", "FOOO"])):
        for j, r in enumerate(rows):
            for i, ch in enumerate(r):
                if ch != "?":
                    g.updates[j, i] = 1
                    g.log_odds[j, i] = 3.0 if ch == "O" else -3.0
    r = a.agreement(b)
    # known in both: 6 cells (not a's (1,1), not b's (3,0)); agree: (0,0) O, (2,0) F, (0,1) F, (2,1) O
    assert (r.known, r.agree, r.occupied_both, r.occupied_either, r.free_both, r.free_either) == (6, 4, 2, 4, 2, 4)
    assert r.occupied_iou == 0.5 and r.free_iou == 0.5 and r.accuracy == pytest.approx(4 / 6)
    e = d.OccupancyGrid((0.0, 0.0), 1.0, (4, 2), device="cpu").agreement(b)
    assert e.known == 0 and math.isnan(e.accuracy) and math.isnan(e.occupied_iou)
    with pytest.raises(ValueError):
        a.agreement(d.OccupancyGrid((0.0, 0.0), 0.5, (4, 2), device="cpu"))


# ---- argument checks ------------------------------------------------------------------------------------------------
def _bad_calls():
    z = torch.ones(1, 8, 10)
    G = dict(GRID, device="cpu")
    g = d.OccupancyGrid(**G)
    c = CALIB
    yield lambda: d.OccupancyGrid((0.0,), 0.2, (10, 10), device="cpu")
    yield lambda: d.OccupancyGrid((0.0, math.nan), 0.2, (10, 10), device="cpu")
    yield lambda: d.OccupancyGrid((0.0, 0.0), 0.0, (10, 10), device="cpu")
    yield lambda: d.OccupancyGrid((0.0, 0.0), 0.2, (0, 10), device="cpu")
    yield lambda: d.OccupancyGrid((0.0, 0.0), 0.2, (1 << 16, 1 << 15), device="cpu")
    yield lambda: d.OccupancyGrid(**G, world_to_grid=np.eye(3))
    yield lambda: d.OccupancyGrid(**G, band=(1.0, 0.5))
    yield lambda: d.OccupancyGrid(**G, band=(0.3, math.nan))
    yield lambda: d.OccupancyGrid(**G, col_width=0)
    yield lambda: d.OccupancyGrid(**G, col_width=65)
    yield lambda: d.OccupancyGrid(**G, range_res=-0.1)
    yield lambda: d.OccupancyGrid(**G, max_depth=math.inf)
    yield lambda: d.OccupancyGrid(**G, max_depth=1000.0, range_res=0.1)
    yield lambda: d.OccupancyGrid(**G, min_hits=0)
    yield lambda: d.OccupancyGrid(**G, min_hits=2.5)
    yield lambda: d.OccupancyGrid(**G, l_hit=0.0)
    yield lambda: d.OccupancyGrid(**G, l_miss=0.1)
    yield lambda: d.OccupancyGrid(**G, l_min=0.5)
    yield lambda: d.OccupancyGrid(**G, l_max=-1.0)
    yield lambda: d.OccupancyGrid(**G, camera_height=math.inf)
    yield lambda: g.integrate(np.ones((1, 8, 10), F32), c, np.eye(4))
    yield lambda: g.integrate(z.double(), c, np.eye(4))
    yield lambda: g.integrate(z, c, np.eye(4), rgb=torch.zeros(1, 8, 10, 3, dtype=torch.uint8))
    yield lambda: g.integrate(z, c, np.eye(4), weight=torch.ones(1, 8, 9))
    yield lambda: g.integrate(z, c, np.eye(4)[None].repeat(2, 0))
    yield lambda: g.integrate(z, c, np.full((4, 4), np.nan))
    yield lambda: g.integrate(z, c, np.eye(4) * 1e300)
    yield lambda: g.integrate(z, c, np.eye(4), window=(0, 0, 8, 11, 0))
    yield lambda: g.integrate(z, c, np.eye(4), max_depth=50.0)
    yield lambda: g.integrate(z, c, np.eye(4), max_depth=0.0)
    yield lambda: g.integrate(torch.ones(0, 8, 10), c, np.zeros((0, 4, 4)))
    yield lambda: g.classes(occupied=0.2, free=0.65)
    yield lambda: g.agreement(fu.TSDFVolume((0.0, 0.0, 0.0), 0.1, (2, 2, 2), colour=False, device="cpu"))


N_BAD = 33


@pytest.mark.parametrize("i", range(N_BAD))
def test_argument_errors_raise_before_any_launch(i):
    calls = list(_bad_calls())
    assert len(calls) == N_BAD
    before = _lib.LAUNCHES
    with pytest.raises(ValueError):
        calls[i]()
    assert _lib.LAUNCHES == before


def test_cpu_tensors_are_refused():
    g = d.OccupancyGrid(**GRID, device="cpu")
    with pytest.raises(_lib.DcaError):
        g.integrate(torch.from_numpy(render(pose(0), STATIC))[None], CALIB, pose(0))


def test_entry_point_rejects_bad_arguments_without_a_device():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    p = 16                                                     # a non-NULL address that is never dereferenced
    M = np.tile(np.eye(4)[:3].reshape(12), (16, 1)).astype(F32)
    nan, inf = math.nan, math.inf
    ok = [p, p, 20, 30, 0.0, 0.0, 0.2, 0, 0, 20, 30, p, None, 10, 80, 1, 8, 10, 700.0, 700.0, 5.0, 4.0, 0, 0,
          M.ctypes.data, M.ctypes.data, 1.65, 0.3, 2.5, 5, 0.1, 40.0, 10, 0.85, -0.4, -2.0, 3.5, p, None]

    def call(**kw):
        args = list(ok)
        for k_, v in kw.items():
            args[int(k_[1:])] = v
        return lib.dca_occupancy_integrate(*args)

    for i in (0, 1, 11, 24, 25, 37):
        assert call(**{f"a{i}": None}) == -1, i
    assert call(a2=0) == call(a3=0) == call(a15=0) == call(a15=17) == call(a16=0) == call(a17=0) == -1
    assert call(a13=9) == call(a14=79) == -1
    assert call(a7=1) == call(a8=-1) == call(a9=0) == call(a10=31) == -1                 # boxes outside the grid
    assert call(a4=nan) == call(a5=nan) == call(a6=0.0) == call(a6=inf) == -1
    assert call(a18=0.0) == call(a19=nan) == call(a20=inf) == call(a21=nan) == -1
    Mbad = M.copy()
    Mbad[0, 3] = nan
    assert call(a24=Mbad.ctypes.data) == call(a25=Mbad.ctypes.data) == -1
    assert call(a26=nan) == call(a27=nan) == call(a28=nan) == call(a27=2.5) == call(a27=3.0) == -1
    assert call(a29=0) == call(a29=65) == call(a30=0.0) == call(a30=nan) == call(a31=inf) == call(a31=0.0) == -1
    assert call(a32=0) == call(a32=(1 << 20) + 1) == -1
    assert call(a33=0.0) == call(a33=nan) == call(a34=0.0) == call(a34=nan) == -1
    assert call(a35=0.0) == call(a36=0.0) == call(a35=nan) == -1
    assert call(a31=1000.0, a30=0.1) == -3                                               # 10,001 range bins
    assert call(a2=1 << 16, a3=1 << 15) == call(a2=1 << 24, a3=1, a10=1) == -3
    assert call(a16=4096, a17=2048, a14=4096 * 2048 * 10, a13=2048) == -3               # 2^23 pixels
    assert call(a22=1 << 24) == call(a23=-(1 << 24)) == -3
