"""CPU-only: the stixel model of include/dca_b200.h section 15 through its numpy restatement (DP optimality, a synthetic
driving scene, a scene without a road), and the argument checks of the Python API, which raise before any launch.

The scene bounds are measured values with a margin; they say nothing about KITTI or any real camera."""
import math

import numpy as np
import pytest
import torch

import _stixel_restatement as R
import dcanet_b200 as d


# ---- the DP is exact without the disparity-dependent priors -----------------------------------------------------
@pytest.mark.parametrize("seed", range(12))
def test_dp_equals_exhaustive_minimum(seed):
    rng = np.random.default_rng(seed)
    H = int(rng.integers(1, 9))
    q = rng.integers(0, 40 * 256, H).astype(np.int64)
    q[rng.random(H) < 0.25] = -1                                         # invalid rows
    g = np.where(rng.random(H) < 0.7, rng.integers(1, 40 * 256, H), 0).astype(np.int64)
    pr = dict(R.DEFAULTS, p_gravity=0, p_order=0, p_seg=int(rng.integers(0, 20000)),
              s_ground=int(rng.integers(64, 1024)), s_object=int(rng.integers(64, 1024)),
              s_sky=int(rng.integers(64, 1024)))
    C, BP, DM = R.dp(q[None], g[None], 40, **pr)
    best = min(e for e in (R.segmentation_energy(q, g, s, 40, **pr) for s in R.all_segmentations(H)) if e is not None)
    assert C[0, H - 1].min() == best
    segs = R.backtrack(C, BP, DM, H)[0]
    assert R.segmentation_energy(q, g, [(nb, nt, c) for nb, nt, c, _ in segs], 40, **pr) == best


def test_cost_floor_matches_the_fp64_formula():
    """The kernel floors a correctly rounded fp64 quotient; below the truncation it equals the integer floor."""
    rng = np.random.default_rng(0)
    for s in (1, 3, 255, 256, 257, 4095, 16384):
        for tau in (1, 3, 8):
            r = rng.integers(0, tau * s + 1, 2000)
            exact = R.cost(r, s, tau)
            with np.errstate(divide="ignore"):
                viafp = np.where(r >= tau * s, tau * tau * 1024,
                                 np.floor((r * r * 1024).astype(np.float64) / float(s * s)).astype(np.int64))
            assert (exact == viafp).all()


# ---- synthetic driving scene ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scene():
    disp, info = R.driving_scene(0)
    prof, line, inl, ok = R.ground_profile(disp[None])
    st = R.stixels(disp[None], prof, width=5)
    return disp, info, prof, line, ok, st


def test_ground_line_on_the_synthetic_road(scene):
    # measured: horizon 159.72 against 160.26 (0.54 rows), slope 0.32172 against 0.32280 (0.33 %)
    _, info, _, line, ok, _ = scene
    assert ok[0]
    assert abs(line[0, 1] - info["yh"]) <= 1.0
    assert abs(line[0, 0] / info["a"] - 1) <= 0.01


def test_boxes_become_one_object_each(scene):
    """Each column lying wholly inside a box holds exactly one object segment over the box's rows.  Measured over the
    104 such columns: top within 1 row, bottom within 4 rows (the road at the foot has nearly the box's disparity),
    free space within 5 rows of the foot, disparity error median 0.01 px and max 1.98 px (the segment's disparity is the
    mean of its samples, which an outlier row pulls)."""
    disp, info, _, _, _, st = scene
    H, W = disp.shape
    errs = []
    for bx in info["boxes"]:
        for k in range(st["count"].shape[1]):
            if not (5 * k >= bx["u0"] and min(5 * k + 4, W - 1) <= bx["u1"]):
                continue
            segs = [(H - 1 - nt, H - 1 - nb, c, m / 256) for nb, nt, c, m in st["segs"][k]]
            hits = [s for s in segs if s[2] == R.OBJECT and s[0] <= bx["foot"] and s[1] >= bx["top"]
                    and abs(s[3] - bx["disp"]) < 3]
            assert len(hits) == 1, (k, segs)
            top, bottom, _, m = hits[0]
            assert abs(top - bx["top"]) <= 2, (k, segs)
            assert abs(bottom - bx["foot"]) <= 6, (k, segs)
            assert abs(int(st["free_space"][0, k]) - bx["foot"]) <= 7, (k, segs)
            errs.append(abs(m - bx["disp"]))
    assert len(errs) == 104
    assert np.median(errs) <= 0.1 and max(errs) <= 2.5


def test_road_columns_start_with_ground(scene):
    disp, info, _, _, _, st = scene
    W = disp.shape[1]
    road = [k for k in range(st["count"].shape[1])
            if all(min(5 * k + 4, W - 1) < bx["u0"] or 5 * k > bx["u1"] for bx in info["boxes"])]
    assert len(road) > 100
    for k in road:
        assert st["segs"][k][0][2] == R.GROUND, (k, st["segs"][k])
        assert abs(int(st["free_space"][0, k]) - info["wall_foot"]) <= 4       # measured: at most 2.9 rows


def test_render_follows_the_segments(scene):
    disp, _, prof, _, _, st = scene
    out, cls = R.render(st, prof, disp.shape[1], 5)
    k = 30                                           # a column of the nearest box
    for nb, nt, c, m in st["segs"][k]:
        y = disp.shape[0] - 1 - nt
        assert cls[0, y, 5 * k] == c
        assert out[0, y, 5 * k] == (prof[0, y] if c == R.GROUND else np.float32(m) / 256 if c == R.OBJECT else 0)


def test_no_road_gives_objects_and_sky():
    disp, _ = R.driving_scene(1, road=False)
    prof, line, inl, ok = R.ground_profile(disp[None])
    assert not ok[0] and (prof == 0).all() and (line == 0).all()
    st = R.stixels(disp[None], prof, width=5)
    assert (st["cls"][st["cls"] >= 0] != R.GROUND).all()
    assert (st["free_space"] == disp.shape[0]).all()


# ---- argument checks -----------------------------------------------------------------------------------------------
def _bad_calls():
    disp = torch.zeros(1, 8, 10)
    prof = torch.zeros(1, 8)
    yield lambda: d.ground_profile(np.zeros((1, 8, 10), np.float32))
    yield lambda: d.ground_profile(disp.double())
    yield lambda: d.ground_profile(torch.zeros(8, 10))
    yield lambda: d.ground_profile(disp, confidence=torch.zeros(1, 8, 9))
    yield lambda: d.ground_profile(disp, label=torch.zeros(1, 8, 10))
    yield lambda: d.ground_profile(disp, confidence=torch.zeros(1, 8, 10), min_confidence=math.nan)
    yield lambda: d.ground_profile(disp, max_disp=0)
    yield lambda: d.ground_profile(disp, max_disp=1025)
    yield lambda: d.ground_profile(disp, max_disp=19.5)
    yield lambda: d.ground_profile(disp, min_inliers=0)
    yield lambda: d.ground_profile(disp, window=(0, 0, 9, 10, 0))
    yield lambda: d.ground_profile(disp, window=(-1, 0, 8, 10, 0))
    yield lambda: d.ground_profile(torch.zeros(1, 4097, 1))
    yield lambda: d.stixels(disp, prof, width=0)
    yield lambda: d.stixels(disp, prof, width=17)
    yield lambda: d.stixels(disp, prof, width=True)
    yield lambda: d.stixels(disp, prof, max_disp=2000)
    yield lambda: d.stixels(disp, prof, sigma_ground=0.0)
    yield lambda: d.stixels(disp, prof, sigma_object=math.inf)
    yield lambda: d.stixels(disp, prof, sigma_sky=math.nan)
    yield lambda: d.stixels(disp, prof, sigma_sky=65.0)
    yield lambda: d.stixels(disp, prof, tau=0)
    yield lambda: d.stixels(disp, prof, tau=9)
    yield lambda: d.stixels(disp, prof, p_seg=-1)
    yield lambda: d.stixels(disp, prof, p_gravity=(1 << 20) + 1)
    yield lambda: d.stixels(disp, prof, p_order=1.5)
    yield lambda: d.stixels(disp, prof, eps_gravity=-1.0)
    yield lambda: d.stixels(disp, prof, eps_order=math.nan)
    yield lambda: d.stixels(disp, torch.zeros(1, 9))
    yield lambda: d.stixels(disp, torch.zeros(1, 8, dtype=torch.float64))
    yield lambda: d.stixels(disp, "ground")
    yield lambda: d.stixels(disp, prof, window=(0, 0, 8, 11, 0))
    yield lambda: d.stixels(disp, prof, confidence=torch.zeros(1, 8, 10), min_confidence=math.nan)
    yield lambda: d.stixels(torch.zeros(1, 769, 4), torch.zeros(1, 769))


@pytest.mark.parametrize("i", range(34))
def test_argument_errors_raise_before_any_launch(i):
    calls = list(_bad_calls())
    assert len(calls) == 34
    before = d._lib.LAUNCHES
    with pytest.raises(ValueError):
        calls[i]()
    assert d._lib.LAUNCHES == before


def test_cpu_tensors_are_refused():
    with pytest.raises(d._lib.DcaError):
        d.ground_profile(torch.zeros(1, 8, 10))
    with pytest.raises(d._lib.DcaError):
        d.stixels(torch.zeros(1, 8, 10), torch.zeros(1, 8))
