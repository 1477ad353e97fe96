"""GPU: the occupancy-grid kernels (csrc/occupancy.cu) bit-exact against their restatement
(tests/_occupancy_restatement.py) at KITTI size for 1, 3 and 17 frames, with pitched windows, holes, odd weights, empty
boxes and frames at the grid's edge; the frustum box against the whole grid; CUDA-graph capture; fuse_files(volume=grid)
on the real forward against a serial loop; and the LiDAR reference path."""
import importlib

import numpy as np
import pytest
import torch
from PIL import Image

import _occupancy_restatement as R
from test_motion_host import CALIB, INTR, _moving_box, pose, render
from test_occupancy_host import GRID, STATIC, classes, mats

pytestmark = pytest.mark.gpu

oc = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.occupancy")
geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
mo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.motion")
io = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.kitti_io")

F32 = np.float32


def _case(B, seed):
    """B (depth, weight, camera-to-world) at 375 x 1242: a box, depth noise, holes (0 and NaN), weights with NaN,
    negative values and values above 1, and poses perturbed around the camera's."""
    rng = np.random.default_rng(seed)
    zs, ws, ps = [], [], []
    start = np.array([rng.uniform(-4, 4), 0.0, rng.uniform(8, 20)])
    _, z0, _ = _moving_box(start, np.array([rng.uniform(-1, 1), 0.0, rng.uniform(-2, 2)]))
    for b in range(B):
        z = z0.copy()
        z *= (1 + rng.normal(0, 0.01, z.shape)).astype(F32)
        z[rng.random(z.shape) < 0.02] = 0
        z[rng.random(z.shape) < 0.01] = np.nan
        w = rng.uniform(-0.2, 1.3, z.shape).astype(F32)
        w[rng.random(z.shape) < 0.01] = np.nan
        p = pose(1)
        p[:3, 3] += rng.normal(0, 0.05, 3)
        zs.append(z)
        ws.append(w)
        ps.append(p)
    return np.stack(zs), np.stack(ws), np.stack(ps)


def _restated(z, w, c2w, u0=0, v0=0, L=None, U=None, **kw):
    """The restatement in calls of 16 frames over the whole grid."""
    L = np.zeros(GRID["dims"][::-1], F32) if L is None else L
    U = np.zeros(GRID["dims"][::-1], np.int32) if U is None else U
    M, Mi = mats(c2w)
    for s in range(0, len(z), 16):
        R.integrate(L, U, GRID["origin"], GRID["cell_size"], z[s:s + 16], M[s:s + 16], Mi[s:s + 16], INTR, u0, v0,
                    weight=None if w is None else w[s:s + 16], **kw)
    return L, U


def _equal(g, L, U):
    assert np.array_equal(g.log_odds.cpu().numpy(), L) and np.array_equal(g.updates.cpu().numpy(), U)


@pytest.mark.parametrize("B,seed", [(1, 0), (3, 1), (17, 2)])
def test_kernels_equal_the_restatement_at_kitti_size(B, seed):
    z, w, c2w = _case(B, seed)
    g = d_grid()
    g.integrate(torch.from_numpy(z).cuda(), CALIB, c2w, weight=torch.from_numpy(w).cuda())
    L, U = _restated(z, w, c2w)
    _equal(g, L, U)
    c = classes(L, U)
    print("B=%d: %d updated, %d occupied, %d free" % (B, (U > 0).sum(), (c == 1).sum(), (c == 0).sum()))
    assert (L > 0).sum() > 5 and (L < 0).sum() > 1000                     # hits and misses both reached the grid
    # the whole grid as one box gives the same
    g2 = d_grid()
    M, Mi = mats(c2w)
    for s in range(0, B, 16):
        oc._integrate_kernel(g2, (0, 0) + GRID["dims"], torch.from_numpy(z[s:s + 16]).cuda(),
                             torch.from_numpy(w[s:s + 16]).cuda(), INTR, 0, 0, M[s:s + 16], Mi[s:s + 16], g2.max_depth)
    assert torch.equal(g.log_odds, g2.log_odds) and torch.equal(g.updates, g2.updates)


def d_grid(**kw):
    return oc.OccupancyGrid(**GRID, **kw)


def test_a_pitched_window_and_other_settings():
    z, w, c2w = _case(3, 3)
    big = np.zeros((3, 400, 1300), F32)
    big[:, 10:385, 20:1262] = z
    bw = np.full((3, 400, 1300), 0.7, F32)
    bw[:, 10:385, 20:1262] = w
    dz, dw = torch.from_numpy(big).cuda(), torch.from_numpy(bw).cuda()
    kw = dict(camera_height=1.6, band=(0.2, 1.5), col_width=3, range_res=0.25, max_depth=30.0, min_hits=3, l_hit=1.2,
              l_miss=-0.3, l_min=-1.5, l_max=2.0)
    g = d_grid(**kw)
    u = (0, 100, 200, 600, 175)                        # (y0, x0, h, w, v_origin): image rows 175..374
    g.integrate(dz[:, 185:385, 120:720], CALIB, c2w, weight=dw[:, 185:385, 120:720], window=u)
    g.integrate(dz[:, 185:385, 120:720], CALIB, c2w, window=u, max_depth=20.0)
    rk = dict(camera_height=1.6, band=(0.2, 1.5), col_width=3, range_res=0.25, min_hits=3, l_hit=1.2, l_miss=-0.3,
              l_min=-1.5, l_max=2.0)
    L, U = _restated(z[:, 175:375, 100:700], w[:, 175:375, 100:700], c2w, 100, 175, max_depth=30.0, **rk)
    L, U = _restated(z[:, 175:375, 100:700], None, c2w, 100, 175, L, U, max_depth=20.0, **rk)
    _equal(g, L, U)
    assert (L > 0).sum() > 5 and (L < 0).sum() > 1000


def test_empty_boxes_and_frames_at_the_grid_edge():
    z = np.stack([render(pose(i), STATIC) for i in range(3)])
    away = pose(0)
    away[:3, :3] = np.diag([-1.0, 1.0, -1.0])          # looking backwards from Z = -30: no cell of the grid
    away[2, 3] = -30.0
    edge = pose(0)
    edge[0, 3] = 19.0                                   # 1 m inside the grid's right edge
    corner = pose(0)
    corner[0, 3], corner[2, 3] = -19.5, 55.0            # near the far-left corner, looking out of the grid
    c2w = np.stack([away, edge, corner])
    g = d_grid()
    g.integrate(torch.from_numpy(z).cuda(), CALIB, c2w)
    L, U = _restated(z, None, c2w)
    _equal(g, L, U)
    assert (U > 0).sum() > 1000
    before = g.log_odds.clone()
    g.integrate(torch.from_numpy(z[:1]).cuda(), CALIB, away)            # no launch
    assert torch.equal(before, g.log_odds)


def test_graph_capture_equals_eager():
    z, w, c2w = _case(4, 5)
    dz, dw = torch.from_numpy(z).cuda(), torch.from_numpy(w).cuda()
    eager = d_grid().integrate(dz, CALIB, c2w, weight=dw)
    g = d_grid()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        g.integrate(dz, CALIB, c2w, weight=dw)                          # warm-up on the side stream
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g.integrate(dz, CALIB, c2w, weight=dw)
    g.reset()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(eager.log_odds, g.log_odds) and torch.equal(eager.updates, g.updates)
    graph.replay()                                                       # a second replay adds the frames again
    twice = d_grid().integrate(torch.cat([dz, dz]), CALIB, np.concatenate([c2w, c2w]),
                               weight=torch.cat([dw, dw]))
    torch.cuda.synchronize()
    assert torch.equal(twice.log_odds, g.log_odds) and torch.equal(twice.updates, g.updates)


def _pairs(tmp_path):
    rng = np.random.default_rng(0)
    items = []
    base = rng.integers(0, 256, (64, 150, 3), dtype=np.uint8)
    for i in range(4):
        left = np.ascontiguousarray(base[:, 2 * i:2 * i + 128])
        right = np.ascontiguousarray(base[:, 2 * i + 4:2 * i + 132])
        left[20:40, 30 + 6 * i:60 + 6 * i] = 255 - 40 * i                 # a patch that moves between the pairs
        Image.fromarray(left).save(tmp_path / f"l{i}.png")
        Image.fromarray(right).save(tmp_path / f"r{i}.png")
        items.append((str(tmp_path / f"l{i}.png"), str(tmp_path / f"r{i}.png")))
    return items


def test_fuse_files_with_a_grid_equals_a_serial_loop(tmp_path):
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    calib = geo.StereoCalib(100.0, 100.0, 64.0, 32.0, 0.5)
    items = _pairs(tmp_path)
    grid = dict(origin=(-20.0, -5.0), cell_size=0.5, dims=(80, 110), camera_height=1.0, band=(0.2, 3.0), min_hits=1,
                max_depth=45.0)
    poses = np.stack([np.eye(4)] * 4)
    for i in range(4):
        poses[i, 0, 3] = 0.05 * i
    win = (0, 0, 64, 128, 0)
    for motion_kw in (None, dict(min_pixels=5, tau=1.0)):
        g = oc.OccupancyGrid(**grid)
        d.fuse_files(net, items, poses, g, calib, crop=(64, 128), motion=motion_kw)
        ref = oc.OccupancyGrid(**grid)
        last, masked = None, 0
        for i, it in enumerate(items):
            pair = io.load_pair(*it)
            with torch.no_grad():
                out = net(torch.from_numpy(pair[None, 0:3]).cuda(), torch.from_numpy(pair[None, 3:6]).cuda(),
                          confidence=True)
            pc = geo.reproject(out[0], calib, window=win)
            wmap = out[2].peak[:, 0]
            if motion_kw is not None and last is not None:
                m = mo.motion(pc.depth, last[0], calib, np.linalg.solve(last[1], poses[i]), window=win, **motion_kw)
                wmap = torch.where(m.instance == 0, wmap, torch.zeros((), device=wmap.device))
                masked += int((m.instance > 0).sum())
            ref.integrate(pc.depth, calib, poses[i], weight=wmap, window=win)
            last = (pc.depth, poses[i])
        print("fuse_files(volume=grid, motion=%s): %d updated cells, %d pixels masked"
              % (motion_kw, int((ref.updates > 0).sum()), masked))
        assert torch.equal(g.log_odds, ref.log_odds) and torch.equal(g.updates, ref.updates)
        assert int((ref.updates > 0).sum()) > 50


def test_the_lidar_reference_path():
    """Synthetic velodyne points of the static scene -> lidar_hints -> reproject -> integrate with min_hits = 1: pixels
    without a hint reach the grid as no depth, and the box's front is occupied."""
    import dcanet_b200 as d
    v2r = np.array([[0, -1, 0, 0], [0, 0, -1, 0], [1, 0, 0, 0]], F32)      # velodyne x forward, y left, z up
    calib = geo.StereoCalib(CALIB.fx, CALIB.fy, CALIB.cx, CALIB.cy, CALIB.baseline, velo_to_rect=v2r)
    z = render(pose(0), STATIC)
    ys, xs = np.mgrid[0:375:6, 0:1242:2]
    zz = z[ys, xs].astype(np.float64)
    keep = (zz > 0) & (zz < 70)
    X = (xs[keep] - CALIB.cx) / CALIB.fx * zz[keep]
    Y = (ys[keep] - CALIB.cy) / CALIB.fy * zz[keep]
    pts = np.stack([zz[keep], -X, -Y, np.zeros_like(X)], 1).astype(F32)
    hints = d.lidar_hints(torch.from_numpy(pts), calib, (375, 1242), max_depth=70.0)
    pc = d.reproject(hints, calib)
    depth = pc.depth.cpu().numpy()
    h = hints[:, 0].cpu().numpy()
    assert (depth[h == 0] == 0).all() and (depth[h > 0] > 0).all() and (h > 0).sum() > 20000
    g = d_grid(min_hits=1)
    g.integrate(pc.depth, calib, pose(0))
    L, U = _restated(depth, None, pose(0)[None], min_hits=1)
    _equal(g, L, U)
    c = g.classes(free=0.45).cpu().numpy()
    assert (c[90, 105:115] == d.OCCUPIED).all() and (c[60:80, 105:115] == d.FREE).all()
