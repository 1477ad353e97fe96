"""GPU: TSDF fusion (csrc/tsdf.cu) bit-exact against its float32 restatement (tests/_tsdf_restatement.py): integration at
odd grids with B = 1..3, with and without weights, colour and the weight cap, on pitched views with window offsets and
sub-boxes; the culling box against the whole grid; the ordered extraction on a grid of more than 2,048 tiles and with a
capacity below the count; no host sync and CUDA-graph capture; the forward, reproject, integrate and extract end to
end."""
import importlib
import math

import numpy as np
import pytest
import torch

import _tsdf_restatement as R
from test_tsdf_host import _random_case, _random_pose, look_at

pytestmark = pytest.mark.gpu

fu = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.fusion")
geo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.geometry")
_lib = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200._lib")

F32 = np.float32


def _used_state(rng, dims, colour):
    """A state as after some fusion: tsdf in [-1, 1], weights in [0, 4) (a quarter 0), colours in [0, 255]."""
    s = R.new_state(dims, colour)
    s[0] = rng.uniform(-1, 1, s[0].shape)
    s[1] = np.where(rng.uniform(0, 1, s[1].shape) < 0.25, 0, rng.uniform(0, 4, s[1].shape))
    if colour:
        s[2:] = rng.uniform(0, 255, s[2:].shape)
    return s.astype(F32)


def _pitched(a, pad, dtype=None):
    """A device view of a with `pad` extra columns per row and one extra row per image (pitch != W)."""
    B, H, W = a.shape[:3]
    big = torch.zeros((B, H + 1, W + pad) + a.shape[3:], dtype=dtype or torch.float32, device="cuda")
    big[:, 1:, pad:] = torch.from_numpy(a).cuda()
    return big[:, 1:, pad:]


@pytest.mark.parametrize("B", [1, 2, 3])
@pytest.mark.parametrize("weighted,colour,cap", [(False, False, math.inf), (True, True, math.inf),
                                                 (True, False, 2.5), (False, True, 1.5)])
def test_integrate_equals_the_restatement_exactly(B, weighted, colour, cap):
    rng = np.random.default_rng(B * 10 + weighted * 4 + colour * 2 + (cap < 5))
    dims, origin, vs = (37, 23, 41), (-0.3, 0.15, -0.45), 0.125
    H, W, u0, v0 = 29, 45, 11, -3
    intr = (40.0, 38.5, 20.25, 16.0)
    poses = np.stack([_random_pose(rng, ("inside", "outside", "away")[b % 3] if b else "inside") for b in range(B)])
    depth, weight, rgb = _random_case(rng, B, H, W)
    rgba = np.concatenate([rgb, rng.integers(0, 256, rgb.shape[:3] + (1,), dtype=np.uint8)], -1)
    vol = fu.TSDFVolume(origin, vs, dims, trunc=0.4, colour=colour, max_weight=cap)
    start = _used_state(rng, dims, colour)
    T = np.linalg.inv(poses)[:, :3].reshape(B, 12).astype(F32)
    for box in [(0, 0, 0) + dims, (3, 0, 5, 30, 23, 17), (36, 22, 40, 1, 1, 1)]:
        vol.state.copy_(torch.from_numpy(start))
        fu._integrate_kernel(vol, box, _pitched(depth, 7), _pitched(weight, 7) if weighted else None,
                             _pitched(rgba, 3, torch.uint8) if colour else None, intr, u0, v0, T, 7.5)
        want = R.integrate(start.copy(), origin, vs, depth, T, intr, u0, v0, weight=weight if weighted else None,
                           rgb=rgba if colour else None, trunc=vol.trunc, max_weight=cap, max_depth=7.5, box=box)
        got = vol.state.cpu().numpy()
        assert np.array_equal(got, want, equal_nan=True), box
        assert (got != start).any() or box[3] * box[4] * box[5] == 1
    print("integrate B=%d weighted=%d colour=%d cap=%s: %d voxels updated" % (B, weighted, colour, cap,
                                                                            int((want != start).any(0).sum())))


def test_one_call_of_b_frames_equals_b_calls_and_the_box_equals_the_whole_grid():
    rng = np.random.default_rng(11)
    dims, origin, vs = (41, 19, 33), (0.0, 0.0, 0.0), 0.15
    B, H, W = 5, 24, 40
    calib = geo.StereoCalib(35.0, 33.0, 25.0, 12.0, 0.5)
    poses = np.stack([_random_pose(rng, "inside" if b % 2 else "outside") for b in range(B)])
    depth, weight, rgb = (torch.from_numpy(a).cuda() for a in _random_case(rng, B, H, W))
    win = (2, 6, H, W, 9)
    for max_depth in (None, math.inf, 3.0):
        one = fu.TSDFVolume(origin, vs, dims, trunc=0.45)
        one.integrate(depth, calib, poses, weight=weight, rgb=rgb, window=win, max_depth=max_depth)
        each = fu.TSDFVolume(origin, vs, dims, trunc=0.45)
        for b in range(B):
            each.integrate(depth[b:b + 1], calib, poses[b], weight=weight[b:b + 1], rgb=rgb[b], window=win,
                           max_depth=max_depth)
        assert torch.equal(one.state, each.state)
        whole = fu.TSDFVolume(origin, vs, dims, trunc=0.45)
        T = np.linalg.inv(poses)[:, :3].reshape(B, 12).astype(F32)
        fu._integrate_kernel(whole, (0, 0, 0) + dims, depth, weight, rgb, (35.0, 33.0, 25.0, 12.0), 6, 9, T,
                             math.inf if max_depth is None else max_depth)
        assert torch.equal(one.state, whole.state) and int((one.weight > 0).sum()) > 100


def _extract_raw(vol, min_weight, capacity):
    nx, ny, nz = vol.dims
    tiles = (nx * ny * nz + fu.TILE - 1) // fu.TILE
    ws = torch.empty(tiles, dtype=torch.int64, device="cuda")
    count = torch.empty(1, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    _lib.call("dca_tsdf_count_surface", vol.state.data_ptr(), vol.planes, nx, ny, nz, min_weight, ws.data_ptr(),
              count.data_ptr(), st)
    xyz = torch.full((capacity + 5, 3), -7.0, device="cuda")
    nrm = torch.full((capacity + 5, 3), -7.0, device="cuda")
    rgb = torch.full((capacity + 5, 3), 7, dtype=torch.uint8, device="cuda")
    _lib.call("dca_tsdf_extract_surface", vol.state.data_ptr(), vol.planes, nx, ny, nz, *vol.origin, vol.voxel_size,
              min_weight, ws.data_ptr(), capacity, xyz.data_ptr(), nrm.data_ptr(), rgb.data_ptr(), st)
    return int(count[0]), xyz, nrm, rgb


@pytest.mark.parametrize("dims", [(37, 23, 41), (161, 129, 103)])
def test_extraction_equals_the_restatement_exactly(dims):
    """(161, 129, 103): 2.14M voxels, 2,089 tiles: the scan runs more than two rounds of its CTA."""
    rng = np.random.default_rng(dims[0])
    vol = fu.TSDFVolume((-1.0, 0.5, 2.0), 0.07, dims)
    s = _used_state(rng, dims, True)
    s[0, :, :, : dims[0] // 3] = np.abs(s[0, :, :, : dims[0] // 3])          # a region without crossings
    vol.state.copy_(torch.from_numpy(s))
    for mw in (0.5, 2.0):
        want = R.surface(s, vol.origin, vol.voxel_size, mw)
        got = vol.extract(mw)
        assert got.xyz.shape == (len(want[0]), 3)
        for g, w in zip(got.numpy(), want):
            assert np.array_equal(g, w)
        plain = vol.extract(mw, normals=False, colours=False)
        assert plain.normal is None and plain.rgb is None and torch.equal(plain.xyz, got.xyz)
        n = len(want[0])
        cap = n // 3
        count, xyz, nrm, rgb = _extract_raw(vol, mw, cap)
        assert count == n
        assert np.array_equal(xyz[:cap].cpu().numpy(), want[0][:cap])
        assert np.array_equal(nrm[:cap].cpu().numpy(), want[1][:cap])
        assert np.array_equal(rgb[:cap].cpu().numpy(), want[2][:cap])
        assert (xyz[cap:] == -7).all() and (nrm[cap:] == -7).all() and (rgb[cap:] == 7).all()
        print("extract %s min_weight %.1f: %d points" % (dims, mw, n))


def test_integrate_does_not_synchronise_and_captures_in_a_graph():
    rng = np.random.default_rng(5)
    dims = (64, 32, 48)
    calib = geo.StereoCalib(50.0, 50.0, 32.0, 24.0, 0.5)
    depth, weight, rgb = (torch.from_numpy(a).cuda() for a in _random_case(rng, 2, 48, 64))
    poses = np.stack([_random_pose(rng, "outside") for _ in range(2)])
    vol = fu.TSDFVolume((0.0, 0.0, 0.0), 0.1, dims)
    ref = fu.TSDFVolume((0.0, 0.0, 0.0), 0.1, dims)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for md in (None, 6.0):
            vol.integrate(depth, calib, poses, weight=weight, rgb=rgb, max_depth=md)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    for md in (None, 6.0):
        ref.integrate(depth, calib, poses, weight=weight, rgb=rgb, max_depth=md)
    assert torch.equal(vol.state, ref.state)
    vol.reset()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            for md in (None, 6.0):
                vol.integrate(depth, calib, poses, weight=weight, rgb=rgb, max_depth=md)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(vol.state, ref.state) and int((vol.weight > 0).sum()) > 0


def test_forward_reproject_integrate_extract_equals_the_restatement():
    import dcanet_b200 as d
    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(48), 0).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(0)
    left = torch.randn(1, 3, 64, 128, device="cuda", generator=g)
    right = torch.roll(left, -4, 3) + 0.1 * torch.randn(1, 3, 64, 128, device="cuda", generator=g)
    calib = geo.StereoCalib(100.0, 100.0, 64.0, 32.0, 0.5)
    with torch.no_grad():
        pred, _, conf, lr = net(left, right, confidence=True, lr_check=True)
    win = (4, 2, 60, 124, 4)
    pc = geo.reproject(pred, calib, confidence=conf.peak, min_confidence=0.05, label=lr.label, window=win,
                       max_depth=60.0)
    peak = conf.peak[:, 0, 4:64, 2:126]
    rgb = torch.randint(0, 256, (1, 60, 124, 3), dtype=torch.uint8, device="cuda", generator=g)
    poses = np.stack([np.eye(4), look_at(np.array([0.4, 0.0, 0.2]), np.array([0.0, 0.0, 12.0]))])
    Z = pc.depth[pc.depth > 0]
    lo, hi = float(Z.min()), float(Z.max())
    vol = fu.TSDFVolume((-0.6 * hi, -0.4 * hi, 0.5 * lo), hi / 100, (121, 81, 101), trunc=hi / 25)
    for p in poses:
        vol.integrate(pc.depth, calib, p, weight=peak, rgb=rgb[0], window=win, max_depth=60.0)
    surf = vol.extract(0.1)
    s = R.new_state(vol.dims)
    T = np.linalg.inv(poses)[:, :3].reshape(2, 12).astype(F32)
    for b in range(2):
        R.integrate(s, vol.origin, vol.voxel_size, pc.depth.cpu().numpy(), T[b:b + 1], (100.0, 100.0, 64.0, 32.0), 2, 4,
                    weight=peak.cpu().numpy(), rgb=rgb.cpu().numpy(), trunc=vol.trunc, max_depth=60.0)
    assert np.array_equal(vol.state.cpu().numpy(), s)
    want = R.surface(s, vol.origin, vol.voxel_size, 0.1)
    for got, w in zip(surf.numpy(), want):
        assert np.array_equal(got, w)
    assert len(want[0]) > 100
    print("forward + reproject + 2 poses: %d of %d pixels with depth, %d surface points" % (
        int((pc.depth > 0).sum()), 60 * 124, len(want[0])))
