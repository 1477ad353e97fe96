"""Cost of camera tracking against a fused volume at KITTI size, on the scene and grid of tsdf_overhead.py: a 375x1242
window with KITTI's intrinsics, an 800x64x800 grid of 0.1 m voxels with colour, max_depth 40 m, synthetic depth maps (a
ground plane and a wall of boxes, 1 % noise) on a forward-driving trajectory; 8 frames are fused at their poses first.

Prints one JSON line:
  raycast_us          one dca_tsdf_raycast of the window (CUDA-event time of STEPS calls captured in one CUDA graph)
  icp_us              one dca_icp_track call with the default levels (4, 10), (2, 5), (1, 4): 19 iterations, 38
                      launches, timed the same way; icp_us_per_iteration = icp_us / 19
  icp_reduce_us, icp_solve_us   per launch of each kernel at each stride (torch.profiler, a separate run)
  track_ms            Tracker.track end to end (raycast, ICP, the D2H copy and its one sync, the host work), host clock
                      over STEPS_TRACK calls
  track_files_pairs_per_s, fuse_files_pairs_per_s   the forward (GwcNet(192), bench weights) on PAIRS synthetic pairs
                      written as PNGs: track_files from the first pose, fuse_files with the known poses
  gpu, power_limit_w  what the numbers were measured on

    python benchmarks/tracking_overhead.py
"""
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dcanet_b200 as d  # noqa: E402
from confidence_overhead import gpu_name_power  # noqa: E402
from tsdf_overhead import CX, CY, FX, FY, H, MAX_DEPTH, W, _depth_maps, _graph_us  # noqa: E402

STEPS_TRACK = 50
PAIRS = 24


def _profile_split(call, dev):
    """Mean device time per launch of each kernel of `call()` (torch.profiler, 5 calls)."""
    from torch.profiler import ProfilerActivity, profile
    call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            call()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if "icp_" in e.key or "raycast" in e.key:
            out[e.key.split("(")[0].split("::")[-1]] = (e.count, round(e.device_time_total / max(e.count, 1), 3))
    return out


def _pairs_per_s(fn, items, reps=1):
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        fn(items)
    torch.cuda.synchronize()
    return round(reps * len(items) / (time.perf_counter() - t), 2)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("tracking_overhead.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    calib = d.StereoCalib(FX, FY, CX, CY, 0.54)
    dims = (800, 64, 800)
    vol = d.TSDFVolume((-40.0, -4.6, -2.0), 0.1, dims, device=dev)
    poses = np.tile(np.eye(4), (10, 1, 1))
    poses[:, 2, 3] = np.arange(10) * 1.0
    poses[:, 0, 3] = np.sin(np.arange(10) * 0.3) * 0.5
    depth = _depth_maps(dev, 10, 0)
    g = torch.Generator(device=dev).manual_seed(1)
    weight = torch.rand((10, H, W), device=dev, generator=g) * 0.5 + 0.5
    rgb = torch.randint(0, 256, (10, H, W, 3), dtype=torch.uint8, device=dev, generator=g)
    vol.integrate(depth[:8], calib, poses[:8], weight=weight[:8], rgb=rgb[:8], max_depth=MAX_DEPTH)

    trk = d.Tracker(vol, calib, (H, W), pose=poses[7], max_depth=MAX_DEPTH)
    intr = trk.intrinsics
    M = poses[7][:3].reshape(12).astype(np.float32)
    A0 = np.linalg.solve(poses[7], poses[8])[:3].reshape(12)
    pose, stats, ok = trk._views(trk._out)

    def raycast():
        d.fusion._raycast_kernel(vol, intr, 0, 0, M, 0.5, 0.0, MAX_DEPTH, trk.model)

    def icp():
        d.tracking._icp_kernel(depth[8], weight[8], intr, 0, 0, MAX_DEPTH, trk.model, A0, trk.levels, 100,
                               trk.workspace, pose, stats, ok)

    raycast_us = _graph_us(raycast)
    icp_us = _graph_us(icp)
    n_it = trk.iterations
    split = _profile_split(lambda: (raycast(), icp()), dev)
    torch.cuda.synchronize()
    hits = int((trk.model.depth > 0).sum())
    inl = stats[:, 0].cpu().numpy().astype(int).tolist()

    # Tracker.track end to end (each call raycasts at the same reference pose: the pose is reset after every call)
    for _ in range(3):
        trk.pose = poses[7]
        trk.track(depth[8], weight[8], init=poses[8])
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(STEPS_TRACK):
        trk.pose = poses[7]
        r = trk.track(depth[8], weight[8], init=poses[8])
    track_ms = round(1e3 * (time.perf_counter() - t) / STEPS_TRACK, 3)
    err = float(np.linalg.norm(r.cam_to_world[:3, 3] - poses[8][:3, 3]))

    # pairs per second: the forward on synthetic pairs (a shifted noise texture), track_files against fuse_files
    import workloads
    from PIL import Image
    net = workloads.init_bench_weights_(d.GwcNet(192), 0).to(dev).eval()
    rng = np.random.default_rng(0)
    base = rng.integers(0, 256, (H, W + 64 + PAIRS, 3), dtype=np.uint8)
    with tempfile.TemporaryDirectory() as tmp:
        items = []
        for i in range(PAIRS):
            for side, x0 in (("l", i + 32), ("r", i)):
                Image.fromarray(np.ascontiguousarray(base[:, x0:x0 + W])).save(os.path.join(tmp, f"{side}{i}.png"))
            items.append((os.path.join(tmp, f"l{i}.png"), os.path.join(tmp, f"r{i}.png")))
        known = np.tile(np.eye(4), (PAIRS, 1, 1))
        known[:, 2, 3] = np.arange(PAIRS) * 0.5
        box = dict(origin=(-40.0, -4.6, -2.0), voxel_size=0.1, dims=dims, device=dev)
        fv, tv = d.TSDFVolume(**box), d.TSDFVolume(**box)
        d.fuse_files(net, items[:3], known[:3], fv, calib, max_depth=MAX_DEPTH)            # warm-up
        d.track_files(net, items[:3], tv, calib, max_depth=MAX_DEPTH)
        fuse_pps = _pairs_per_s(lambda it: d.fuse_files(net, it, known, fv.reset(), calib, max_depth=MAX_DEPTH),
                                items)
        track_pps = _pairs_per_s(lambda it: d.track_files(net, it, tv.reset(), calib, max_depth=MAX_DEPTH), items)
        traj = d.track_files(net, items, tv.reset(), calib, max_depth=MAX_DEPTH)
    print(json.dumps({
        "workload": f"{H}x{W} window, KITTI intrinsics, grid {dims} x 0.1 m with colour, max_depth {MAX_DEPTH} m, "
                    f"8 fused synthetic frames, the 9th tracked",
        "gpu": name, "power_limit_w": plimit,
        "raycast_us": raycast_us, "raycast_hits": hits,
        "icp_us": icp_us, "icp_iterations": n_it, "icp_us_per_iteration": round(icp_us / n_it, 3),
        "icp_inliers_per_iteration": inl, "profiler_us_per_launch": split,
        "track_ms": track_ms, "track_translation_error_m": round(err, 5),
        "fuse_files_pairs_per_s": fuse_pps, "track_files_pairs_per_s": track_pps,
        "track_files_ok": int(traj.ok.sum()), "pairs": PAIRS, "steps": 200,
    }), flush=True)


if __name__ == "__main__":
    main()
