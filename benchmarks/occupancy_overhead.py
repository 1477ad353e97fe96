"""Cost of the occupancy grid at KITTI size: a 375x1242 window with KITTI's intrinsics, the road, wall and static box of
tests/test_occupancy_host.py, the camera 1 m forward per frame, a 4000x4000 grid of 0.2 m cells (800 m x 800 m) with
the default settings.

Prints one JSON line:
  integrate_us_b1 / _b8    one OccupancyGrid.integrate call (memset and three kernels on the frustum box; CUDA-event
                           time of STEPS calls captured in one CUDA graph)
  box_cells_b1 / _b8       cells of the frustum box each call visits
  split_us_b1 / _b8        per kernel of one call (torch.profiler, a separate run)
  fuse_grid_ms_per_frame, fuse_tsdf_ms_per_frame   fuse_files of FRAMES random 375x1242 pairs (GwcNet(192) with the
                           bench weights) into the grid and into a 400x100x400 colour TSDF volume of 0.1 m voxels,
                           alternated ROUNDS times in one process (host clock around each call, which ends in a
                           synchronise; the medians, per frame)
  gpu, power_limit_w       what the numbers were measured on

    python benchmarks/occupancy_overhead.py
"""
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dcanet_b200 as d  # noqa: E402
from confidence_overhead import gpu_name_power  # noqa: E402
from stixel_overhead import _graph_us, _split  # noqa: E402
from test_motion_host import CALIB, pose, render  # noqa: E402
from test_occupancy_host import STATIC  # noqa: E402

FRAMES = 8
ROUNDS = 3
GRID = dict(origin=(-399.9, -399.9), cell_size=0.2, dims=(4000, 4000))


def main():
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    res = {}
    g = d.OccupancyGrid(**GRID, device=dev)
    intr = (CALIB.fx, CALIB.fy, CALIB.cx, CALIB.cy)
    for B in (1, 8):
        z = torch.from_numpy(np.stack([render(pose(i), STATIC) for i in range(B)])).to(dev)
        c2w = np.stack([pose(i) for i in range(B)])
        box = d.occupancy.frustum_box(g.dims, g.origin, g.cell_size, intr, (0, 0, 375, 1242), g.world_to_grid @ c2w,
                                      g.max_depth, g.range_res)
        res[f"box_cells_b{B}"] = box[2] * box[3]
        res[f"integrate_us_b{B}"] = _graph_us(lambda: g.integrate(z, CALIB, c2w))
        res[f"split_us_b{B}"] = _split(lambda: g.integrate(z, CALIB, c2w))
    g.reset()

    import workloads
    from PIL import Image
    net = workloads.init_bench_weights_(d.GwcNet(192), 0).to(dev).eval()
    rng = np.random.default_rng(0)
    with tempfile.TemporaryDirectory() as tmp:
        items = []
        base = rng.integers(0, 256, (375, 1242 + 4 * FRAMES + 8, 3), dtype=np.uint8)
        for i in range(FRAMES):
            for s, o in (("l", 2 * i), ("r", 2 * i + 6)):
                Image.fromarray(np.ascontiguousarray(base[:, o:o + 1242])).save(os.path.join(tmp, f"{s}{i}.png"))
            items.append((os.path.join(tmp, f"l{i}.png"), os.path.join(tmp, f"r{i}.png")))
        poses = np.stack([pose(i) for i in range(FRAMES)])
        vol = d.TSDFVolume((-20.0, -5.0, 0.0), 0.1, (400, 100, 400), device=dev)

        def run(target):
            target.reset()
            torch.cuda.synchronize()
            t = time.perf_counter()
            d.fuse_files(net, items, poses, target, CALIB, max_depth=40.0)
            torch.cuda.synchronize()
            return 1e3 * (time.perf_counter() - t) / FRAMES

        run(g), run(vol)
        a, b = [], []
        for _ in range(ROUNDS):
            a.append(run(g))
            b.append(run(vol))
    res["fuse_grid_ms_per_frame"] = round(float(np.median(a)), 3)
    res["fuse_tsdf_ms_per_frame"] = round(float(np.median(b)), 3)
    res.update(gpu=name, power_limit_w=plimit)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
