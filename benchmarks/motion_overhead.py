"""Cost of the moving-object test at KITTI size: a 375x1242 window with KITTI's intrinsics, a road, a wall at 60 m and a
box approaching at 2 m per frame beyond the camera's 1 m (tests/test_motion_host.py's scene), the default thresholds.

Prints one JSON line:
  labels_us_b1 / _b8       one dca_motion_labels call (CUDA-event time of STEPS calls captured in one CUDA graph)
  components_us_b1 / _b8   one dca_motion_components call (eight launches), timed the same way
  motion_us_b1 / _b8       one motion() call (both, and the output allocations), timed the same way
  split_us_b1              per kernel of one motion() call at B = 1 (torch.profiler, a separate run)
  fuse_ms_per_frame, fuse_motion_ms_per_frame   fuse_files of FRAMES random 375x1242 pairs (GwcNet(192) with the
                           bench weights, a 400x100x400 colour volume of 0.1 m voxels), without and with motion=True,
                           alternated ROUNDS times in one process (host clock around each call, which ends in a
                           synchronise; the medians, per frame)
  gpu, power_limit_w       what the numbers were measured on

    python benchmarks/motion_overhead.py
"""
import importlib
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
from test_motion_host import CALIB, _moving_box, pose  # noqa: E402

mo = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.motion")

FRAMES = 8
ROUNDS = 3


def main():
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    res = {}
    prev1, cur1, _ = _moving_box([0.0, 0.0, 10.0], [0.0, 0.0, -2.0])
    A1 = np.linalg.solve(pose(0), pose(1))
    intr = (CALIB.fx, CALIB.fy, CALIB.cx, CALIB.cy)
    fB = CALIB.focal_baseline
    for B in (1, 8):
        cur = torch.from_numpy(np.stack([cur1] * B)).to(dev)
        prev = torch.from_numpy(np.stack([prev1] * B)).to(dev)
        A = np.stack([A1] * B)
        m = d.motion(cur, prev, CALIB, A)
        Af = A[:, :3].reshape(B, 12).astype(np.float32)
        res[f"labels_us_b{B}"] = _graph_us(lambda: mo._labels_kernel(cur, prev, intr, fB, 0.0, 0, 0, Af, 3.0, 0.05, 1,
                                                                     m.label, m.residual))
        res[f"components_us_b{B}"] = _graph_us(lambda: mo._components_kernel(cur, m.label, m.residual, intr, fB, 0.0,
                                                                             0, 0, 1.0, 100, m.instance, m.objects))
        res[f"motion_us_b{B}"] = _graph_us(lambda: d.motion(cur, prev, CALIB, A))
        if B == 1:
            res["objects_b1"] = int(m.objects.counts()[0])
            res["split_us_b1"] = _split(lambda: d.motion(cur, prev, CALIB, A))

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

        def run(motion):
            vol.reset()
            torch.cuda.synchronize()
            t = time.perf_counter()
            d.fuse_files(net, items, poses, vol, CALIB, max_depth=40.0, motion=motion)
            torch.cuda.synchronize()
            return 1e3 * (time.perf_counter() - t) / FRAMES

        run(None), run(True)
        a, b = [], []
        for _ in range(ROUNDS):
            a.append(run(None))
            b.append(run(True))
    res["fuse_ms_per_frame"] = round(float(np.median(a)), 3)
    res["fuse_motion_ms_per_frame"] = round(float(np.median(b)), 3)
    res.update(gpu=name, power_limit_w=plimit)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
