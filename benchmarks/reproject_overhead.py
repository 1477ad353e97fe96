"""Cost of the reprojection to depth and points (dca_reproject) and of the depth errors (dca_depth_metrics) at KITTI size,
384x1248, maxdisp 192, parity precision, synthetic weights.

Prints one JSON line:
  reproject_us         one dca_reproject call (its count and scatter launches) on the forward's pred4, per call: `graph` =
                       CUDA-event time of STEPS calls captured in one CUDA graph, `eager` = CUDA-event time of STEPS calls
                       launched one by one; `plain` without filters, `filtered` with the peak (>= 0.3) and the left-right
                       label filters and the velodyne transform
  depth_metrics_us     one dca_depth_metrics over the same pred4 against a seeded GT map, measured the same way
  bytes_est            bytes each kernel moves per pair, from the shapes and the kept count, and the time that takes at
                       7.7 TB/s
  kept_fraction        share of the pixels kept by each reprojection (synthetic weights: says nothing about accuracy)
  files_pairs_per_s    ImagePipeline.run against reproject_files (without and with PLY + depth-PNG writing) on the same
                       seeded synthetic 375x1242 PNG pairs (written to a temporary directory), alternated twice
  gpu, power_limit_w   what the numbers were measured on

    python benchmarks/reproject_overhead.py
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
import workloads  # noqa: E402
from confidence_overhead import gpu_name_power, time_ms  # noqa: E402

STEPS = 200
PAIRS = 16
HBM_TBPS = 7.7                    # HGX B200 data sheet, one GPU


def _kernel_us(call):
    """(graph, eager) microseconds per call of `call(stream_handle)`."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call(s.cuda_stream)                                  # module load outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(STEPS):
            call(torch.cuda.current_stream().cuda_stream)
    graph_us = 1e3 * time_ms(graph.replay, 5, warmup=2) / (5 * STEPS)
    eager_us = 1e3 * time_ms(lambda: call(torch.cuda.current_stream().cuda_stream), STEPS, warmup=20) / STEPS
    return round(graph_us, 3), round(eager_us, 3)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("reproject_overhead.py needs a CUDA device")
    H, W, maxdisp, B = workloads.CONFIGS["kitti_384x1248"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    net = workloads.init_bench_weights_(d.GwcNet(maxdisp, precision="parity"), 0).to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(0)
    left = torch.randn(B, 3, H, W, device=dev, generator=g)
    right = torch.roll(left, -8, 3) + 0.1 * torch.randn(B, 3, H, W, device=dev, generator=g)
    with torch.no_grad():
        pred, _, conf, lr = net(left, right, confidence=True, lr_check=True)
    s = np.random.default_rng(0)
    calib = d.StereoCalib(721.5377, 721.5377, 609.5593, 172.854, 0.5327,
                          rect_to_velo=np.hstack([np.eye(3), s.normal(0, 0.1, (3, 1))]))
    n = B * H * W
    tiles = (H * W + 1023) // 1024
    depth = torch.empty(B, H, W, device=dev)
    xyz = torch.empty(B, H * W, 3, device=dev)
    index = torch.empty(B, H * W, dtype=torch.int32, device=dev)
    count = torch.empty(B, dtype=torch.int64, device=dev)
    ws = torch.empty(B, tiles, dtype=torch.int32, device=dev)
    q, t = calib.Q(), np.ascontiguousarray(calib.rect_to_velo)
    variants = {"plain": (0, 0, None, 0.0), "filtered": (conf.peak.data_ptr(), lr.label.data_ptr(), t.ctypes.data, 0.3)}
    reproject_us, kept, bytes_est = {}, {}, {}
    for k, (peak, label, T, mp) in variants.items():
        args = (pred.data_ptr(), peak, label, W, H * W, B, H, W, 0, 0, q.ctypes.data, T, mp, 1e-3, 80.0,
                depth.data_ptr(), xyz.data_ptr(), index.data_ptr(), count.data_ptr(), ws.data_ptr())
        reproject_us[k] = dict(zip(("graph", "eager"), _kernel_us(lambda st, a=args: d._lib.call("dca_reproject", *a,
                                                                                                   st))))
        kept_n = int(count.sum())
        kept[k] = round(kept_n / n, 4)
        maps = 4 + (4 if peak else 0) + (1 if label else 0)          # disp, peak, label: read by both launches
        bytes_est[k] = {"read": 2 * maps * n, "written": 4 * n + 16 * kept_n}
    gt = (torch.rand(B, H, W, generator=torch.Generator().manual_seed(1)) * 100).to(dev)
    rows = torch.zeros(B, d.evaluation.DEPTH_COUNT, dtype=torch.int64, device=dev)
    dm_args = (pred.data_ptr(), gt.data_ptr(), rows.data_ptr(), B, H, W, 192.0, calib.focal_baseline, 0.0, 1e-3, 80.0)
    depth_us = dict(zip(("graph", "eager"), _kernel_us(lambda st: d._lib.call("dca_depth_metrics", *dm_args, st))))
    bytes_est["depth_metrics"] = {"read": 8 * n, "written": 0}

    # files in: ImagePipeline.run against reproject_files on the same PNG pairs
    from PIL import Image
    rng = np.random.default_rng(0)
    runs = {"image_pipeline": [], "reproject_files": [], "reproject_files_ply": []}
    with tempfile.TemporaryDirectory() as tmp:
        pairs = []
        for i in range(PAIRS):
            base = rng.integers(0, 256, (375, 1242 + 16, 3), dtype=np.uint8)
            Image.fromarray(base[:, :1242]).save(os.path.join(tmp, f"l{i}.png"))
            Image.fromarray(base[:, 16:]).save(os.path.join(tmp, f"r{i}.png"))
            pairs.append((os.path.join(tmp, f"l{i}.png"), os.path.join(tmp, f"r{i}.png")))
        pipe = d.kitti_io.ImagePipeline(net, H, W)
        outs = {"image_pipeline": lambda: pipe.run([(l, r, None) for l, r in pairs]),
                "reproject_files": lambda: d.reproject_files(net, [(l, r, None, None) for l, r in pairs], calib,
                                                             min_depth=1e-3, max_depth=80.0),
                "reproject_files_ply": lambda: d.reproject_files(
                    net, [(l, r, os.path.join(tmp, f"p{i}.ply"), os.path.join(tmp, f"d{i}.png"))
                          for i, (l, r) in enumerate(pairs)], calib, min_depth=1e-3, max_depth=80.0)}
        for f in outs.values():                              # warm-up: module loads, pinned buffers
            f()
        for _ in range(2):
            for k, f in outs.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                runs[k].append(round(PAIRS / (time.perf_counter() - t0), 2))
    hbm = {k: round((v["read"] + v["written"]) / (HBM_TBPS * 1e12) * 1e6, 3) for k, v in bytes_est.items()}
    print(json.dumps({
        "workload": f"{H}x{W} maxdisp {maxdisp} B={B}, parity precision, synthetic weights",
        "gpu": name, "power_limit_w": plimit,
        "reproject_us": reproject_us, "depth_metrics_us": depth_us,
        "bytes_est": bytes_est, "hbm_time_us_at_7.7_tbps": hbm, "kept_fraction": kept,
        "files_pairs_per_s": runs, "pairs": PAIRS, "steps": STEPS,
    }), flush=True)


if __name__ == "__main__":
    main()
