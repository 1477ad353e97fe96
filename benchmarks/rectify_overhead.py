"""Cost of rectifying raw stereo pairs on the device (dca_rectify + dca_standardise_frame) and what it does to the
files-in throughput, synthetic weights.

Prints one JSON line:
  kernel_us            one rectify call per case (the moments zero-fill, dca_rectify and dca_standardise_frame), per
                       call and per pair: `graph` = CUDA-event time of STEPS calls captured in one CUDA graph, `eager` =
                       CUDA-event time of STEPS calls launched one by one, after a warm-up.  Cases:
                         kitti_b1    KITTI raw 1392x512 RGB -> 1242x375 -> fit 384x1248, B = 1 (the pipeline's case; its
                                     ~26 MB working set stays in the 126 MB L2 between calls)
                         kitti_b16   the same at B = 16 (~300 MB: beyond the L2)
                         middlebury  2880x1988 RGB -> 2880x1988 -> pad16, B = 1
  bytes_est            compulsory bytes per call from the shapes: raw pair read once, maps read once per pair, the
                       uint8 rectified pair written and read back, the fp32 network input written; and the time that
                       takes at 7.7 TB/s
  files_pairs_per_s    rectify_files on raw 1392x512 PNGs against ImagePipeline.run on the pre-rectified 1242x375 PNGs
                       of the same pairs (same model, PAIRS pairs, written to a temporary directory), alternated twice
  gpu, power_limit_w   what the numbers were measured on

    python benchmarks/rectify_overhead.py
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


def _rot(ax, ay):
    cx, sx, cy, sy = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay)
    return np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])


def rig(raw, rect_size, f_raw, f_rect, baseline):
    """A distorted rig of KITTI raw's magnitudes scaled to the sizes."""
    K = np.array([[f_raw, 0.0, raw[0] / 2 + 0.3], [0.0, f_raw * 0.997, raw[1] / 2 - 31.0], [0.0, 0.0, 1.0]])
    Kr = np.array([[f_rect, 0.0, rect_size[0] / 2 - 11.5], [0.0, f_rect, rect_size[1] / 2 - 14.6], [0.0, 0.0, 1.0]])
    D = [-0.37, 0.20, 0.001, -0.001, -0.07]
    P1 = Kr @ np.hstack([np.eye(3), np.zeros((3, 1))])
    P2 = Kr @ np.hstack([np.eye(3), [[-baseline], [0.0], [0.0]]])
    return d.StereoRectifier(K, D, _rot(0.004, -0.009), P1, K, D, _rot(-0.003, 0.006), P2, raw, rect_size)


def _kernel_us(call):
    """(graph, eager) microseconds per call of `call()`."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()                                               # module load outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(STEPS):
            call()
    graph_us = 1e3 * time_ms(graph.replay, 5, warmup=2) / (5 * STEPS)
    eager_us = 1e3 * time_ms(call, STEPS, warmup=20) / STEPS
    return round(graph_us, 3), round(eager_us, 3)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("rectify_overhead.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    kitti = rig((1392, 512), (1242, 375), 959.8, 721.5, 0.5327)
    middlebury = rig((2880, 1988), (2880, 1988), 3979.9, 3979.9, 0.193)
    rng = np.random.default_rng(0)
    cases = {"kitti_b1": (kitti, 1, "fit"), "kitti_b16": (kitti, 16, "fit"), "middlebury": (middlebury, 1, "pad16")}
    kernel_us, bytes_est, hbm = {}, {}, {}
    for k, (r, B, mode) in cases.items():
        Ws, Hs = r.raw_size
        W, H = r.rect_size
        left = torch.from_numpy(rng.integers(0, 256, (B, Hs, Ws, 3), dtype=np.uint8)).to(dev)
        right = torch.from_numpy(rng.integers(0, 256, (B, Hs, Ws, 3), dtype=np.uint8)).to(dev)
        x = d.rectify(left, right, r, mode)                 # uploads the maps
        Hn, Wn = x.left.shape[2:]
        g, e = _kernel_us(lambda: d.rectify(left, right, r, mode))
        kernel_us[k] = {"graph": g, "eager": e, "graph_per_pair": round(g / B, 3), "eager_per_pair": round(e / B, 3)}
        b = {"raw_read": 2 * B * Hs * Ws * 3, "maps_read": B * 2 * H * W * 8, "rgb_written": 2 * B * H * W * 3,
             "rgb_read": 2 * B * H * W * 3, "input_written": 2 * B * 3 * Hn * Wn * 4}
        b["total"] = sum(b.values())
        bytes_est[k] = b
        hbm[k] = round(b["total"] / (HBM_TBPS * 1e12) * 1e6, 3)
    # files in: rectify_files on raw PNGs against ImagePipeline on the pre-rectified PNGs of the same pairs
    from PIL import Image
    H, W, maxdisp, _ = workloads.CONFIGS["kitti_384x1248"]
    net = workloads.init_bench_weights_(d.GwcNet(maxdisp, precision="parity"), 0).to(dev).eval()
    runs = {"image_pipeline_rectified_png": [], "rectify_files_raw_png": []}
    with tempfile.TemporaryDirectory() as tmp:
        raw_items, rect_items = [], []
        for i in range(PAIRS):
            base = rng.integers(0, 256, (512, 1392 + 16, 3), dtype=np.uint8)
            names = [os.path.join(tmp, f"{s}{i}.png") for s in ("rl", "rr", "l", "r")]
            Image.fromarray(base[:, :1392]).save(names[0])
            Image.fromarray(base[:, 16:]).save(names[1])
            x = d.rectify(torch.from_numpy(base[None, :, :1392].copy()).to(dev),
                          torch.from_numpy(base[None, :, 16:].copy()).to(dev), kitti)
            Image.fromarray(x.rgb[0, 0].cpu().numpy()).save(names[2])
            Image.fromarray(x.rgb[0, 1].cpu().numpy()).save(names[3])
            raw_items.append((names[0], names[1], None))
            rect_items.append((names[2], names[3], None))
        pipe = d.kitti_io.ImagePipeline(net, H, W)
        outs = {"image_pipeline_rectified_png": lambda: pipe.run(rect_items),
                "rectify_files_raw_png": lambda: d.rectify_files(net, raw_items, kitti, H, W)}
        for f in outs.values():                              # warm-up: module loads, pinned buffers
            f()
        for _ in range(2):
            for k, f in outs.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                runs[k].append(round(PAIRS / (time.perf_counter() - t0), 2))
    print(json.dumps({
        "workload": "KITTI raw 1392x512 -> 1242x375 -> fit 384x1248 (B=1, B=16); 2880x1988 -> pad16 (B=1); files: "
                    f"{H}x{W} maxdisp {maxdisp} parity precision, synthetic weights",
        "gpu": name, "power_limit_w": plimit,
        "kernel_us": kernel_us, "bytes_est": bytes_est, "hbm_time_us_at_7.7_tbps": hbm,
        "files_pairs_per_s": runs, "pairs": PAIRS, "steps": STEPS,
    }), flush=True)


if __name__ == "__main__":
    main()
