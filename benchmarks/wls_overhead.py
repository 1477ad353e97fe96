"""Cost of the edge-aware refinement (dca_wls_filter: prepare, then a row pass and a column pass per iteration).

Prints one JSON line:
  call_us          one wls_filter call per case, with peak and label: `graph` = CUDA-event time of STEPS calls captured in
                   one CUDA graph, `eager` = CUDA-event time of STEPS calls launched one by one, after a warm-up; per call
                   and per image.  Cases:
                     kitti_b1_t1, kitti_b1_t3     the KITTI window 375x1242, B = 1, T = 1 and 3 (working set ~8 MB:
                                                  it stays in the 126 MB L2 between calls and passes)
                     kitti_b16_t1, kitti_b16_t3   the same at B = 16 (~130 MB: about the size of the L2)
                     middlebury_t3                a 1988x2880 window, B = 1, T = 3 (~100 MB)
  kernel_us        the same cases under torch.profiler (a separate run of PROFILE_CALLS eager calls): mean device time
                   per call of the prepare kernel, and of one row pass and one column pass, each split into its
                   boundary-value (wls_seg_kernel), separator (wls_reduce_kernel) and segment-solve (wls_solve_kernel)
                   launches
  bytes_est        bytes per call from the shapes: prepare reads disp, peak, label and the guide and writes U, V and two
                   weight maps (28 B / px with an RGB guide); a pass reads U, V and the weights twice (boundary values,
                   then the segment solve) and writes U, V (32 B / px; the separator system and the 8 boundary values
                   per segment are left out; the last column pass also reads disp); and the time that takes at 7.7 TB/s
  gpu, power_limit_w   what the numbers were measured on

    python benchmarks/wls_overhead.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dcanet_b200 as d  # noqa: E402
from confidence_overhead import gpu_name_power, time_ms  # noqa: E402

STEPS = 200
PROFILE_CALLS = 20
HBM_TBPS = 7.7                    # HGX B200 data sheet, one GPU
CASES = {"kitti_b1_t1": (1, 375, 1242, 1), "kitti_b1_t3": (1, 375, 1242, 3), "kitti_b16_t1": (16, 375, 1242, 1),
         "kitti_b16_t3": (16, 375, 1242, 3), "middlebury_t3": (1, 1988, 2880, 3)}
PHASES = ("wls_seg_kernel", "wls_reduce_kernel", "wls_solve_kernel")     # per pass; <true> = rows, <false> = columns


def _inputs(B, H, W, dev, rng):
    """A blocky colour image with matching piecewise-constant disparities, noise, and 70 % confident pixels."""
    blocks = rng.integers(0, 256, (B, H // 25 + 1, W // 40 + 1, 3), dtype=np.uint8)
    guide = np.repeat(np.repeat(blocks, 25, 1), 40, 2)[:, :H, :W]
    disp = guide[..., 0].astype(np.float32) / 4 + rng.normal(0, 0.5, (B, H, W)).astype(np.float32)
    peak = np.where(rng.random((B, H, W)) < 0.7, rng.uniform(0.3, 1.0, (B, H, W)), 0.0).astype(np.float32)
    label = np.where(rng.random((B, H, W)) < 0.9, 0, 1).astype(np.uint8)
    return [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (disp, guide, peak, label)]


def _call_us(call):
    """(graph, eager) microseconds per call of `call()`."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()                                               # module load and weight table outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(STEPS):
            call()
    graph_us = 1e3 * time_ms(graph.replay, 5, warmup=2) / (5 * STEPS)
    eager_us = 1e3 * time_ms(call, STEPS, warmup=20) / STEPS
    return round(graph_us, 3), round(eager_us, 3)


def _kernel_us(call, T):
    """Mean device microseconds from torch.profiler: the prepare kernel per call, and per pass (rows, columns) the
    boundary-value, separator and segment-solve kernels and their sum."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(PROFILE_CALLS):
            call()
        torch.cuda.synchronize()
    tot = {"prepare": 0.0}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA or "wls_" not in e.name:
            continue
        if "wls_prepare_kernel" in e.name:
            tot["prepare"] += e.device_time
            continue
        kind = "row" if "<true>" in e.name else "col"
        phase = next(p for p in PHASES if p in e.name)
        tot[f"{kind}:{phase}"] = tot.get(f"{kind}:{phase}", 0.0) + e.device_time
    out = {"prepare": round(tot.pop("prepare") / PROFILE_CALLS, 3)}
    for kind in ("row", "col"):
        parts = {p: round(tot.get(f"{kind}:{p}", 0.0) / (PROFILE_CALLS * T), 3) for p in PHASES}
        out[f"{kind}_pass"] = round(sum(parts.values()), 3)
        out[f"{kind}_pass_parts"] = parts
    return out


def main():
    if not torch.cuda.is_available():
        raise SystemExit("wls_overhead.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    rng = np.random.default_rng(0)
    call_us, kernel_us, bytes_est, hbm = {}, {}, {}, {}
    for k, (B, H, W, T) in CASES.items():
        disp, guide, peak, label = _inputs(B, H, W, dev, rng)
        call = lambda: d.wls_filter(disp, guide, confidence=peak, label=label, num_iter=T)
        g, e = _call_us(call)
        call_us[k] = {"graph": g, "eager": e, "graph_per_image": round(g / B, 3), "eager_per_image": round(e / B, 3)}
        kernel_us[k] = _kernel_us(call, T)
        px = B * H * W
        b = {"prepare": 28 * px, "passes": T * 2 * 32 * px + 4 * px}
        b["total"] = sum(b.values())
        bytes_est[k] = b
        hbm[k] = round(b["total"] / (HBM_TBPS * 1e12) * 1e6, 3)
        del disp, guide, peak, label
    print(json.dumps({
        "workload": "wls_filter with peak and label, lam 8000, sigma 1.5, min_support 1e-3, RGB guide; KITTI window "
                    "375x1242 at B = 1 / 16 and T = 1 / 3, a 1988x2880 window at B = 1, T = 3",
        "gpu": name, "power_limit_w": plimit,
        "call_us": call_us, "kernel_us": kernel_us, "bytes_est": bytes_est, "hbm_time_us_at_7.7_tbps": hbm,
        "steps": STEPS, "profile_calls": PROFILE_CALLS,
    }), flush=True)


if __name__ == "__main__":
    main()
