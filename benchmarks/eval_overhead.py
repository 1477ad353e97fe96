"""Cost of scoring against ground truth (evaluation.DisparityMeter) at KITTI size, 384x1248, maxdisp 192.

Synthetic weights and feature maps; the ground truth is the model's own prediction plus noise, with the top 30 % of the
rows set to 0 (no GT, as in KITTI).  Prints one JSON line:
  kernel_us          CUDA-event time per launch of dca_disparity_metrics / dca_class_confusion, mean over 200
                     back-to-back launches (their inputs, 3.8 MB + 0.7 MB, stay resident in L2 between launches, as they
                     are right after the forward that wrote them)
  pairs_per_s        hot_path_graphed alone and followed by meter.update, 200 steps each, measured twice in the order
                     A B A B; `overhead_us_per_pair` compares the better run of each
  gpu, power_limit_w what the numbers were measured on

    python benchmarks/eval_overhead.py
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import dcanet_b200 as d  # noqa: E402
import workloads  # noqa: E402

STEPS = 200


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return float(out.stdout.strip().splitlines()[0])
    except Exception:
        return None


def time_ms(fn, n, warmup=20):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("eval_overhead.py needs a CUDA device")
    ev = d.evaluation
    H, W, maxdisp, B = workloads.CONFIGS["kitti_384x1248"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    plimit = power_limit_w()
    net = workloads.init_bench_weights_(d.GwcNet(maxdisp), 0).to(dev).eval()
    feats = [t.to(dev) for t in workloads.feature_maps(0, B, H // 4, W // 4)]
    with torch.no_grad():
        pred4, pv = net.hot_path_graphed(*feats)
        g = torch.Generator(device=dev).manual_seed(0)
        gt = (pred4[:, 0] + 2.0 * torch.randn(pred4[:, 0].shape, generator=g, device=dev)).clamp_(min=0.0)
        gt[:, : (3 * H) // 10] = 0.0
    D8, H8, W8 = pv.shape[1:]

    rows = torch.zeros((B, ev.METRIC_COUNT), dtype=torch.int64, device=dev)
    conf = torch.zeros((D8, D8), dtype=torch.int64, device=dev)
    pred = pred4[:, 0]
    kernel_us = {
        "dca_disparity_metrics": 1e3 * time_ms(lambda: ev._disparity_metrics(pred, gt, rows, float(maxdisp)), STEPS) / STEPS,
        "dca_class_confusion": 1e3 * time_ms(lambda: ev._class_confusion(pv, gt, conf, float(maxdisp)), STEPS) / STEPS,
    }
    bytes_read = {"dca_disparity_metrics": 2 * B * H * W * 4, "dca_class_confusion": B * (D8 + 1) * H8 * W8 * 4}
    gbps = {k: bytes_read[k] / (kernel_us[k] * 1e-6) / 1e9 for k in kernel_us}

    def forward_only():
        net.hot_path_graphed(*feats)

    meter = ev.DisparityMeter(maxdisp, device=dev, capacity=4 * STEPS)

    def forward_and_update():
        p, v = net.hot_path_graphed(*feats)
        meter.update(p, gt, v)

    runs = {"forward": [], "forward+update": []}
    with torch.no_grad():
        for _ in range(2):
            runs["forward"].append(STEPS / (time_ms(forward_only, STEPS, warmup=10) * 1e-3))
            runs["forward+update"].append(STEPS / (time_ms(forward_and_update, STEPS, warmup=10) * 1e-3))
    best = {k: max(v) for k, v in runs.items()}
    s = meter.summary()
    print(json.dumps({
        "workload": f"{H}x{W} maxdisp {maxdisp} B={B}, synthetic weights / features / GT",
        "gpu": torch.cuda.get_device_name(dev), "power_limit_w": plimit,
        "kernel_us": {k: round(v, 2) for k, v in kernel_us.items()},
        "kernel_bytes": bytes_read, "kernel_gb_per_s": {k: round(v, 1) for k, v in gbps.items()},
        "pairs_per_s": {k: [round(x, 1) for x in v] for k, v in runs.items()},
        "overhead_us_per_pair": round(1e6 / best["forward+update"] - 1e6 / best["forward"], 1),
        "steps": STEPS, "meter_rows": len(meter),
        "meter_epe_px": round(s["epe"], 4), "meter_bad3": round(s["bad3"], 4), "meter_miou": round(s["miou"], 4),
    }), flush=True)


if __name__ == "__main__":
    main()
