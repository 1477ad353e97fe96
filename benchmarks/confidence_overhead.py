"""Cost of the per-pixel confidence maps (hot_path(..., confidence=True)) at KITTI size, 384x1248, maxdisp 192, parity
precision, synthetic weights and seeded feature maps on the device.

Prints one JSON line:
  pair_ms              hot_path_graphed with and without confidence, STEPS steps each after a warm-up, alternated
                       A B A B in this process (CUDA events); `delta_pct` compares the better run of each
  kernel_us            CUDA-event time per launch of dca_softmax_confidence_upsample alone, and of one
                       DisparityMeter.update with a confidence map (its three kernels), mean over STEPS back-to-back
                       launches (inputs resident in L2, as right after the forward that wrote them)
  bytes_est            bytes the confidence adds per pair, from the shapes (logits write + read with the ring, mask, outputs)
  gpu, power_limit_w   what the numbers were measured on

    python benchmarks/confidence_overhead.py
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


def gpu_name_power(dev):
    """(name, power limit in W) of the card behind `dev`, asked of nvidia-smi by the device's UUID (torch's ordinal is
    not nvidia-smi's index under CUDA_VISIBLE_DEVICES); the power limit is None when nvidia-smi cannot say."""
    uuid = str(torch.cuda.get_device_properties(dev).uuid)
    uuid = uuid if uuid.startswith(("GPU-", "MIG-")) else "GPU-" + uuid
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=uuid,name,power.limit", "--format=csv,noheader,nounits",
                              "-i", uuid], capture_output=True, text=True, timeout=30)
        got, name, limit = [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")]
        if got != uuid:
            raise ValueError(f"nvidia-smi answered for {got}, asked for {uuid}")
        return name, float(limit)
    except Exception:
        return torch.cuda.get_device_name(dev), None


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
        raise SystemExit("confidence_overhead.py needs a CUDA device")
    E, ev = d.engine, d.evaluation
    H, W, maxdisp, B = workloads.CONFIGS["kitti_384x1248"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    net = workloads.init_bench_weights_(d.GwcNet(maxdisp, precision="parity"), 0).to(dev).eval()
    feats = [t.to(dev) for t in workloads.feature_maps(0, B, H // 4, W // 4)]
    keep = {}
    with torch.no_grad():
        pred4, pv, conf = net.hot_path(*feats, keep=keep, confidence=True)
        g = torch.Generator(device=dev).manual_seed(0)
        gt = (pred4[:, 0] + 2.0 * torch.randn(pred4[:, 0].shape, generator=g, device=dev)).clamp_(min=0.0)
        gt[:, : (3 * H) // 10] = 0.0
    logits, mask = keep["classif3_logits"], keep["mask"]
    D4, H4, W4 = logits.shape[1:]

    runs = {"plain": [], "confidence": []}
    with torch.no_grad():
        fns = {"plain": lambda: net.hot_path_graphed(*feats),
               "confidence": lambda: net.hot_path_graphed(*feats, confidence=True)}
        for _ in range(2):
            for k in ("plain", "confidence"):
                runs[k].append(time_ms(fns[k], STEPS, warmup=10) / STEPS)
        meter = ev.DisparityMeter(maxdisp, device=dev, capacity=4 * STEPS)
        peak = conf.peak
        kernel_us = {
            "dca_softmax_confidence_upsample": 1e3 * time_ms(lambda: E.softmax_confidence_upsample(logits, mask),
                                                             STEPS) / STEPS,
            "meter_update_with_confidence": 1e3 * time_ms(lambda: meter.update(pred4, gt, pv, peak), STEPS) / STEPS,
        }
    best = {k: min(v) for k, v in runs.items()}
    n4 = B * H4 * W4
    bytes_est = {"logits_write": 4 * n4 * D4, "logits_read_with_ring": 4 * n4 * D4 * 340 // 256,   # (8+2) x (32+2) / 256
                 "mask": 4 * 144 * n4, "outputs": 2 * 4 * 16 * n4}
    s = meter.summary()
    print(json.dumps({
        "workload": f"{H}x{W} maxdisp {maxdisp} B={B}, parity precision, synthetic weights / features / GT",
        "gpu": name, "power_limit_w": plimit,
        "pair_ms": {k: [round(x, 4) for x in v] for k, v in runs.items()},
        "delta_us_per_pair": round(1e3 * (best["confidence"] - best["plain"]), 2),
        "delta_pct": round(100.0 * (best["confidence"] / best["plain"] - 1.0), 3),
        "kernel_us": {k: round(v, 2) for k, v in kernel_us.items()},
        "bytes_est": bytes_est, "bytes_est_total_mb": round(sum(bytes_est.values()) / 1e6, 2),
        "steps": STEPS, "meter_epe_px": round(s["epe"], 4), "meter_ause_px": round(s["ause_epe"], 4),
    }), flush=True)


if __name__ == "__main__":
    main()
