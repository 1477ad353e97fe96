"""Cost of the left-right consistency check (GwcNet(left, right, lr_check=True)) at KITTI size, 384x1248, maxdisp 192,
parity precision, synthetic weights and seeded images on the device.

Prints one JSON line:
  pair_ms              model(l, r) and model(l, r, lr_check=True) from images, STEPS steps each after a warm-up,
                       alternated A B A B in this process (CUDA events); `ratio` compares the better run of each
  kernel_us            dca_lr_consistency alone (mirrored right view, right output written): `graph` = CUDA-event time
                       of STEPS launches captured in one CUDA graph, per launch; `profiler` = mean device time of the
                       kernel in torch.profiler over STEPS launches (a run of its own, after the timings)
  bytes_est            bytes the kernel moves per pair, from the shapes, and the time that takes at 7.7 TB/s
  left_outputs_identical   pred / prob_volume of the two forwards are bit-identical
  label_fraction       share of each label (consistent, occluded, mismatch, out of view); synthetic weights, so this
                       says nothing about accuracy
  gpu, power_limit_w   what the numbers were measured on

    python benchmarks/lr_check_overhead.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

import dcanet_b200 as d  # noqa: E402
import workloads  # noqa: E402
from confidence_overhead import gpu_name_power, time_ms  # noqa: E402

STEPS = 200
HBM_TBPS = 7.7                    # HGX B200 data sheet, one GPU


def main():
    if not torch.cuda.is_available():
        raise SystemExit("lr_check_overhead.py needs a CUDA device")
    E = d.engine
    H, W, maxdisp, B = workloads.CONFIGS["kitti_384x1248"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    net = workloads.init_bench_weights_(d.GwcNet(maxdisp, precision="parity"), 0).to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(0)
    imgs = [(torch.randn(B, 3, H, W, device=dev, generator=g), torch.randn(B, 3, H, W, device=dev, generator=g))
            for _ in range(2)]
    step = {"plain": 0, "lr_check": 0}

    def fwd(k):
        l, r = imgs[step[k] % 2]
        step[k] += 1
        return net(l, r, lr_check=(k == "lr_check"))

    runs = {"plain": [], "lr_check": []}
    with torch.no_grad():
        for _ in range(2):
            for k in ("plain", "lr_check"):
                runs[k].append(time_ms(lambda: fwd(k), STEPS, warmup=10) / STEPS)
        pred, pv = net(*imgs[0])
        pred2, pv2, lr = net(*imgs[0], lr_check=True)
        identical = bool(torch.equal(pred, pred2) and torch.equal(pv, pv2))
        frac = (torch.bincount(lr.label.flatten().long(), minlength=4).double() / lr.label.numel()).tolist()

        # the kernel alone, on the two halves of a 2-pair pred4 as the forward launches it
        both = torch.cat((pred, lr.disp_right.flip(-1)), 0).contiguous()
        dl, dr = both[:B], both[B:]
        label = torch.empty(dl.shape, dtype=torch.uint8, device=dev)
        filled, right = torch.empty_like(dl), torch.empty_like(dl)
        args = (dl.data_ptr(), dr.data_ptr(), 1, label.data_ptr(), filled.data_ptr(), right.data_ptr(), B, H, W, 1.0)
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            d._lib.call("dca_lr_consistency", *args, s.cuda_stream)          # module load outside the capture
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(STEPS):
                d._lib.call("dca_lr_consistency", *args, torch.cuda.current_stream().cuda_stream)
        graph_us = 1e3 * time_ms(graph.replay, 5, warmup=2) / (5 * STEPS)
        assert torch.equal(label, lr.label) and torch.equal(filled, lr.filled) and torch.equal(right, lr.disp_right)

        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(STEPS):
                E.lr_consistency(dl, dr, 1.0, mirrored=True, want_right=True)
            torch.cuda.synchronize()
        ev = [e for e in prof.key_averages() if "lr_consistency_kernel" in e.key]
        prof_us = None
        if ev:
            tot = getattr(ev[0], "device_time_total", None)
            tot = getattr(ev[0], "cuda_time_total", 0.0) if tot is None else tot
            prof_us = tot / ev[0].count
    best = {k: min(v) for k, v in runs.items()}
    n = B * H * W
    bytes_est = {"read": 2 * 4 * n, "written": (1 + 4 + 4) * n}
    tot = sum(bytes_est.values())
    print(json.dumps({
        "workload": f"{H}x{W} maxdisp {maxdisp} B={B}, parity precision, synthetic weights, seeded images on the device",
        "gpu": name, "power_limit_w": plimit,
        "pair_ms": {k: [round(x, 4) for x in v] for k, v in runs.items()},
        "delta_ms_per_pair": round(best["lr_check"] - best["plain"], 4),
        "ratio": round(best["lr_check"] / best["plain"], 4),
        "kernel_us": {"graph": round(graph_us, 3), "profiler": None if prof_us is None else round(prof_us, 3)},
        "bytes_est": bytes_est, "bytes_est_total_mb": round(tot / 1e6, 2),
        "hbm_time_us_at_7.7_tbps": round(tot / (HBM_TBPS * 1e12) * 1e6, 2),
        "left_outputs_identical": identical, "label_fraction": [round(x, 4) for x in frac], "steps": STEPS,
    }), flush=True)


if __name__ == "__main__":
    main()
