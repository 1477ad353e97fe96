#!/usr/bin/env python
"""Benchmark of the DCANet cost-volume hot path (feature maps -> disparity) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config kitti_384x1248]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE stereo pair through the whole hot path at BASELINE.json's configs[1]
(KITTI 384x1248, maxdisp 192, batch 1).  Pairs shard by rank with no collective (weak scaling).
Prints ONE JSON line on rank 0.  The inputs and weights are seeded, so the same arguments give the same inputs on every
run; --dump-outputs writes what rank 0's last timed step returned, to compare two builds output for output.
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import workloads  # noqa: E402

METRIC = "KITTI 384x1248 pairs/s"
UNIT = "pairs/s"


def ncu_traffic(kernel_key):
    """DRAM bytes per launch (read+write) of a kernel from the committed `ncu --set full` capture, or None."""
    best = None
    for fn in sorted(os.listdir(os.path.join(ROOT, "profiles"))):
        if fn.endswith("_ncu_traffic.json"):
            z = json.load(open(os.path.join(ROOT, "profiles", fn)))
            for k, v in z.items():
                if kernel_key in k and v:
                    best = {"bytes": v[0]["dram_read_bytes"] + v[0]["dram_write_bytes"], "source": f"profiles/{fn}",
                            "tensor_pipe_pct": v[0].get("tensor_pipe_pct"), "dram_pct": v[0].get("dram_pct")}
    return best


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        z = json.load(open(p))
        return z["hbm_gbs"], z["bf16_tflops"], z.get("bf16_tflops_sustained", z["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region, through NVML in this process (the library behind
    nvidia-smi; `nvidia_ml_py`).  Spawning `nvidia-smi` itself is NOT harmless: its start-up takes driver locks and was
    measured to stall the launch stream for 50-250 ms about once in five runs (value 66-260 pairs/s at an unchanged
    p50 of 3.27 ms), so the process-spawning form is only the fallback when NVML cannot be imported."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.stop_flag = gpu_index, [], False
        self.nvml, self.handle, self.max_mhz = None, None, None
        self.interval = float(os.environ.get("DCA_BENCH_CLOCK_INTERVAL", "0.05"))
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        self.samples.append((mhz, self.max_mhz, {name for bit, name in self.REASONS if mask & bit}))

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                             capture_output=True, text=True, timeout=5).stdout
        for line in out.strip().splitlines():
            c = [v.strip() for v in line.split(",")]
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            self.samples.append((float(c[0]), float(c[1]), {n for n, v in zip(names, c[2:6]) if v.lower().startswith("active")}))

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            time.sleep(self.interval if self.nvml is not None else max(0.25, self.interval))

    def stop(self):
        self.stop_flag = True

    def summary(self):
        sm = [s[0] for s in self.samples]
        mx = [s[1] for s in self.samples if s[1]]
        reasons = set()
        for s in self.samples:
            reasons |= s[2]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def common_config(cfg, n_gpus, batch=0, sub_batch=4):
    """The workload description shared, key for key, by both arms (the driver compares the dicts)."""
    H, W, maxdisp, B = workloads.CONFIGS[cfg]
    if batch:
        z = common_config(cfg, n_gpus)
        z["batch_per_gpu"] = batch // n_gpus
        z["batch_total"] = batch
        z["parallelism"] = (f"{batch} pairs per step, {batch // n_gpus} per GPU over {n_gpus} GPU(s) in forwards of up to "
                            f"{sub_batch} pairs, no collective")
        return z
    return {"workload": cfg, "H": H, "W": W, "maxdisp": maxdisp, "batch_per_gpu": B, "groups": 40,
            "precision": "parity (|d disp| <= 0.05 px of the fp32 torch forward)",
            "parallelism": f"pairs sharded over {n_gpus} GPU(s), no collective",
            "l2": "inputs rotate over 4 feature sets (320 MB) and every step streams >3 GB of activations, both > 126 MB L2",
            "path": "feature maps -> disparity (volume, dres0/1, 3x cva, classif3, regression, convex upsample)",
            "algorithmic_gflop_per_pair": workloads.hot_path_flops(H, W, maxdisp) / 1e9}


def cpu_arm(cfg, steps, warmup, budget_s):
    """CPU arm: the reference's own torch forward from baseline/_ref when it is staged (kind "reference"), else the
    oracle port (kind "port").  Returns (pairs/s, ms/pair, cores, kind, sample)."""
    from baseline import reference_arm
    if reference_arm.available() and os.environ.get("DCA_BENCH_CPU_ARM", "reference") != "port":
        import dcanet_b200 as d
        H, W, maxdisp, B = workloads.CONFIGS[cfg]
        net = workloads.init_bench_weights_(d.GwcNet(maxdisp), 0)       # state_dict layout == the reference's
        v, ms, cores, sample, _ = reference_arm.run(H, W, maxdisp, B, steps, warmup, net.state_dict(), budget_s)
        return v, ms, cores, "reference", sample
    v, ms, cores, sample = cpu_reference_run(cfg, steps, warmup, budget_s)
    return v, ms, cores, "port", sample


def cpu_reference_run(cfg, steps, warmup, budget_s=150.0):
    """The reference's CPU implementation of the path = the oracle port (torch fp32 on all host cores),
    timed on a bounded sample of the workload: an H-crop of the KITTI pair, scaled by the row fraction."""
    from oracle import dcanet_oracle as O      # checker used as the timed CPU arm ONLY here
    import dcanet_b200 as d
    H, W, maxdisp, B = workloads.CONFIGS[cfg]
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    net = workloads.init_bench_weights_(d.GwcNet(maxdisp), 0)
    sd = {k: v for k, v in net.state_dict().items() if not k.startswith(("feature_extraction.", "guidance."))}
    rows4 = H // 4
    frac_rows = rows4
    # pick the crop so that (warmup + steps) steps fit the budget: probe with 1/8 of the rows first
    probe_rows = max(8, (rows4 // 8) // 8 * 8)
    feats = workloads.feature_maps(0, B, probe_rows, W // 4)
    t0 = time.perf_counter()
    with torch.no_grad():
        O.hot_path(sd, *feats, maxdisp=maxdisp)
    t_probe = time.perf_counter() - t0
    per_row = t_probe / probe_rows
    n_total = max(1, steps + warmup)
    frac_rows = int(min(rows4, max(8, (budget_s / n_total / per_row) // 8 * 8)))
    feats = workloads.feature_maps(0, B, frac_rows, W // 4)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.hot_path(sd, *feats, maxdisp=maxdisp)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    scale = rows4 / frac_rows
    t_pair = statistics.mean(times) * scale
    sample = (f"{frac_rows * 4}x{W} crop ({frac_rows}/{rows4} of the 1/4-res rows, full W and maxdisp) of the "
              f"{H}x{W} pair, time scaled by {scale:.2f}; {warmup} warm-up + {steps} timed; torch {torch.__version__} fp32")
    return 1.0 / t_pair, t_pair * 1e3, cores, sample


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """Writes every array as out_dir/<name>.npy in float32.  When they exceed `limit` bytes in all, each one is replaced by
    a fixed sample of its flattened elements (sorted indices drawn by numpy's default_rng(0)), sized in proportion, so that
    two runs with the same arguments still compare element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {name: a.numpy().astype(np.float32, copy=False) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > limit:
            idx = np.sort(np.random.default_rng(0).choice(a.size, a.size * limit // total, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def halo_plan_bytes(H, W, maxdisp, B, planes=2):
    """Bytes ONE rank sends to ONE neighbour per forward in the H-sharded mode (the plan of hshard.hot_path_steps: only
    the one live row next to a cut travels).  1/4-res 32-ch plane rows: dres0.0/2, dres1.0/2, 3 x (fused, out), classif3.0
    = 11; 1/8-res rows: 3 x (pooled, cost_down, h: 32 ch; c1, c2: 64 ch; logits fp32); feature maps (fp32, 332 + 332 +
    ... channels), prop m1 (128 ch) and the regressed disparity."""
    D4, W4, D8, W8 = maxdisp // 4, W // 4, maxdisp // 8, W // 8
    row4 = planes * B * D4 * W4 * 32 * 2
    row8 = planes * B * D8 * W8 * 32 * 2
    total = 11 * row4 + 3 * (3 * row8 + 2 * 2 * row8 + B * D8 * W8 * 4)
    total += B * W4 * 4 * (320 + 320 + 12 + 12 + 64)          # fp32 feature-map rows
    total += planes * B * W4 * 128 * 2 + B * W4 * 4          # prop m1 row, regressed disparity row
    return total


def measure_hshard(cfg, transport, d, net, dist, dev, rank, world, barrier, K, Wm):
    """Single-pair H-sharded mode (BASELINE configs[4], SURVEY 8e): every step is ONE pair whose 1/4-res rows are split
    over the ranks; the data path has a real exchange (halo rows with both neighbours after every k3 layer, one
    [B, D/8] all-reduce per cva), so this is strong scaling.  Returns the record (valid on every rank)."""
    H, W, maxdisp, B = workloads.CONFIGS[cfg]
    hs = d.hshard
    nsets = 2
    slabs = []
    for s in range(nsets):       # every rank builds the same seeded pair and keeps only the rows it owns
        full = workloads.feature_maps(s, B, H // 4, W // 4)
        slabs.append([hs.owned_rows(t, world, rank).to(dev) for t in full])
        del full
    with torch.no_grad():
        for i in range(Wm):
            net.hot_path_hsharded(*slabs[i % nsets], rank=rank, world=world, transport=transport)
        d._lib.LAUNCHES = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_host0 = time.perf_counter()
        e0.record()
        for i in range(K):
            net.hot_path_hsharded(*slabs[i % nsets], rank=rank, world=world, transport=transport)
        e1.record()
        t_issue = time.perf_counter() - t_host0          # host time to ISSUE the K forwards (no sync inside)
        barrier()
        t1 = time.perf_counter()                         # one forward issued into an IDLE device: the host-side cost alone
        net.hot_path_hsharded(*slabs[0], rank=rank, world=world, transport=transport)
        t_single = time.perf_counter() - t1
        barrier()
    for peer in hs._PEERS.values():      # p2p transport: a timed-out wait (neighbour never pushed) invalidates the run
        peer.check()
    launches = d._lib.LAUNCHES
    tt = torch.tensor([e0.elapsed_time(e1), t_issue * 1e3], dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms = float(tt[0])
    r0, r1 = hs.row_partition(H // 4, world)[0]
    halo = halo_plan_bytes(H, W, maxdisp, B)
    del slabs
    torch.cuda.empty_cache()
    return {"workload": cfg, "H": H, "W": W, "maxdisp": maxdisp, "batch": B, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_pair": ms / K / B, "pairs_per_s": K * B / (ms * 1e-3), "transport": transport,
            "host_issue_ms_per_pair": float(tt[1]) / K / B, "host_issue_ms_idle_device": t_single * 1e3,
            "rows_per_rank": r1 - r0, "halo_rows_per_side": 2,
            "halo_bytes_per_neighbour_per_step": halo,
            "exchanges_per_step": 36, "allreduces_per_step": 3,
            "nvlink_roofline_ms": halo / 770e9 * 1e3,
            "gpu_launches": launches,
            "algorithmic_gflop_per_pair": workloads.hot_path_flops(H, W, maxdisp) / 1e9}


def run_hshard(args, d, net, dist, dev, rank, world, barrier, K, Wm):
    """`--hshard`: the H-sharded mode as the whole run (strong scaling).  Not part of the default run; the default run at
    N > 1 appends the same measurement as the `hshard` sub-record."""
    assert dist is not None and world > 1, "--hshard needs torchrun with more than one rank"
    rec = measure_hshard(args.config, args.hshard_transport, d, net, dist, dev, rank, world, barrier, K, Wm)
    if rank == 0:
        print(json.dumps({
            "metric": f"{args.config} pairs/s (one pair H-sharded over {world} GPUs)", "value": rec["pairs_per_s"],
            "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": rec["ms_per_pair"],
            "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16x2 split operands, fp32 accumulate",
            "data": "synthetic",
            "config": {"workload": args.config, "H": rec["H"], "W": rec["W"], "maxdisp": rec["maxdisp"], "batch": rec["batch"],
                       "parallelism": f"rows of one pair over {world} ranks: {rec['rows_per_rank']} quarter-res rows + 2 halo rows "
                                      "per side each; halo rows by " + args.hshard_transport + ", 3 all-reduces of [B, D/8]"},
            "hshard": rec, "gpu_launches": rec["gpu_launches"]}))
    dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="kitti_384x1248", choices=list(workloads.CONFIGS))
    ap.add_argument("--precision", default="parity", choices=["parity", "fast"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tc", action="store_true", help="force the CUDA-core conv kernels")
    ap.add_argument("--breakdown", action="store_true", help="print per-entry-point GPU time of one forward and exit")
    ap.add_argument("--hshard", action="store_true",
                    help="configs[4] mode: ONE pair per step, its rows split over the N ranks (halo exchange + 3 "
                         "all-reduces per forward, strong scaling); needs torchrun with N > 1")
    ap.add_argument("--batch", type=int, default=0,
                    help="configs[2] mode: a step is BATCH pairs in total, split BATCH/N per GPU (each rank runs its share "
                         "as consecutive single-pair forwards); 0 (default) = one pair per GPU per step")
    ap.add_argument("--sub-batch", type=int, default=4,
                    help="--batch mode: pairs per forward call (a rank's share is processed in forwards of this many pairs)")
    ap.add_argument("--latency-steps", type=int, default=200,
                    help="extra latency loop after the K timed steps (p50/p90 in the `latency` key; 0 = skip)")
    ap.add_argument("--no-images", action="store_true", help="skip the images -> disparity record (`e2e_images` key)")
    ap.add_argument("--no-graph", action="store_true", help="skip the CUDA-graph latency record (`graph` key)")
    ap.add_argument("--no-hshard-record", action="store_true",
                    help="N > 1: skip the H-sharded Middlebury sub-record (configs[4]) appended to the line")
    ap.add_argument("--hshard-transport", default="p2p", choices=["nccl", "p2p"],
                    help="halo rows by NCCL send/recv or by peer-memory stores (csrc/halo_p2p.cu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write pred4 and prob_volume2 of rank 0's last timed step as DIR/<name>.npy "
                         "(float32, pairs of the step concatenated; a fixed sample when over 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.hshard or args.breakdown):
        ap.error("--dump-outputs applies to the --impl ours throughput run (not --hshard or --breakdown)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    H, W, maxdisp, B = workloads.CONFIGS[args.config]
    global METRIC
    if args.config != "kitti_384x1248":
        METRIC = f"{args.config} pairs/s"

    if args.impl == "reference":
        if rank != 0:
            return 0
        steps, warmup = max(1, args.steps), max(0, args.warmup)
        v, ms, cores, kind, sample = cpu_arm(args.config, steps, warmup, 150.0)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
                "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": common_config(args.config, args.gpus, args.batch, args.sub_batch),
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    assert torch.cuda.is_available(), "bench.py --impl ours needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import dcanet_b200 as d
    affinity0 = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa = d.pipeline.bind_host_to_gpu_numa(local_rank)      # before any pinned allocation (first touch)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)

    if args.no_tc:
        d.engine.Options.use_tc = False
    K, Wm = max(1, args.steps), max(3, args.warmup)
    if args.batch and args.batch % world:
        raise SystemExit(f"--batch {args.batch} does not split over {world} ranks")
    ppr = args.batch // world if args.batch else 1          # pairs per rank and step
    if args.batch:
        # configs[2]: a rank's share of the batch runs as forwards over `sub_batch` pairs each: the kernels' grids scale with
        # the batch, which fills the last wave of every single-wave persistent kernel (KITTI: +3 % at 2, +5.5 % at 4 pairs
        # per forward, results bit-identical per pair: benchmarks/batch_probe.py)
        sb = max(1, min(args.sub_batch, ppr))
        while ppr % sb:
            sb -= 1
        B, ppr = sb, ppr // sb
    net = workloads.init_bench_weights_(d.GwcNet(maxdisp, precision=args.precision), 0).to(dev).eval()
    H4, W4 = H // 4, W // 4

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    if args.hshard:
        return run_hshard(args, d, net, dist, dev, rank, world, barrier, K, Wm)

    nsets = 4   # rotate input sets: 4 x 80 MB > L2, and every step streams a 368 MB volume (>> 126 MB L2)
    host_sets = [workloads.feature_maps(100 * rank + s, B, H4, W4, pin=True) for s in range(nsets)]
    dev_sets = [[t.to(dev, non_blocking=True) for t in hs] for hs in host_sets]
    torch.cuda.synchronize()

    if args.breakdown:
        with torch.no_grad():
            for i in range(3):
                net.hot_path(*dev_sets[i % nsets])
            torch.cuda.synchronize()
            d._lib.PROFILE = []
            n_rep = 5
            for i in range(n_rep):
                net.hot_path(*dev_sets[i % nsets])
            agg = d._lib.profile_summary()
            d._lib.PROFILE = None
        tot = sum(v[1] for v in agg.values())
        print(f"per-forward GPU time by entry point ({args.config}, {args.precision}); total {tot / n_rep:.3f} ms")
        for k, (n, ms) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            print(f"{ms / n_rep:8.3f} ms  {n // n_rep:3d}x  {100 * ms / tot:5.1f}%  {k}")
        return 0

    # ---------------- device-resident throughput ----------------
    with torch.no_grad():
        def step(i, keep=None):
            for j in range(ppr):
                res = net.hot_path(*dev_sets[(i * ppr + j) % nsets])
                if keep is not None:
                    keep.append(res)

        for i in range(Wm):
            step(i)
        d._lib.LAUNCHES = 0
        gc.collect()
        gc.disable()                     # no collector pause inside the timed regions
        sampler = ClockSampler(local_rank)
        if rank == 0 and sampler.interval > 0:
            sampler.start()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        last_step = [] if args.dump_outputs and rank == 0 else None
        barrier()
        ev[0].record()
        for i in range(K):
            step(i, last_step if i == K - 1 else None)
            ev[i + 1].record()
        barrier()
        launches = d._lib.LAUNCHES
        step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(K)]
        total_ms = ev[0].elapsed_time(ev[K])
        if last_step is not None:        # to the host before anything else runs; written at the end
            outputs = {"pred4": torch.cat([p for p, _ in last_step]).float().cpu(),
                       "prob_volume2": torch.cat([v for _, v in last_step]).float().cpu()}
            del last_step

        # ---------------- roofline of the dominant kernel: conv3d k3 s1 32->32 at 1/4 res ----------------
        # (timed right after the headline loop: the long latency / graph / two-stream loops further down leave the GPU at its
        #  power cap, and a kernel timed alone after them reads 12 % low)
        roof = None
        extra = {}
        if rank == 0:
            hbm, tf_burst, tf_sust, src = measured_peaks()
            E = d.engine
            P = net._planes
            x = E.Planes(B, maxdisp // 4, H4, W4, 32, P, dev)
            x.t.normal_()
            pc = net.packed().dres0_2
            for _ in range(3):
                E.conv(x, pc, E.K3S1, E.ACT_RELU)
            n_it = 10
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(n_it):
                E.conv(x, pc, E.K3S1, E.ACT_RELU)
            b_.record()
            torch.cuda.synchronize()
            conv_ms = a.elapsed_time(b_) / n_it
            fl = workloads.conv_k3s1_flops(H, W, maxdisp) * B
            ach = fl / (conv_ms * 1e-3) / 1e12
            kernel_name = "conv3d_tc" if (E.Options.use_tc and pc.w_tc is not None and E.tc_supported(E.K3S1, 32, 32)) \
                else "conv_direct_kernel<32,16> (CUDA-core fp32)"
            tr = ncu_traffic("conv_tc_march_kernel<32, %d, 0" % P) if kernel_name == "conv3d_tc" else None
            issued = 3.0 if (P == 2 and kernel_name == "conv3d_tc") else 1.0
            roof = {"kernel": f"{kernel_name} (conv_tc_march_kernel, tcgen05) k3 s1 32->32 @ {maxdisp // 4}x{H4}x{W4}", "bound": "tensor",
                    "achieved": ach, "peak": tf_sust, "unit": "TFLOP/s", "frac": ach / tf_sust,
                    "traffic": tr["bytes"] if tr else None,
                    "peak_source": f"{src} (bf16 sustained; burst {tf_burst})", "ms_per_launch": conv_ms,
                    "algorithmic_flops_per_launch": fl,
                    "issued_tflops": ach * issued,
                    "note": ("parity precision issues 3 16-bit (kind::f16, same rate as bf16) MMAs per algorithmic MAC (hi*Whi, hi*Wlo, lo*Whi); "
                             "`achieved` counts algorithmic FLOPs only") if issued > 1 else "",
                    "ncu": tr}
            # the same kernel with single-plane operands (precision="fast": ONE MMA per MAC), to separate the tensor-core
            # efficiency of the kernel from the 3x MMA cost of the parity format
            try:
                x1 = E.Planes(B, maxdisp // 4, H4, W4, 32, 1, dev)
                x1.t.normal_()
                pc1 = E.pack_convbn(net.dres0[2])
                pc1.pack_tc(1)
                for _ in range(3):
                    E.conv(x1, pc1, E.K3S1, E.ACT_RELU)
                torch.cuda.synchronize()
                a.record()
                for _ in range(n_it):
                    E.conv(x1, pc1, E.K3S1, E.ACT_RELU)
                b_.record()
                torch.cuda.synchronize()
                f_ms = a.elapsed_time(b_) / n_it
                extra["roofline_fast_mode"] = {"kernel": "conv_tc_march_kernel<32,1> (single fp16 plane, one MMA per MAC)",
                                               "bound": "tensor", "achieved": fl / (f_ms * 1e-3) / 1e12, "peak": tf_sust,
                                               "unit": "TFLOP/s", "frac": fl / (f_ms * 1e-3) / 1e12 / tf_sust,
                                               "ms_per_launch": f_ms, "note": "not the parity configuration; context only"}
                del x1, pc1
            except Exception as e:          # context record only
                extra["roofline_fast_mode"] = {"error": str(e)}
            # volume kernel (HBM bound)
            fs = dev_sets[0]
            for _ in range(3):
                E.fused_volume(fs[0], fs[1], fs[2], fs[3], maxdisp // 4, 40, P)
            torch.cuda.synchronize()
            a.record()
            for i in range(n_it):
                fs = dev_sets[i % nsets]
                E.fused_volume(fs[0], fs[1], fs[2], fs[3], maxdisp // 4, 40, P)
            b_.record()
            torch.cuda.synchronize()
            vol_ms = a.elapsed_time(b_) / n_it
            vb = workloads.volume_bytes(H, W, maxdisp, P) * B
            extra["roofline_volume"] = {"kernel": "volume_fused3_kernel (TMA-staged)", "bound": "hbm",
                                        "achieved": vb / (vol_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                        "frac": vb / (vol_ms * 1e-3) / 1e9 / hbm,
                                        "traffic": (ncu_traffic("volume_fused3_kernel") or {}).get("bytes"),
                                        "ms_per_launch": vol_ms, "algorithmic_bytes_per_launch": vb,
                                        "peak_source": src}

        # ---------------- end to end: pinned host feature maps -> H2D -> hot path -> D2H disparity ----------
        out4 = torch.empty((B, 1, H, W), dtype=torch.float32).pin_memory()
        outpv = torch.empty((B, maxdisp // 8, H // 8, W // 8), dtype=torch.float32).pin_memory()
        h2d = sum(t.numel() * 4 for t in host_sets[0])
        d2h = out4.numel() * 4 + outpv.numel() * 4

        # the repo's public streaming API: H2D of pair i+1 overlaps the kernels of pair i (2 streams + events);
        # every pair's inputs start in pinned HOST memory and its results end in pinned HOST memory
        pipe = d.HotPathPipeline(net, depth=2)
        for i in range(3):
            pipe.wait(pipe.submit(i, host_sets[i % nsets]))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(pipe.copy_stream)
        last = 0
        for i in range(K * ppr):
            last = pipe.submit(i, host_sets[i % nsets])
        pipe.wait(last)
        e1.record(pipe.compute_stream)
        barrier()
        e2e_ms = e0.elapsed_time(e1)
        if rank == 0:
            sampler.stop()

        # ---------------- end to end from IMAGES (SURVEY 8d config 2: "including the front end, reported separately") -------
        img_rec = None
        if not args.no_images and not args.batch:
            gi = torch.Generator().manual_seed(1234 + rank)
            imgs = [(torch.randn(B, 3, H, W, generator=gi).pin_memory(), torch.randn(B, 3, H, W, generator=gi).pin_memory())
                    for _ in range(2)]

            def img_steps(n):
                for i in range(n):
                    l, r = imgs[i % 2]
                    p4, pv_ = net(l.to(dev, non_blocking=True), r.to(dev, non_blocking=True))
                    out4.copy_(p4, non_blocking=True)
                    outpv.copy_(pv_, non_blocking=True)

            def fe_steps(n):
                with d.frontend._no_tf32():          # as GwcNet.forward runs it: cuDNN in true fp32
                    for i in range(n):
                        l, r = imgs[i % 2]
                        ld = l.to(dev, non_blocking=True)
                        net.feature_extraction(torch.cat((ld, r.to(dev, non_blocking=True)), 0))
                        net.guidance(ld)

            img_rec = {"h2d_bytes_per_step": 2 * B * 3 * H * W * 4, "d2h_bytes_per_step": d2h, "n_gpus": world,
                       "what": "GwcNet(left, right): pinned host images -> H2D -> feature_extraction (left+right as one batch) "
                               "+ Guidance -> hot path -> D2H of pred4 + prob_volume2.  kernel_front_end: every conv of the front end "
                               "on this repo's kernels (frontend.py); torch_front_end: the same modules on cuDNN in true "
                               "fp32 (TF32 off)"}
            for tag, on in (("kernel_front_end", True), ("torch_front_end", False)):
                d.frontend.Options.enabled = on
                for fn, key in ((img_steps, "pairs_per_s"), (fe_steps, "front_end_ms")):
                    fn(8)                   # (cuDNN picks its algorithms and the allocator grows during the first calls)
                    a_, b__ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    barrier()
                    a_.record()
                    fn(K)
                    b__.record()
                    barrier()
                    ms_ = a_.elapsed_time(b__) / K
                    if dist is not None:                     # max over ranks, as for the headline
                        t_ = torch.tensor([ms_], dtype=torch.float64, device=dev)
                        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
                        ms_ = float(t_[0])
                    img_rec.setdefault(tag, {})[key] = (world * B / (ms_ * 1e-3)) if key == "pairs_per_s" else ms_
            d.frontend.Options.enabled = True

        # ---------------- latency distribution (SURVEY 8d config 2: 20 warm-up + 200 timed), extra key only ----------
        n_lat = max(0, args.latency_steps)
        lat = None
        if n_lat:
            evl = [torch.cuda.Event(enable_timing=True) for _ in range(n_lat + 1)]
            for i in range(20):
                net.hot_path(*dev_sets[i % nsets])
            barrier()
            evl[0].record()
            for i in range(n_lat):
                net.hot_path(*dev_sets[i % nsets])
                evl[i + 1].record()
            barrier()
            ls = sorted(evl[i].elapsed_time(evl[i + 1]) / B for i in range(n_lat))
            lat = {"steps": n_lat, "warmup": 20, "p50_ms_per_pair": ls[n_lat // 2], "p90_ms_per_pair": ls[int(0.9 * n_lat)],
                   "p99_ms_per_pair": ls[min(n_lat - 1, int(0.99 * n_lat))], "mean_ms_per_pair": sum(ls) / n_lat,
                   "pairs_per_s": n_lat * B / (evl[0].elapsed_time(evl[n_lat]) * 1e-3)}
        # ---------------- the same forward as ONE CUDA graph (engine.GraphedHotPath), extra key only ----------
        graph_rec = None
        if n_lat and not args.no_graph:
            def p50_of(fn, n, warm, sync=barrier):
                evg = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
                for i in range(warm):
                    fn(i)
                sync()
                evg[0].record()
                for i in range(n):
                    fn(i)
                    evg[i + 1].record()
                sync()
                ts = sorted(evg[i].elapsed_time(evg[i + 1]) for i in range(n))
                return ts[n // 2], ts[int(0.9 * n)], n / (evg[0].elapsed_time(evg[n]) * 1e-3)

            p50, p90, pps = p50_of(lambda i: net.hot_path_graphed(*dev_sets[i % nsets]), n_lat, 20)
            graph_rec = {"what": "hot_path_graphed: the whole forward as one cudaGraphLaunch per pair (one graph per input "
                                 "set, shared pool); results copied out of the graph's buffers",
                         "steps": n_lat, "p50_ms_per_pair": p50 / B, "p90_ms_per_pair": p90 / B, "pairs_per_s": pps * B}
            if rank == 0:
                # the launch-bound regime: tiny_64x128 (maxdisp 48), eager launches vs graph replay
                tH, tW, tD, tB = workloads.CONFIGS["tiny_64x128"]
                tnet = workloads.init_bench_weights_(d.GwcNet(tD, precision=args.precision), 0).to(dev).eval()
                tf = [t.to(dev) for t in workloads.feature_maps(7, tB, tH // 4, tW // 4)]
                e50, e90, _ = p50_of(lambda i: tnet.hot_path(*tf), 100, 10, torch.cuda.synchronize)
                g50, g90, _ = p50_of(lambda i: tnet.hot_path_graphed(*tf), 100, 10, torch.cuda.synchronize)
                graph_rec["tiny_64x128"] = {"eager_p50_ms": e50, "eager_p90_ms": e90, "graph_p50_ms": g50, "graph_p90_ms": g90}
                del tnet, tf
        # ---------------- independent pairs in flight on two streams (throughput only), extra key ----------
        ms_rec = None
        if n_lat and not args.no_graph:
            sts = [torch.cuda.Stream(device=dev) for _ in range(2)]
            for i in range(4):
                with torch.cuda.stream(sts[i % 2]):
                    net.hot_path(*dev_sets[i % nsets])
            barrier()
            m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            m0.record()
            for st_ in sts:
                st_.wait_event(m0)
            for i in range(n_lat):
                with torch.cuda.stream(sts[i % 2]):
                    net.hot_path(*dev_sets[i % nsets])
            for st_ in sts:
                torch.cuda.current_stream().wait_stream(st_)
            m1.record()
            barrier()
            ms_rec = {"streams": 2, "steps": n_lat, "pairs_per_s_per_gpu": n_lat * B / (m0.elapsed_time(m1) * 1e-3),
                      "what": "the same forwards issued alternately on two CUDA streams: a pair's kernels take the SMs that "
                              "the tail of the other pair's single-wave persistent kernel leaves idle (compare with "
                              "latency.pairs_per_s, the one-stream rate over the same number of steps)"}
        gc.enable()

    # ---------------- configs[4] sub-record: one Middlebury pair H-sharded over the N ranks ----------------
    hrec = None
    if dist is not None and not args.no_hshard_record and not args.batch:
        del dev_sets, host_sets, pipe
        torch.cuda.empty_cache()
        mcfg = "middlebury_1536x2048"
        mnet = workloads.init_bench_weights_(d.GwcNet(workloads.CONFIGS[mcfg][2], precision=args.precision), 0).to(dev).eval()
        hrec = measure_hshard(mcfg, args.hshard_transport, d, mnet, dist, dev, rank, world, barrier, 10, 3)
        # the un-sharded time of the same pair on ONE GPU (rank 0's device; the other ranks idle), for the speed-up
        if rank == 0:
            fm = [t.to(dev) for t in workloads.feature_maps(0, 1, 1536 // 4, 2048 // 4)]
            with torch.no_grad():
                for _ in range(2):
                    mnet.hot_path(*fm)
                a1, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a1.record()
                for _ in range(5):
                    mnet.hot_path(*fm)
                b1.record()
                torch.cuda.synchronize()
            hrec["unsharded_ms_per_pair_1gpu"] = a1.elapsed_time(b1) / 5
            hrec["speedup_vs_1gpu"] = hrec["unsharded_ms_per_pair_1gpu"] / hrec["ms_per_pair"]
            del fm
        del mnet
        barrier()

    # max over ranks
    tt = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = float(tt[0]), float(tt[1])
    pairs = K * B * ppr * world
    if rank == 0:
        line = {"metric": METRIC, "value": pairs / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
                "warmup": Wm, "ms_per_step": total_ms / K, "p50_ms_per_pair": statistics.median(step_ms) / B / ppr,
                "max_step_ms": max(step_ms), "max_step_index": step_ms.index(max(step_ms)),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16x2 split operands (hi+lo fp16 planes, 22-bit significand), fp32 accumulate" if args.precision == "parity"
                else "f16 operands, fp32 accumulate",
                "data": "synthetic",
                "config": common_config(args.config, world, args.batch, args.sub_batch),
                "precision_mode": args.precision,
                "clocks": sampler.summary(),
                "e2e": {"value": pairs / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d * ppr,
                        "d2h_bytes_per_step": d2h * ppr, "ms_per_step": e2e_ms / K,
                        "what": "HotPathPipeline: pinned host feature maps -> H2D (copy stream, overlapped) -> hot path -> D2H of pred4 + prob_volume2 into pinned host buffers"},
                "gpu_launches": launches,
                "roofline": roof}
        line.update(extra)
        if lat is not None:
            line["latency"] = lat
        if graph_rec is not None:
            line["graph"] = graph_rec
        if img_rec is not None:
            line["e2e_images"] = img_rec
        if ms_rec is not None:
            line["multi_stream"] = ms_rec
        if hrec is not None:
            line["hshard"] = hrec
        line["host"] = {"numa_node_bound": numa, "cpus": len(os.sched_getaffinity(0)) if affinity0 is not None else None}
        if affinity0 is not None:
            os.sched_setaffinity(0, affinity0)          # the CPU arm below uses every host core again
        if world == 1 and not args.no_cpu_baseline:
            v, ms, cores, kind, sample = cpu_arm(args.config, 2, 1, 25.0)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                                    "ms_per_pair": ms}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
