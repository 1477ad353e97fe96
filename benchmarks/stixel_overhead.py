"""Cost of the Stixel World at KITTI size: a 375x1242 window with KITTI's intrinsics and a synthetic disparity (a road
seen from 1.65 m at 1 degree of pitch, five boxes 8..38 m ahead, a wall at 60 m, a sky band; +-0.3 px noise, 5 %
outliers, 10 % invalid pixels), max_disp 192, the default priors and width 5.

Prints one JSON line:
  ground_us_b1 / _b8     one ground_profile call (CUDA-event time of STEPS calls captured in one CUDA graph)
  stixels_us_b1 / _b8    one stixels call, timed the same way (column reduction, object lut, DP)
  render_us_b1 / _b8     one Stixels.render call, timed the same way
  split_us_b1            per kernel of one ground_profile + stixels + render at B = 1 (torch.profiler, a separate run)
  forward_ms, forward_stixels_ms   GwcNet(192) with the bench weights on a 384x1248 pair, from images, without and with
                         ground_profile + stixels + render of the 375x1242 window, alternated ROUNDS times in one process
                         (CUDA events, FWD_STEPS calls per round; the medians)
  segments_per_column    the mean segment count of the synthetic scene
  gpu, power_limit_w     what the numbers were measured on

    python benchmarks/stixel_overhead.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dcanet_b200 as d  # noqa: E402
from _stixel_restatement import driving_scene  # noqa: E402
from confidence_overhead import gpu_name_power, time_ms  # noqa: E402

STEPS = 50
ROUNDS = 5
FWD_STEPS = 10


def _graph_us(call):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(STEPS):
            call()
    return round(1e3 * time_ms(graph.replay, 3, warmup=1) / (3 * STEPS), 2)


def _split(call):
    from torch.profiler import ProfilerActivity, profile
    call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            call()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.count:
            name = e.key.split("(")[0].replace("void ", "").replace("dca::", "")
            out[name] = round(e.device_time_total / e.count, 2) if hasattr(e, "device_time_total") else None
    return out


def main():
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    res = {}
    for B in (1, 8):
        disp = torch.from_numpy(np.stack([driving_scene(b)[0] for b in range(B)])).to(dev)
        g = d.ground_profile(disp)
        st = d.stixels(disp, g)
        res[f"ground_us_b{B}"] = _graph_us(lambda: d.ground_profile(disp))
        res[f"stixels_us_b{B}"] = _graph_us(lambda: d.stixels(disp, g))
        res[f"render_us_b{B}"] = _graph_us(lambda: st.render(g))
        if B == 1:
            res["segments_per_column"] = round(float(st.count.float().mean()), 3)
            res["split_us_b1"] = _split(lambda: (lambda gg: d.stixels(disp, gg).render(gg))(d.ground_profile(disp)))

    import workloads
    net = workloads.init_bench_weights_(d.GwcNet(192), 0).to(dev).eval()
    gen = torch.Generator(device=dev).manual_seed(0)
    left = torch.randn(1, 3, 384, 1248, device=dev, generator=gen)
    right = torch.roll(left, -4, 3)
    window = (9, 0, 375, 1242, 0)

    def plain():
        with torch.no_grad():
            net(left, right)

    def with_stixels():
        with torch.no_grad():
            out = net(left, right)
            pred = out[0] if isinstance(out, (tuple, list)) else out
            gg = d.ground_profile(pred, window=window)
            d.stixels(pred, gg, window=window).render(gg)

    plain(), with_stixels()
    a, b = [], []
    for _ in range(ROUNDS):
        a.append(time_ms(plain, FWD_STEPS, warmup=2) / FWD_STEPS)
        b.append(time_ms(with_stixels, FWD_STEPS, warmup=2) / FWD_STEPS)
    res["forward_ms"] = round(float(np.median(a)), 3)
    res["forward_stixels_ms"] = round(float(np.median(b)), 3)
    res.update(gpu=name, power_limit_w=plimit)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
