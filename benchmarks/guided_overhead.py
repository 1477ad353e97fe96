"""Cost of the LiDAR guidance (include/dca_b200.h section 14) at KITTI size, 384x1248, maxdisp 192, parity precision,
synthetic weights and a synthetic 120k-point scan on the device.

Prints one JSON line:
  volume_us            dca_volume_gwc_concat vs dca_volume_gwc_concat_guided (TMA-staged kernel, 40 groups) per launch,
                       at B = 1 and B = 8, alternated A B A B in this process (CUDA events over STEPS launches each);
                       `ratio` compares the better run of each.  The hint map is the projected scan (its 1/4-res
                       coverage is reported as hq_density)
  quarter_us           dca_guide_quarter of one 384x1248 hint map
  lidar_hints_us       guide.lidar_hints of one 120k-point device scan (three launches and the offsets upload)
  pair_ms              model(l, r) and model(l, r, hints=) from images, alternated; `ratio` as above
  gpu, power_limit_w   what the numbers were measured on

    python benchmarks/guided_overhead.py
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
import workloads  # noqa: E402
from confidence_overhead import gpu_name_power, time_ms  # noqa: E402

STEPS = 200


def kitti_like_calib():
    """A KITTI-like rig: velodyne x forward, y left, z up, 8 cm above and 27 cm behind camera 2."""
    V = np.array([[0.0, -1.0, 0.0, 0.0], [0.0, 0.0, -1.0, -0.08], [1.0, 0.0, 0.0, -0.27]])
    R = np.vstack([V, [0, 0, 0, 1]])
    return d.StereoCalib(721.5377, 721.5377, 609.5593, 172.854, 0.5372, 0.0, np.linalg.inv(R)[:3], V)


def scan(calib, n, seed=0):
    """n points over the camera's view and around it, depth 2..80 m -> float32 [n, 4] in the velodyne frame."""
    rng = np.random.default_rng(seed)
    u, v, Z = rng.uniform(-100, 1342, n), rng.uniform(-50, 425, n), rng.uniform(2.0, 80.0, n)
    P = np.stack([(u - calib.cx) * Z / calib.fx, (v - calib.cy) * Z / calib.fy, Z, np.ones(n)], -1)
    T = np.vstack([calib.rect_to_velo.astype(np.float64), [0, 0, 0, 1]])
    return np.hstack([(P @ T.T)[:, :3], rng.uniform(0, 1, (n, 1))]).astype(np.float32)


def alternate(fns, steps, rounds=2):
    runs = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            runs[k].append(time_ms(fn, steps, warmup=10) / steps)
    return runs


def main():
    if not torch.cuda.is_available():
        raise SystemExit("guided_overhead.py needs a CUDA device")
    E = d.engine
    H, W, maxdisp, _ = workloads.CONFIGS["kitti_384x1248"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    calib = kitti_like_calib()
    pts = torch.from_numpy(scan(calib, 120_000)).to(dev)
    with torch.no_grad():
        hints = d.lidar_hints(pts, calib, (H, W), window=(9, 0, 375, 1242, 0))
        hq1 = E.guide_quarter(hints[:, 0].contiguous(), maxdisp)
    k, s = 10.0, d.guide.modulation_scale(10.0, 1.0)
    out = {"config": f"{H}x{W} maxdisp {maxdisp}, parity, 120k-point synthetic scan, k={k} c=1.0",
           "hint_density": float((hints > 0).float().mean()), "hq_density": float((hq1 > 0).float().mean())}

    vol = {}
    for B in (1, 8):
        f = [t.to(dev) for t in workloads.feature_maps(0, B, H // 4, W // 4)]
        hq = hq1.expand(B, -1, -1).contiguous()
        fns = {"plain": lambda: E.fused_volume(f[0], f[1], f[2], f[3], maxdisp // 4, 40, 2),
               "guided": lambda: E.fused_volume(f[0], f[1], f[2], f[3], maxdisp // 4, 40, 2, guide=(hq, k, s))}
        runs = alternate(fns, STEPS)
        vol[f"B{B}"] = {kk: [round(1e3 * x, 2) for x in v] for kk, v in runs.items()}
        vol[f"B{B}"]["ratio"] = round(min(runs["guided"]) / min(runs["plain"]), 4)
        del f, hq
    out["volume_us"] = vol

    hm = hints[:, 0].contiguous()
    out["quarter_us"] = round(1e3 * time_ms(lambda: E.guide_quarter(hm, maxdisp), STEPS) / STEPS, 2)
    out["lidar_hints_us"] = round(1e3 * time_ms(lambda: d.lidar_hints(pts, calib, (H, W)), STEPS) / STEPS, 2)

    net = workloads.init_bench_weights_(d.GwcNet(maxdisp, precision="parity"), 0).to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(0)
    left, right = torch.randn(1, 3, H, W, device=dev, generator=g), torch.randn(1, 3, H, W, device=dev, generator=g)
    with torch.no_grad():
        runs = alternate({"plain": lambda: net(left, right), "guided": lambda: net(left, right, hints=hints)}, 50)
    out["pair_ms"] = {kk: [round(x, 3) for x in v] for kk, v in runs.items()}
    out["pair_ms"]["ratio"] = round(min(runs["guided"]) / min(runs["plain"]), 4)
    out.update(gpu=name, power_limit_w=plimit)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
