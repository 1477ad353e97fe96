"""Cost of TSDF fusion (dca_tsdf_integrate) and of the surface extraction (dca_tsdf_count_surface +
dca_tsdf_extract_surface) at KITTI size: a 375x1242 window with KITTI's intrinsics, 0.1 m voxels, an 800x64x800 grid with
colour (80 m x 6.4 m x 80 m, 0.82 GB of state), synthetic depth maps (a ground plane and a wall of boxes, 1 % noise)
on a forward-driving trajectory.

Prints one JSON line:
  integrate_us        per dca_tsdf_integrate call at B = 1 and B = 8: `boxed` = the box of TSDFVolume.integrate at
                      max_depth 40 m, `whole` = the whole grid with the same max_depth; CUDA-event time of STEPS calls
                      captured in one CUDA graph, after a warm-up; `per_frame` = the B = 8 time / 8; `no_depth` =
                      the B = 8 boxed call on depth maps of zeros (every voxel projected, none updated)
  box_voxels          voxels of each box; `updated_voxels` = the voxels the frames update (a fresh volume's voxels
                      with weight > 0 after one call)
  count_us, extract_us, surface_points   the two extraction calls on a volume fused from 16 frames, timed the same way
  bytes_est           bytes per call from the shapes and the counts (integration: the 20 B state of each updated voxel
                      read and written, a voxel no frame updates is neither read nor written, plus the depth, weight
                      and colour maps once) and the time that takes at 7.7 TB/s
  gpu, power_limit_w  what the numbers were measured on

    python benchmarks/tsdf_overhead.py
"""
import json
import math
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
HBM_TBPS = 7.7                    # HGX B200 data sheet, one GPU
H, W = 375, 1242
FX, FY, CX, CY = 721.5377, 721.5377, 609.5593, 172.854
MAX_DEPTH = 40.0


def _graph_us(call):
    """Microseconds per call of `call()`: STEPS calls captured in one CUDA graph, replayed after a warm-up."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()                                               # module load outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(STEPS):
            call()
    return round(1e3 * time_ms(graph.replay, 3, warmup=1) / (3 * STEPS), 3)


def _depth_maps(dev, B, seed):
    """Camera-frame depth [B,H,W]: the ground 1.65 m below the camera and a wall of boxes 12..38 m ahead, 1 % noise."""
    g = torch.Generator(device=dev).manual_seed(seed)
    v = torch.arange(H, device=dev, dtype=torch.float64)[:, None] - CY
    u = torch.arange(W, device=dev, dtype=torch.float64)[None, :] - CX
    ground = torch.where(v > 0, 1.65 * FY / v.clamp(min=1e-9), torch.full_like(v, math.inf)).expand(H, W)
    cols = (u / 40).floor() + seed
    wall = 12 + (torch.sin(cols * 12.9898) * 43758.5453).frac().abs() * 26
    z = torch.minimum(ground, wall.expand(H, W))[None].repeat(B, 1, 1)
    z = z * (1 + 0.01 * torch.randn(z.shape, device=dev, generator=g, dtype=torch.float64))
    return z.float().contiguous()


def main():
    if not torch.cuda.is_available():
        raise SystemExit("tsdf_overhead.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plimit = gpu_name_power(dev)
    calib = d.StereoCalib(FX, FY, CX, CY, 0.54)
    dims = (800, 64, 800)
    vol = d.TSDFVolume((-40.0, -4.6, -2.0), 0.1, dims, device=dev)
    g = torch.Generator(device=dev).manual_seed(1)
    poses = np.tile(np.eye(4), (16, 1, 1))
    poses[:, 2, 3] = np.arange(16) * 1.0                      # 1 m per frame along the optical axis
    poses[:, 0, 3] = np.sin(np.arange(16) * 0.3) * 0.5
    depth = _depth_maps(dev, 16, 0)
    weight = torch.rand((16, H, W), device=dev, generator=g) * 0.5 + 0.5
    rgb = torch.randint(0, 256, (16, H, W, 3), dtype=torch.uint8, device=dev, generator=g)
    intr = (calib.fx, calib.fy, calib.cx, calib.cy)
    T = np.linalg.inv(poses)[:, :3].reshape(16, 12).astype(np.float32)

    integrate_us, box_voxels, updated, bytes_est = {}, {}, {}, {}
    for B in (1, 8):
        boxes = {"boxed": d.fusion.frustum_box(vol.dims, vol.origin, vol.voxel_size, intr, (0, 0, H, W), poses[:B],
                                               MAX_DEPTH, vol.trunc),
                 "whole": (0, 0, 0) + dims}
        vol.reset()
        d.fusion._integrate_kernel(vol, boxes["boxed"], depth[:B], weight[:B], rgb[:B], intr, 0, 0, T[:B], MAX_DEPTH)
        n_up = int((vol.weight > 0).sum())
        updated[f"B{B}"] = n_up
        for k, box in boxes.items():
            vol.reset()
            integrate_us[f"B{B}_{k}"] = _graph_us(lambda box=box: d.fusion._integrate_kernel(
                vol, box, depth[:B], weight[:B], rgb[:B], intr, 0, 0, T[:B], MAX_DEPTH))
            box_voxels[f"B{B}_{k}"] = box[3] * box[4] * box[5]
            bytes_est[f"integrate_B{B}_{k}"] = 2 * 20 * n_up + B * H * W * (4 + 4 + 3)
    integrate_us["B8_boxed_per_frame"] = round(integrate_us["B8_boxed"] / 8, 3)
    # the same call with every depth 0: each frame still projects every voxel of the box, but none is updated, so no
    # state is read or written; the difference to B8_boxed is what the state traffic and the update cost
    no_depth = torch.zeros_like(depth[:8])
    vol.reset()
    integrate_us["B8_boxed_no_depth"] = _graph_us(lambda: d.fusion._integrate_kernel(
        vol, boxes["boxed"], no_depth, weight[:8], rgb[:8], intr, 0, 0, T[:8], MAX_DEPTH))

    vol.reset()
    vol.integrate(depth, calib, poses, weight=weight, rgb=rgb, max_depth=MAX_DEPTH)
    surf = vol.extract(0.5)
    n = int(surf.xyz.shape[0])
    N = math.prod(dims)
    tiles = (N + d.fusion.TILE - 1) // d.fusion.TILE
    ws = torch.empty(tiles, dtype=torch.int64, device=dev)
    cnt = torch.empty(1, dtype=torch.int64, device=dev)
    xyz, nrm = torch.empty((n, 3), device=dev), torch.empty((n, 3), device=dev)
    col = torch.empty((n, 3), dtype=torch.uint8, device=dev)

    def count():
        d._lib.call("dca_tsdf_count_surface", vol.state.data_ptr(), 5, *dims, 0.5, ws.data_ptr(), cnt.data_ptr(),
                    torch.cuda.current_stream().cuda_stream)

    def extract():
        d._lib.call("dca_tsdf_extract_surface", vol.state.data_ptr(), 5, *dims, *vol.origin, vol.voxel_size, 0.5,
                    ws.data_ptr(), n, xyz.data_ptr(), nrm.data_ptr(), col.data_ptr(),
                    torch.cuda.current_stream().cuda_stream)

    count_us = _graph_us(count)
    extract_us = _graph_us(extract)
    assert int(cnt[0]) == n and torch.equal(xyz, surf.xyz) and torch.equal(col, surf.rgb)
    bytes_est["count"] = 8 * N + 8 * tiles
    bytes_est["extract"] = 8 * N + 8 * tiles + 27 * n
    hbm = {k: round(v / (HBM_TBPS * 1e12) * 1e6, 3) for k, v in bytes_est.items()}
    print(json.dumps({
        "workload": f"{H}x{W} window, KITTI intrinsics, grid {dims} x 0.1 m with colour ({vol.nbytes / 1e9:.2f} GB), "
                    f"max_depth {MAX_DEPTH} m, synthetic depth",
        "gpu": name, "power_limit_w": plimit,
        "integrate_us": integrate_us, "box_voxels": box_voxels, "updated_voxels": updated,
        "count_us": count_us, "extract_us": extract_us, "surface_points": n,
        "bytes_est": bytes_est, "hbm_time_us_at_7.7_tbps": hbm, "steps": STEPS,
    }), flush=True)


if __name__ == "__main__":
    main()
