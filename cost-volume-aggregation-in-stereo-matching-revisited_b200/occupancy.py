"""2-D occupancy grid of posed depth maps on the GPU, in log-odds (include/dca_b200.h section 17).

  OccupancyGrid   log_odds fp32 [ny, nx] and updates int32 [ny, nx] of a fixed grid on the ground plane of the world;
                  .integrate(depth, calib, cam_to_world, weight=, window=, max_depth=) runs one
                  dca_occupancy_integrate per 16 frames (a workspace memset and three launches, no host sync) on the
                  cells the frames can reach.  Per frame, the pixels between h_lo and h_hi above the road are obstacle
                  hits of the cell they fall in, and along each group of col_width image columns the road in front of
                  the first obstacle is free (the polar free-space model of Badino, Franke & Mester 2007).
                  .probability(), .classes() (FREE / OCCUPIED / UNKNOWN), .save_map(stem) (a ROS map_server
                  trinary PGM + YAML) and .agreement(other) (the same cells of two maps compared, e.g. stereo against
                  a LiDAR map of the same drive)

fuse_files(..., volume=grid) fills a grid through the same FusePipeline as a TSDF volume; motion= and the filters
apply unchanged, since moving objects reach the grid as zero weights.  The default band and min_hits were chosen on a
synthetic road scene; they are not tuned for DCANet or KITTI.
"""
import math
import os
from typing import NamedTuple

import numpy as np
import torch

from . import _lib, engine
from .fusion import _bhw, _poses, _window_origin

FREE, OCCUPIED, UNKNOWN = 0, 1, 2            # classes()
MAX_FRAMES = 16                              # DCA_OCC_MAX_FRAMES: frames per dca_occupancy_integrate call
MAX_COL_WIDTH = 64                           # DCA_OCC_MAX_COL_WIDTH
MAX_BINS = 8192                              # DCA_OCC_MAX_BINS
MAX_HITS = 1 << 20                           # DCA_OCC_MAX_HITS
# KITTI's camera world frame (X right, Y down, Z forward) -> grid x = X, grid y = Z, up = -Y
KITTI_WORLD_TO_GRID = np.array([[1.0, 0, 0, 0], [0, 0, 1, 0], [0, -1, 0, 0], [0, 0, 0, 1]])


def nbins(max_depth, range_res):
    """DCA_OCC_BINS: floorf(max_depth / range_res) + 1 in fp32."""
    return int(np.floor(np.float32(max_depth) / np.float32(range_res))) + 1


def workspace_bytes(B, bi, bj, ncols, bins):
    """DCA_OCC_WORKSPACE_BYTES: hits int32 [B][bj][bi], occ int32 [B][ncols][bins], near / far / first [B][ncols]."""
    return 4 * B * (bi * bj + ncols * (bins + 3))


def _integrate_kernel(grid, box, depth, weight, intrinsics, u0, v0, M, Minv, max_depth):
    """One dca_occupancy_integrate of B <= 16 frames: depth (and weight) fp32 [B,h,w] sharing one layout (unit column
    stride), M / Minv float32 [B,12] (grid <- camera, camera <- grid), box (i0, j0, bi, bj)."""
    engine._require_cuda(grid.log_odds, depth, weight)
    B, H, W = depth.shape
    pitch_row = depth.stride(1)
    pitch_img = depth.stride(0) if B > 1 else H * pitch_row
    ncols = (W + grid.col_width - 1) // grid.col_width
    ws = torch.empty((workspace_bytes(B, box[2], box[3], ncols, nbins(max_depth, grid.range_res)),), dtype=torch.uint8,
                     device=depth.device)
    m, mi = np.ascontiguousarray(M, np.float32), np.ascontiguousarray(Minv, np.float32)
    nx, ny = grid.dims
    _lib.call("dca_occupancy_integrate", grid.log_odds.data_ptr(), grid.updates.data_ptr(), nx, ny, *grid.origin,
              grid.cell_size, *box, depth.data_ptr(), 0 if weight is None else weight.data_ptr(), pitch_row, pitch_img,
              B, H, W, *intrinsics, u0, v0, m.ctypes.data, mi.ctypes.data, grid.camera_height, *grid.band,
              grid.col_width, grid.range_res, max_depth, grid.min_hits, grid.l_hit, grid.l_miss, grid.l_min,
              grid.l_max, ws.data_ptr(), torch.cuda.current_stream(depth.device).cuda_stream)


def frustum_box(dims, origin, cell_size, intrinsics, window, cam_to_grid, max_depth, range_res):
    """The cell box (i0, j0, bi, bj) that holds every cell the frames can update, or None when no cell can: the float64
    bounds in the grid plane of the camera centres and of the window corners (pixel edges, +-0.5 px) at camera
    Z = max_depth + range_res (the farthest a free cell's sample can lie), grown by one cell and clipped to the grid.
    The whole grid when those bounds are not finite."""
    fx, fy, cx, cy = intrinsics
    u0, v0, h, w = window
    Z = float(max_depth) + float(range_res)
    pts = [(0.0, 0.0, 0.0)]
    for u in (u0 - 0.5, u0 + w - 0.5):
        for v in (v0 - 0.5, v0 + h - 0.5):
            pts.append(((u - cx) / fx * Z, (v - cy) / fy * Z, Z))
    pts = np.array(pts, np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        g = np.einsum("bij,nj->bni", cam_to_grid[:, :2, :3], pts) + cam_to_grid[:, None, :2, 3]
    if not np.isfinite(g).all():
        return (0, 0) + tuple(dims)
    lo, hi = g.reshape(-1, 2).min(0), g.reshape(-1, 2).max(0)
    o, n = np.asarray(origin, np.float64), np.asarray(dims)
    with np.errstate(over="ignore"):
        a = np.maximum(np.floor((lo - o) / cell_size) - 1, 0)
        b = np.minimum(np.ceil((hi - o) / cell_size) + 1, n - 1)
    if (a > b).any():
        return None
    a, b = a.astype(int), b.astype(int)
    return int(a[0]), int(a[1]), int(b[0] - a[0] + 1), int(b[1] - a[1] + 1)


class Agreement(NamedTuple):
    """Two maps compared over the cells known (FREE or OCCUPIED) in both: known = their number, agree = those of the
    same class; occupied_both / occupied_either and free_both / free_either count the cells of that class in both / in
    either map.  occupied_iou = occupied_both / occupied_either, free_iou likewise, accuracy = agree / known (NaN over
    an empty set)."""
    known: int
    agree: int
    occupied_both: int
    occupied_either: int
    free_both: int
    free_either: int
    occupied_iou: float
    free_iou: float
    accuracy: float


def _f32(v, what, test, hint):
    f = float(np.float32(v)) if isinstance(v, (int, float, np.floating, np.integer)) and not isinstance(v, bool) \
        else math.nan
    if not test(f):
        raise ValueError(f"{what} must be {hint}, got {v!r}")
    return f


def _int(v, what, lo, hi):
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not lo <= v <= hi:
        raise ValueError(f"{what} must be an int in {lo}..{hi}, got {v!r}")
    return int(v)


class OccupancyGrid:
    """A 2-D occupancy grid of dims = (nx, ny) cells of cell_size metres; cell (i, j) is centred at
    origin + cell_size (i, j) in the grid plane.  The grid frame is world_to_grid (4x4, float64) applied to the world
    frame of the poses, with x, y horizontal and z up; the default maps KITTI's camera world frame (X right, Y down, Z
    forward) to grid x = X, grid y = Z, up = -Y.

    camera_height   metres from the camera centre down to the road; each frame's road level is the camera's grid z
                    minus it
    band            (h_lo, h_hi): a depth pixel h metres above the road is an obstacle when h_lo <= h <= h_hi, road
                    (ground) below h_lo, and ignored above h_hi (overhangs, bridges, trees)
    col_width       image columns per polar column of the free-space test (1..64)
    range_res       metres per range bin of that test
    max_depth       depths beyond it are ignored; it fixes the number of range bins
    min_hits        full-weight obstacle pixels (256 units of quantised weight each) that make a cell occupied in a
                    frame, and that end a column's free space
    l_hit, l_miss, l_min, l_max   log-odds of a hit and of a miss, and the clamping bounds: OctoMap's 0.7, 0.4, 0.12
                    and 0.97 (Hornung et al. 2013), rounded
    The default band and min_hits were chosen on a synthetic road scene; they are not tuned for KITTI."""

    def __init__(self, origin, cell_size, dims, *, world_to_grid=KITTI_WORLD_TO_GRID, camera_height=1.65,
                 band=(0.3, 2.5), col_width=5, range_res=0.1, max_depth=40.0, min_hits=10, l_hit=0.85, l_miss=-0.4,
                 l_min=-2.0, l_max=3.5, device=None):
        self.origin = tuple(float(np.float32(v)) for v in origin)
        self.dims = tuple(int(v) for v in dims)
        if len(self.origin) != 2 or len(self.dims) != 2 or not all(math.isfinite(v) for v in self.origin):
            raise ValueError(f"origin {origin!r} and dims {dims!r}: two finite coordinates and two sizes expected")
        nx, ny = self.dims
        if min(nx, ny) <= 0 or max(nx, ny) >= 2 ** 24 or nx * ny >= 2 ** 31:
            raise ValueError(f"dims {self.dims}: each in 1..2^24 - 1 and fewer than 2^31 cells in all")
        pos = (lambda f: math.isfinite(f) and f > 0, "finite and > 0")
        self.cell_size = _f32(cell_size, "cell_size", *pos)
        m = np.asarray(world_to_grid, np.float64)
        if m.shape not in ((3, 4), (4, 4)) or not np.isfinite(m).all():
            raise ValueError(f"world_to_grid: a finite [4,4] or [3,4] matrix expected, got {m.shape}")
        self.world_to_grid = np.eye(4)
        self.world_to_grid[:3] = m[:3]
        self.camera_height = _f32(camera_height, "camera_height", math.isfinite, "finite")
        if len(band) != 2:
            raise ValueError(f"band must be (h_lo, h_hi), got {band!r}")
        self.band = tuple(_f32(v, "band", math.isfinite, "finite") for v in band)
        if not self.band[0] < self.band[1]:
            raise ValueError(f"band {band!r}: h_lo < h_hi expected")
        self.col_width = _int(col_width, "col_width", 1, MAX_COL_WIDTH)
        self.range_res = _f32(range_res, "range_res", *pos)
        self.max_depth = _f32(max_depth, "max_depth", *pos)
        if nbins(self.max_depth, self.range_res) > MAX_BINS:
            raise ValueError(f"max_depth / range_res = {self.max_depth / self.range_res:.0f}: at most {MAX_BINS - 1}")
        self.min_hits = _int(min_hits, "min_hits", 1, MAX_HITS)
        self.l_hit = _f32(l_hit, "l_hit", lambda f: f > 0, "> 0")
        self.l_miss = _f32(l_miss, "l_miss", lambda f: f < 0, "< 0")
        self.l_min = _f32(l_min, "l_min", lambda f: f < 0, "< 0")
        self.l_max = _f32(l_max, "l_max", lambda f: f > 0, "> 0")
        dev = torch.device("cuda") if device is None else device
        self.log_odds = torch.empty((ny, nx), dtype=torch.float32, device=dev)
        self.updates = torch.empty((ny, nx), dtype=torch.int32, device=dev)
        self.reset()

    colour = False                           # FusePipeline passes no colours to a grid

    def reset(self):
        """log_odds = 0 (probability 0.5), updates = 0 (no host sync)."""
        self.log_odds.zero_()
        self.updates.zero_()
        return self

    @property
    def nbytes(self):
        return self.log_odds.numel() * 8

    def integrate(self, depth, calib, cam_to_world, *, weight=None, rgb=None, window=None, max_depth=None):
        """Add B depth maps in order, without a host sync.

        depth         fp32 [B,h,w] or [B,1,h,w] metric depth, 0 (or non-finite) = no depth: PointCloud.depth of
                      geometry.reproject
        calib         the StereoCalib of the depth maps (fx, fy, cx, cy)
        cam_to_world  [B,4,4] or [B,3,4] float64 on the host: the pose of the camera the depth maps are in; composed
                      with world_to_grid and inverted in float64, stored float32
        weight        fp32 map shaped like depth (e.g. the window of Confidence.peak), clamped to [0, 1], NaN = 0;
                      None = 1.  A pixel of weight 0 is not observed at all (motion masks)
        rgb           refused: a grid keeps no colour
        window        the (y0, x0, h, w, v_origin) given to reproject; None = (0, 0, h, w, 0)
        max_depth     None = the grid's max_depth; a finite value may only lower it
        Only the cells the frames can reach are visited (the same result as the whole grid).  Batches above 16
        frames are split into calls of 16, in order."""
        if rgb is not None:
            raise ValueError("an occupancy grid keeps no colour: rgb= is not used")
        depth = _bhw(depth, "depth", torch.float32)
        if depth.device != self.log_odds.device:
            raise ValueError(f"depth on {depth.device}, the grid on {self.log_odds.device}")
        B, h, w = depth.shape
        if B < 1 or h < 1 or w < 1:
            raise ValueError(f"depth {tuple(depth.shape)}: an empty batch or window")
        if weight is not None:
            weight = _bhw(weight, "weight", torch.float32)
            if weight.shape != depth.shape or weight.device != depth.device:
                raise ValueError(f"weight {tuple(weight.shape)} on {weight.device}: expected {tuple(depth.shape)} on "
                                 f"{depth.device}")
        u0, v0 = _window_origin(window, h, w)
        md = self.max_depth
        if max_depth is not None:
            md = float(np.float32(max_depth))
            if not 0 < md <= self.max_depth:
                raise ValueError(f"max_depth must be in (0, {self.max_depth}] (the grid's) or None, got {max_depth!r}")
        M = self.world_to_grid @ _poses(cam_to_world, B)
        Minv = np.linalg.inv(M)
        with np.errstate(over="ignore"):
            Mf = M[:, :3].reshape(B, 12).astype(np.float32)
            Mif = Minv[:, :3].reshape(B, 12).astype(np.float32)
        if not (np.isfinite(Mf).all() and np.isfinite(Mif).all()):
            raise ValueError("cam_to_world: the grid pose or its inverse overflows float32")
        if any(m.stride(2) != 1 for m in (depth, weight) if m is not None) or \
                (weight is not None and weight.stride() != depth.stride()):
            depth = depth.contiguous()
            weight = None if weight is None else weight.contiguous()
        intr = (calib.fx, calib.fy, calib.cx, calib.cy)
        for s in range(0, B, MAX_FRAMES):
            e = min(B, s + MAX_FRAMES)
            box = frustum_box(self.dims, self.origin, self.cell_size, intr, (u0, v0, h, w), M[s:e], md,
                              self.range_res)
            if box is None:
                continue
            _integrate_kernel(self, box, depth[s:e], None if weight is None else weight[s:e], intr, u0, v0, Mf[s:e],
                              Mif[s:e], md)
        return self

    def probability(self):
        """sigmoid(log_odds), fp32 [ny, nx] on the grid's device."""
        return torch.sigmoid(self.log_odds)

    def classes(self, occupied=0.65, free=0.2):
        """uint8 [ny, nx] on the grid's device: OCCUPIED where the probability is >= occupied, FREE where it is
        <= free, UNKNOWN elsewhere and wherever no frame updated the cell."""
        if not 0 < free < occupied < 1:
            raise ValueError(f"0 < free < occupied < 1 expected, got free={free!r}, occupied={occupied!r}")
        p = self.probability()
        seen = self.updates > 0
        out = torch.full(p.shape, UNKNOWN, dtype=torch.uint8, device=p.device)
        out[seen & (p <= free)] = FREE
        out[seen & (p >= occupied)] = OCCUPIED
        return out

    def save_map(self, stem, occupied=0.65, free=0.2):
        """Write stem.pgm and stem.yaml in ROS map_server's trinary format: 254 free, 0 occupied, 205 unknown; image row
        0 is the largest grid y; the YAML origin is the corner of cell (0, 0).  Returns the two paths."""
        c = self.classes(occupied, free).cpu().numpy()
        img = np.full(c.shape, 205, np.uint8)
        img[c == FREE] = 254
        img[c == OCCUPIED] = 0
        img = np.ascontiguousarray(img[::-1])
        stem = os.fspath(stem)
        pgm, yml = stem + ".pgm", stem + ".yaml"
        nx, ny = self.dims
        with open(pgm, "wb") as f:
            f.write(b"P5\n%d %d\n255\n" % (nx, ny))
            f.write(img.tobytes())
        half = self.cell_size / 2
        with open(yml, "w") as f:
            f.write(f"image: {os.path.basename(pgm)}\nmode: trinary\nresolution: {self.cell_size!r}\n"
                    f"origin: [{self.origin[0] - half!r}, {self.origin[1] - half!r}, 0.0]\nnegate: 0\n"
                    f"occupied_thresh: 0.65\nfree_thresh: 0.196\n")
        return pgm, yml

    def agreement(self, other, occupied=0.65, free=0.2):
        """Compare with another grid of the same geometry over the cells known in both -> Agreement (synchronises)."""
        if not isinstance(other, OccupancyGrid) or (other.origin, other.cell_size, other.dims) != \
                (self.origin, self.cell_size, self.dims) or not np.array_equal(other.world_to_grid, self.world_to_grid):
            raise ValueError("agreement needs an OccupancyGrid of the same origin, cell_size, dims and world_to_grid")
        a = self.classes(occupied, free)
        b = other.classes(occupied, free).to(a.device)
        known = (a != UNKNOWN) & (b != UNKNOWN)
        n = [int(v) for v in torch.stack([known.sum(), (known & (a == b)).sum(),
                                          (known & (a == OCCUPIED) & (b == OCCUPIED)).sum(),
                                          (known & ((a == OCCUPIED) | (b == OCCUPIED))).sum(),
                                          (known & (a == FREE) & (b == FREE)).sum(),
                                          (known & ((a == FREE) | (b == FREE))).sum()]).cpu()]

        def ratio(x, y):
            return x / y if y else math.nan
        return Agreement(*n, ratio(n[2], n[3]), ratio(n[4], n[5]), ratio(n[1], n[0]))
