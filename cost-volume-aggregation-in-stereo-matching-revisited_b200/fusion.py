"""TSDF fusion of posed depth maps into a dense voxel volume on the GPU, and the oriented, coloured surface of the fused
volume (include/dca_b200.h section 12).

  TSDFVolume         the planar fp32 state (tsdf, weight and optionally r, g, b) of an nx x ny x nz grid on a device;
                     .integrate(depth, calib, cam_to_world, weight=, rgb=, window=, max_depth=) runs one
                     dca_tsdf_integrate per 16 frames (one launch, no host sync) on the voxel box that can see them;
                     .extract() -> SurfacePoints(xyz, normal, rgb): the zero crossings of the tsdf between neighbouring
                     voxels, in voxel order (count, one sync to read the total, then the ordered scatter)
                     .raycast(cam_to_world, calib, shape, window=) -> Rendered(depth, vertex, normal, rgb): the fused
                     surface seen from any pose (dca_tsdf_raycast, one launch, no host sync)
  read_kitti_poses   KITTI odometry poses.txt -> camera-to-world [N, 4, 4] float64 (camera 0, or with the sequence's
                     calib.txt the rectified left colour camera the depth maps live in); save_kitti_poses writes them back
  fuse_files         stereo pairs on disk + poses -> one fused volume: ReprojectPipeline with the forward, reproject and
                     integrate on the compute stream, pair after pair in input order
"""
import math
from typing import NamedTuple

import numpy as np
import torch

from . import _lib, engine
from .geometry import ReprojectPipeline, _floats, _read_kv, reproject, save_ply

MAX_FRAMES = 16                # DCA_TSDF_MAX_FRAMES: frames per dca_tsdf_integrate call
TILE = 1024                    # DCA_TSDF_TILE: voxels per tile of the extraction workspace


class SurfacePoints(NamedTuple):
    """Device tensors of one extraction: xyz fp32 [n,3] (world metres), normal fp32 [n,3] unit (or zero) vectors from
    behind the surface towards the cameras, or None; rgb uint8 [n,3] or None."""
    xyz: torch.Tensor
    normal: torch.Tensor
    rgb: torch.Tensor

    def numpy(self):
        """(xyz, normal or None, rgb or None) on the host."""
        return tuple(None if t is None else t.cpu().numpy() for t in self)


def _integrate_kernel(vol, box, depth, weight, rgb, intrinsics, u0, v0, T, max_depth):
    """One dca_tsdf_integrate of B <= 16 frames: depth (and weight) fp32 [B,h,w] sharing one layout (unit column
    stride), rgb uint8 [B,h,w,3|4] (unit channel stride, packed pixels) or None, T float32 [B,12] world-to-camera."""
    engine._require_cuda(vol.state, depth, weight, rgb)
    B, H, W = depth.shape
    pitch_row = depth.stride(1)
    pitch_img = depth.stride(0) if B > 1 else H * pitch_row
    C = c_row = c_img = 0
    if rgb is not None:
        C, c_row = rgb.shape[3], rgb.stride(1)
        c_img = rgb.stride(0) if B > 1 else H * c_row
    t = np.ascontiguousarray(T, np.float32)
    nx, ny, nz = vol.dims
    _lib.call("dca_tsdf_integrate", vol.state.data_ptr(), vol.planes, nx, ny, nz, *vol.origin, vol.voxel_size, *box,
              depth.data_ptr(), 0 if weight is None else weight.data_ptr(), pitch_row, pitch_img, B, H, W,
              0 if rgb is None else rgb.data_ptr(), C, c_row, c_img, *intrinsics, u0, v0, t.ctypes.data, vol.trunc,
              vol.max_weight, max_depth, torch.cuda.current_stream(vol.state.device).cuda_stream)


class Rendered(NamedTuple):
    """Device maps of one raycast, [h, w] of the window: depth fp32 (camera Z, 0 = no hit, as PointCloud.depth), vertex
    fp32 [h,w,3] in the camera frame (NaN = no hit), normal fp32 [h,w,3] unit vectors in the camera frame pointing
    towards the camera (NaN = no hit), rgb uint8 [h,w,3] or None (a volume without colour)."""
    depth: torch.Tensor
    vertex: torch.Tensor
    normal: torch.Tensor
    rgb: torch.Tensor


def _raycast_kernel(vol, intrinsics, u0, v0, M, min_weight, min_depth, max_depth, out):
    """One dca_tsdf_raycast into the Rendered `out` (contiguous maps of one window); M float32 [12] camera-to-world."""
    engine._require_cuda(vol.state, *out)
    h, w = out.depth.shape
    nx, ny, nz = vol.dims
    m = np.ascontiguousarray(M, np.float32)
    _lib.call("dca_tsdf_raycast", vol.state.data_ptr(), vol.planes, nx, ny, nz, *vol.origin, vol.voxel_size, vol.trunc,
              float(min_weight), *intrinsics, u0, v0, h, w, m.ctypes.data, float(min_depth), float(max_depth),
              out.depth.data_ptr(), w, out.vertex.data_ptr(), 3 * w, out.normal.data_ptr(), 3 * w,
              0 if out.rgb is None else out.rgb.data_ptr(), 3 * w, torch.cuda.current_stream(vol.state.device).cuda_stream)


def _extract_kernel(vol, min_weight, normals, colours):
    """dca_tsdf_count_surface, one host sync to read the total, then dca_tsdf_extract_surface into exactly that many
    rows -> SurfacePoints."""
    engine._require_cuda(vol.state)
    dev = vol.state.device
    nx, ny, nz = vol.dims
    st = torch.cuda.current_stream(dev).cuda_stream
    ws = torch.empty(((nx * ny * nz + TILE - 1) // TILE,), dtype=torch.int64, device=dev)
    count = torch.empty((1,), dtype=torch.int64, device=dev)
    _lib.call("dca_tsdf_count_surface", vol.state.data_ptr(), vol.planes, nx, ny, nz, float(min_weight), ws.data_ptr(),
              count.data_ptr(), st)
    n = int(count[0])
    xyz = torch.empty((n, 3), dtype=torch.float32, device=dev)
    normal = torch.empty((n, 3), dtype=torch.float32, device=dev) if normals else None
    rgb = torch.empty((n, 3), dtype=torch.uint8, device=dev) if colours else None
    if n:
        _lib.call("dca_tsdf_extract_surface", vol.state.data_ptr(), vol.planes, nx, ny, nz, *vol.origin, vol.voxel_size,
                  float(min_weight), ws.data_ptr(), n, xyz.data_ptr(), 0 if normal is None else normal.data_ptr(),
                  0 if rgb is None else rgb.data_ptr(), st)
    return SurfacePoints(xyz, normal, rgb)


def _poses(cam_to_world, B=None):
    """[B,4,4] or [B,3,4] (or one [4,4] / [3,4]) -> float64 [B,4,4]."""
    m = np.asarray(cam_to_world, np.float64)
    if m.ndim == 2:
        m = m[None]
    if m.ndim != 3 or m.shape[1:] not in ((3, 4), (4, 4)) or (B is not None and m.shape[0] != B):
        raise ValueError(f"cam_to_world: expected [{B if B is not None else 'B'},4,4] or [.,3,4], got {m.shape}")
    if not np.isfinite(m).all():
        raise ValueError("cam_to_world is not finite")
    out = np.tile(np.eye(4), (m.shape[0], 1, 1))
    out[:, :3] = m[:, :3]
    return out


def frustum_box(dims, origin, voxel_size, intrinsics, window, cam_to_world, max_depth, trunc):
    """The voxel box (i0, j0, k0, bi, bj, bk) that holds every voxel the frames can update, or None when no voxel can:
    the float64 AABB of the camera centres and of the window corners (pixel edges, +-0.5 px) at Z = max_depth + trunc,
    grown by one voxel and clipped to the grid.  window = (u0, v0, h, w) in image pixels.  The whole grid when that
    AABB is not finite (max_depth = inf, or so large that the corners overflow)."""
    fx, fy, cx, cy = intrinsics
    u0, v0, h, w = window
    whole = (0, 0, 0) + tuple(int(v) for v in dims)
    Z = float(max_depth) + float(trunc)
    if not math.isfinite(Z):
        return whole
    pts = [(0.0, 0.0, 0.0)]
    for u in (u0 - 0.5, u0 + w - 0.5):
        for v in (v0 - 0.5, v0 + h - 0.5):
            pts.append(((u - cx) / fx * Z, (v - cy) / fy * Z, Z))
    pts = np.array(pts, np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        world = np.einsum("bij,nj->bni", cam_to_world[:, :3, :3], pts) + cam_to_world[:, None, :3, 3]
    if not np.isfinite(world).all():
        return whole
    lo, hi = world.reshape(-1, 3).min(0), world.reshape(-1, 3).max(0)
    o, n = np.asarray(origin, np.float64), np.asarray(dims)
    with np.errstate(over="ignore"):
        a = np.maximum(np.floor((lo - o) / voxel_size) - 1, 0)
        b = np.minimum(np.ceil((hi - o) / voxel_size) + 1, n - 1)
    if (a > b).any():
        return None
    a, b = a.astype(int), b.astype(int)
    return tuple(int(x) for x in a) + tuple(int(x) for x in b - a + 1)


class TSDFVolume:
    """A dense TSDF volume of dims = (nx, ny, nz) voxels of voxel_size metres; voxel (i, j, k) is centred at
    origin + voxel_size (i, j, k) in the world frame.  state = fp32 [planes, nz, ny, nx] on `device`: tsdf (starts at 1),
    weight (starts at 0) and, with colour=True, r, g, b (start at 0).  trunc = the truncation distance in metres (3
    voxels by default); max_weight caps the weight of a voxel (inf = a plain running average)."""

    def __init__(self, origin, voxel_size, dims, trunc=None, colour=True, device=None, max_weight=math.inf):
        self.origin = tuple(float(np.float32(v)) for v in origin)
        self.voxel_size = float(np.float32(voxel_size))
        self.dims = tuple(int(v) for v in dims)
        if len(self.origin) != 3 or len(self.dims) != 3 or not all(math.isfinite(v) for v in self.origin):
            raise ValueError(f"origin {origin!r} and dims {dims!r}: three finite coordinates and three sizes expected")
        if not (math.isfinite(self.voxel_size) and self.voxel_size > 0):
            raise ValueError(f"voxel_size must be finite and > 0, got {voxel_size!r}")
        if min(self.dims) <= 0 or math.prod(self.dims) >= 2 ** 31:
            raise ValueError(f"dims {self.dims}: each > 0 and fewer than 2^31 voxels in all")
        self.trunc = float(np.float32(3 * self.voxel_size if trunc is None else trunc))
        if not (math.isfinite(self.trunc) and self.trunc > 0):
            raise ValueError(f"trunc must be finite and > 0, got {trunc!r}")
        self.max_weight = float(np.float32(max_weight))
        if not self.max_weight > 0:
            raise ValueError(f"max_weight must be > 0, got {max_weight!r}")
        self.colour = bool(colour)
        self.planes = 5 if self.colour else 2
        nx, ny, nz = self.dims
        self.state = torch.empty((self.planes, nz, ny, nx), dtype=torch.float32,
                                 device=torch.device("cuda") if device is None else device)
        self.reset()

    def reset(self):
        """tsdf = 1, weight = colour = 0 (no host sync)."""
        self.state[0].fill_(1.0)
        self.state[1:].zero_()
        return self

    @property
    def nbytes(self):
        return self.state.numel() * 4

    @property
    def tsdf(self):
        return self.state[0]

    @property
    def weight(self):
        return self.state[1]

    def integrate(self, depth, calib, cam_to_world, *, weight=None, rgb=None, window=None, max_depth=None):
        """Fuse B depth maps in order, without a host sync.

        depth         fp32 [B,h,w] or [B,1,h,w] metric depth, 0 (or non-finite) = no depth: PointCloud.depth of
                      geometry.reproject
        calib         the StereoCalib of the depth maps (fx, fy, cx, cy)
        cam_to_world  [B,4,4] or [B,3,4] float64 on the host: the pose of the camera the depth maps are in; inverted in
                      float64 and stored float32
        weight        fp32 map shaped like depth (e.g. the window of Confidence.peak), clamped to [0, 1], NaN = 0;
                      None = 1
        rgb           uint8 [B,h,w,3|4] (or [h,w,3|4] when B = 1) colours of the depth pixels; required by a volume
                      with colour, refused by one without
        window        the (y0, x0, h, w, v_origin) given to reproject: depth pixel (x, y) is image pixel
                      (x0 + x, v_origin + y); h and w must be the depth map's.  None = (0, 0, h, w, 0)
        max_depth     depths beyond it are ignored, and only the voxel box the frames can reach within max_depth + trunc
                      is visited (same result as the whole grid); None or inf = no limit, the whole grid
        Batches above 16 frames are split into calls of 16, in order."""
        depth = _bhw(depth, "depth", torch.float32)
        if depth.device != self.state.device:
            raise ValueError(f"depth on {depth.device}, the volume on {self.state.device}")
        B, h, w = depth.shape
        if weight is not None:
            weight = _bhw(weight, "weight", torch.float32)
            if weight.shape != depth.shape or weight.device != depth.device:
                raise ValueError(f"weight {tuple(weight.shape)} on {weight.device}: expected {tuple(depth.shape)} on "
                                 f"{depth.device}")
        if self.colour and rgb is None:
            raise ValueError("this volume keeps colour: pass rgb=, or build it with colour=False")
        if not self.colour and rgb is not None:
            raise ValueError("this volume keeps no colour (colour=False): rgb= is not used")
        if rgb is not None:
            if not torch.is_tensor(rgb):
                raise ValueError(f"rgb: expected a torch tensor, got {type(rgb).__name__}")
            if rgb.dim() == 3 and B == 1:
                rgb = rgb[None]
            if rgb.dim() != 4 or rgb.dtype != torch.uint8 or tuple(rgb.shape[:3]) != (B, h, w) \
                    or rgb.shape[3] not in (3, 4) or rgb.device != depth.device:
                raise ValueError(f"rgb: expected uint8 [{B},{h},{w},3|4] on {depth.device}, got {rgb.dtype} "
                                 f"{tuple(rgb.shape)} on {rgb.device}")
            if rgb.stride(3) != 1 or rgb.stride(2) != rgb.shape[3]:
                rgb = rgb.contiguous()
        u0, v0 = _window_origin(window, h, w)
        if max_depth is not None and not max_depth > 0:
            raise ValueError(f"max_depth must be > 0 (inf = no limit) or None, got {max_depth!r}")
        c2w = _poses(cam_to_world, B)
        T = np.linalg.inv(c2w)[:, :3].reshape(B, 12).astype(np.float32)
        if any(m.stride(2) != 1 for m in (depth, weight) if m is not None) or \
                (weight is not None and weight.stride() != depth.stride()):
            depth = depth.contiguous()
            weight = None if weight is None else weight.contiguous()
        intr = (calib.fx, calib.fy, calib.cx, calib.cy)
        md = math.inf if max_depth is None else float(max_depth)
        for s in range(0, B, MAX_FRAMES):
            e = min(B, s + MAX_FRAMES)
            if math.isinf(md):
                box = (0, 0, 0) + self.dims
            else:
                box = frustum_box(self.dims, self.origin, self.voxel_size, intr, (u0, v0, h, w), c2w[s:e], md,
                                  self.trunc)
                if box is None:
                    continue
            _integrate_kernel(self, box, depth[s:e], None if weight is None else weight[s:e],
                              None if rgb is None else rgb[s:e], intr, u0, v0, T[s:e], md)
        return self

    def raycast(self, cam_to_world, calib, shape, window=None, min_weight=0.5, min_depth=0.0, max_depth=40.0):
        """Render the fused surface from one pose, without a host sync -> Rendered on the volume's device.

        cam_to_world  [4,4] or [3,4] float64 on the host, stored float32
        calib         the StereoCalib of the rendered camera (fx, fy, cx, cy)
        shape         (h, w) of the window
        window        the (y0, x0, h, w, v_origin) of reproject: rendered pixel (x, y) is image pixel (x0 + x,
                      v_origin + y); None = (0, 0, h, w, 0)
        min_weight    a march sample whose 8 voxels do not all reach it is unknown (skipped, never a hit)
        min_depth, max_depth   the march along camera Z; max_depth must be finite, the ray marches to it
        The first crossing from positive to negative tsdf is the hit (include/dca_b200.h section 13).
        save_depth_png writes Rendered.depth."""
        h, w = (int(v) for v in shape)
        if h <= 0 or w <= 0:
            raise ValueError(f"shape {tuple(shape)}: two sizes > 0 expected")
        u0, v0 = _window_origin(window, h, w)
        if not min_weight == min_weight:
            raise ValueError("min_weight is NaN")
        if not (math.isfinite(max_depth) and 0 <= min_depth <= max_depth):
            raise ValueError(f"min_depth {min_depth!r}, max_depth {max_depth!r}: 0 <= min_depth <= max_depth, finite")
        M = _poses(cam_to_world, 1)[0, :3].reshape(12).astype(np.float32)
        out = self._maps(h, w)
        _raycast_kernel(self, (calib.fx, calib.fy, calib.cx, calib.cy), u0, v0, M, min_weight, min_depth, max_depth,
                        out)
        return out

    def _maps(self, h, w):
        dev = self.state.device
        return Rendered(torch.empty((h, w), dtype=torch.float32, device=dev),
                        torch.empty((h, w, 3), dtype=torch.float32, device=dev),
                        torch.empty((h, w, 3), dtype=torch.float32, device=dev),
                        torch.empty((h, w, 3), dtype=torch.uint8, device=dev) if self.colour else None)

    def extract(self, min_weight=0.5, normals=True, colours=None):
        """The surface points: crossings of the tsdf's sign between neighbouring voxels whose weights are both
        >= min_weight, ordered by voxel then axis -> SurfacePoints on the volume's device.  colours None = when the
        volume has colour.  Synchronises once (to size the outputs)."""
        if not min_weight == min_weight:
            raise ValueError("min_weight is NaN")
        colours = self.colour if colours is None else bool(colours)
        if colours and not self.colour:
            raise ValueError("colours=True on a volume without colour")
        return _extract_kernel(self, min_weight, bool(normals), colours)

    def save_ply(self, path, min_weight=0.5, normals=True):
        """extract() written as a binary PLY (x y z [nx ny nz] [red green blue]); returns the SurfacePoints."""
        s = self.extract(min_weight, normals)
        xyz, nrm, rgb = s.numpy()
        save_ply(path, xyz, rgb, normal=nrm)
        return s


def _window_origin(window, h, w):
    """reproject's window (y0, x0, h, w, v_origin) of an h x w map -> (u0, v0), the image pixel of map pixel (0, 0)."""
    if window is None:
        return 0, 0
    _, x0, wh, ww, v_origin = (int(v) for v in window)
    if (wh, ww) != (h, w):
        raise ValueError(f"window {tuple(window)}: its size is not the {h}x{w} of the depth map")
    return x0, v_origin


def _bhw(t, what, dtype):
    if not torch.is_tensor(t):
        raise ValueError(f"{what}: expected a torch tensor, got {type(t).__name__}")
    if t.dim() == 4 and t.shape[1] == 1:
        t = t[:, 0]
    if t.dim() != 3 or t.dtype != dtype:
        raise ValueError(f"{what}: expected {dtype} [B,H,W] or [B,1,H,W], got {t.dtype} {tuple(t.shape)}")
    return t


# ---- poses -------------------------------------------------------------------------------------------------------
def read_kitti_poses(poses_txt, calib_path=None):
    """KITTI odometry poses.txt (12 floats per line: the 3x4 pose of camera 0 in the world = camera 0 of the first frame)
    -> float64 [N,4,4] camera-to-world.  With the sequence's calib.txt the poses are of the rectified left colour camera
    (camera 2), the frame of the depth maps of geometry.reproject: each pose is composed with camera 2's offset
    (-P2[0,3] / fx, -P2[1,3] / fy, 0), the same shift read_kitti_calib uses for rect_to_velo."""
    rows = []
    with open(poses_txt) as f:
        for n, line in enumerate(f, 1):
            if line.strip():
                v = np.array([float(x) for x in line.split()], np.float64)
                if v.size != 12:
                    raise ValueError(f"{poses_txt}:{n}: 12 numbers expected, got {v.size}")
                rows.append(v)
    out = np.tile(np.eye(4), (len(rows), 1, 1))
    if rows:
        out[:, :3] = np.stack(rows).reshape(-1, 3, 4)
    if calib_path is not None:
        out = out @ _camera2_shift(calib_path)
    return out


def _camera2_shift(calib_path):
    """[4,4] pose of camera 2 in camera 0 from a KITTI calib.txt: the translation (-P2[0,3] / fx, -P2[1,3] / fy, 0)."""
    kv = _read_kv(calib_path, ":")
    key = "P2" if "P2" in kv else "P_rect_02"
    if key not in kv:
        raise ValueError(f"{calib_path}: no P2 (or P_rect_02) projection matrix")
    P2 = _floats(kv[key]).reshape(3, 4)
    shift = np.eye(4)
    shift[:3, 3] = (-P2[0, 3] / P2[0, 0], -P2[1, 3] / P2[1, 1], 0.0)
    return shift


def save_kitti_poses(path, cam_to_world, calib_path=None):
    """The inverse of read_kitti_poses: camera-to-world [N,4,4] or [N,3,4] float64 -> a KITTI odometry poses.txt (12
    numbers per line, %.17g, so read_kitti_poses gives the poses back exactly).  With the sequence's calib.txt the poses
    are of camera 2 (those of read_kitti_poses with that file, of TSDFVolume.integrate and of track_files) and camera 2's
    offset is removed again, so the file holds camera 0 as the KITTI odometry devkit expects."""
    m = _poses(cam_to_world)
    if calib_path is not None:
        m = m @ np.linalg.inv(_camera2_shift(calib_path))
    with open(path, "w") as f:
        for p in m:
            f.write(" ".join("%.17g" % v for v in p[:3].ravel()) + "\n")


# ---- files in, one fused volume out ---------------------------------------------------------------------------------
class FusePipeline(ReprojectPipeline):
    """ReprojectPipeline whose compute stream runs, pair after pair in input order, the forward (with confidence when
    the weights or a filter need it, with the left-right check when asked), reproject on the window that undoes the
    framing (with the filters) and TSDFVolume.integrate of the depth map with the pair's pose, the window of
    Confidence.peak as weights (weight="peak") and the left image of the window as colours.  Nothing comes back to the
    host per pair."""

    def __init__(self, model, calibs, volume, mode="fit", crop_height=384, crop_width=1248, min_confidence=None,
                 lr_check=False, lr_threshold=1.0, min_depth=0.0, max_depth=None, weight="peak", depth=3, workers=2,
                 rectifier=None, motion=None):
        if weight not in ("peak", None):
            raise ValueError(f"weight must be 'peak' or None, got {weight!r}")
        from .motion import _options
        self.motion = _options(motion)
        self._reference = None                                   # (depth, calib values, window, pose) last integrated
        # the rectifier is set up here rather than by ReprojectPipeline, whose per-slot point-cloud and colour
        # read-back buffers fusion does not use
        super().__init__(model, calibs, mode, crop_height, crop_width, min_confidence, lr_check, lr_threshold,
                         "camera", min_depth, math.inf if max_depth is None else max_depth, depth, workers, None)
        self.volume, self.weight, self.fuse_max_depth = volume, weight, max_depth
        self.rgb_host = [None] * self.depth
        self.rgb_dev = [None] * self.depth
        if rectifier is not None:
            from .rectify import RawSlots, framing
            W, H = rectifier.rect_size
            framing(H, W, mode, (crop_height, crop_width))       # a rectified size the crop cannot frame raises here
            self.rectifier = rectifier
            self.in_host = self.in_dev = None                    # the fp32 input slots are not used
            self.raw = RawSlots(self, rectifier)

    def _ensure_input(self, slot, Hn, Wn):
        if tuple(self.in_host[slot].shape) != (6, Hn, Wn):
            self.in_host[slot] = self._host((6, Hn, Wn), torch.float32)
            self.in_dev[slot] = torch.empty((6, Hn, Wn), dtype=torch.float32, device=self.dev) if self.cuda \
                else self.in_host[slot]

    def _put_rgb(self, slot, rgb):
        if self.rgb_host[slot] is None or tuple(self.rgb_host[slot].shape) != rgb.shape:
            self.rgb_host[slot] = self._host(rgb.shape, torch.uint8)
            self.rgb_dev[slot] = torch.empty(rgb.shape, dtype=torch.uint8, device=self.dev) if self.cuda \
                else self.rgb_host[slot]
        np.copyto(self.rgb_host[slot].numpy(), rgb)

    def _observe(self, slot, calib, window):
        """The forward and reproject of the pair in `slot` -> (depth, weight map or None, colours, window)."""
        if self.rectifier is not None:
            from .rectify import rectify
            raw = self.raw.dev[slot]
            x = rectify(raw[0:1], raw[1:2], self.rectifier, self.mode, (self.ch, self.cw))
            left, right, window = x.left, x.right, x.window
            y0, x0, h, w, vo = window
            rgb = x.rgb[:, 0, vo:vo + h, x0:x0 + w]
        else:
            x = self.in_dev[slot]
            left, right, rgb = x[None, 0:3], x[None, 3:6], self.rgb_dev[slot][None]
        conf = self.min_confidence is not None or self.weight == "peak"
        kw = {}
        if conf:
            kw["confidence"] = True
        if self.lr_check:
            kw.update(lr_check=True, lr_threshold=self.lr_threshold)
        out = self.model(left, right, **kw)
        pred = out[0] if isinstance(out, (tuple, list)) else out
        filt = self.min_confidence is not None
        pc = reproject(pred, calib, confidence=out[2].peak if filt else None,
                       min_confidence=self.min_confidence if filt else 0.0,
                       label=out[-1].label if self.lr_check else None, min_depth=self.min_depth,
                       max_depth=self.max_depth, window=window)
        wmap = None
        if self.weight == "peak":
            y0, x0, h, w, _ = window
            wmap = out[2].peak[:, 0, y0:y0 + h, x0:x0 + w]
        return pc.depth, wmap, rgb, window

    def _integrate(self, obs, calib, pose):
        depth, wmap, rgb, window = obs
        if self.motion is not None:
            wmap = self._mask_moving(depth, wmap, calib, window, pose)
        self.volume.integrate(depth, calib, pose, weight=wmap, rgb=rgb if self.volume.colour else None,
                              window=window, max_depth=self.fuse_max_depth)

    def _mask_moving(self, depth, wmap, calib, window, pose):
        """With motion= set: the weight map of a frame with its moving objects' pixels at 0, tested against the last
        frame integrated (motion.motion with T(previous <- current) from the two integration poses).  A frame without
        such a reference (the first, or one whose window or calibration differs) keeps its weights."""
        from .motion import motion as moving
        key = (calib.fx, calib.fy, calib.cx, calib.cy, calib.baseline, calib.doffs)
        win = None if window is None else tuple(int(v) for v in window)
        ref, self._reference = self._reference, (depth, key, win, pose)
        if ref is None or ref[0].shape != depth.shape or ref[1] != key or ref[2] != win:
            return wmap
        m = moving(depth, ref[0], calib, np.linalg.solve(ref[3], pose), window=window, **self.motion)
        still = m.instance == 0
        return still.to(torch.float32) if wmap is None else torch.where(still, wmap, torch.zeros((), device=wmap.device))

    def _fuse(self, slot, calib, window, pose):
        """The device work of one pair, on the compute stream; returns what _finish needs (None here)."""
        self._integrate(self._observe(slot, calib, window), calib, pose)

    def _finish(self, pending):
        """The host step of a pair whose _fuse returned `pending`, run after the next pair's copy is queued (nothing
        here)."""

    def run(self, items, poses):
        """items: (left, right) file pairs; poses: camera-to-world [N,4,4] or [N,3,4] aligned with them.  Returns the
        volume."""
        from concurrent.futures import ThreadPoolExecutor
        items = list(items)
        poses = _poses(poses, len(items))
        calibs = self.calibs if self.calibs is not None else getattr(self.rectifier, "calib", None)
        calibs = calibs if isinstance(calibs, (list, tuple)) else [calibs] * len(items)
        if len(calibs) != len(items):
            raise ValueError(f"{len(calibs)} calibrations for {len(items)} items")
        raw = self.rectifier is not None
        was_training = getattr(self.model, "training", False)
        if hasattr(self.model, "eval"):
            self.model.eval()
        try:
            with ThreadPoolExecutor(self.workers) as pool, torch.no_grad():
                load = self.raw.load if raw else self._load_item
                futs = [pool.submit(load, it[0], it[1]) for it in items]
                pending = None                                   # (slot, what _fuse returned) of the previous pair
                for i, fut in enumerate(futs):
                    got = fut.result()
                    slot = i % self.depth
                    if pending is not None and pending[0] == slot:
                        self._close(pending)                     # one slot: the pair in it is finished first
                        pending = None
                    if self.cuda and i >= self.depth:
                        self.free[slot].synchronize()            # the slot's previous pair is fused: its buffers are free
                    window = None
                    if raw:
                        self.raw.put(slot, got)
                    else:
                        fitted, rgb, window = got
                        self._ensure_input(slot, fitted.shape[1], fitted.shape[2])
                        np.copyto(self.in_host[slot].numpy(), fitted)
                        self._put_rgb(slot, rgb)
                    if self.cuda:
                        with torch.cuda.stream(self.copy_stream):
                            if i >= self.depth:
                                self.copy_stream.wait_event(self.free[slot])     # kernels of the slot's previous pair
                            if raw:
                                self.raw.h2d(slot)
                            else:
                                self.in_dev[slot].copy_(self.in_host[slot], non_blocking=True)
                                self.rgb_dev[slot].copy_(self.rgb_host[slot], non_blocking=True)
                            self.h2d[slot].record(self.copy_stream)
                        if pending is not None:
                            self._close(pending)                 # after pair i's copy is queued
                        with torch.cuda.stream(self.compute_stream):
                            self.compute_stream.wait_event(self.h2d[slot])
                            pending = (slot, self._fuse(slot, calibs[i], window, poses[i]))
                    else:
                        if pending is not None:
                            self._close(pending)
                        pending = (slot, self._fuse(slot, calibs[i], window, poses[i]))
                if pending is not None:
                    self._close(pending)
            if self.cuda:
                torch.cuda.current_stream(self.dev).wait_stream(self.compute_stream)
        finally:
            if was_training and hasattr(self.model, "train"):
                self.model.train()
        return self.volume

    def _close(self, pending):
        slot, state = pending
        if self.cuda:
            with torch.cuda.stream(self.compute_stream):
                self._finish(state)
                self.free[slot].record(self.compute_stream)
        else:
            self._finish(state)


def fuse_files(model, items, poses, volume, calib=None, rectifier=None, mode="fit", crop=(384, 1248),
               min_confidence=None, lr_check=False, max_depth=None, weight="peak", ply=None, min_weight=0.5,
               lr_threshold=1.0, min_depth=0.0, depth=3, workers=2, motion=None):
    """Stereo pairs on disk and their poses -> the fused TSDFVolume (or the filled OccupancyGrid).

    items      (left, right) file pairs, fused in this order
    poses      camera-to-world [N,4,4] or [N,3,4] float64 of the rectified left camera (read_kitti_poses with the
               sequence's calib.txt for KITTI odometry)
    volume     a TSDFVolume, or an occupancy.OccupancyGrid, on the model's device (fused into, not reset); a grid takes
               no colours, and max_depth may not exceed the grid's
    calib      one StereoCalib or a list aligned with items; with a rectifier (rectify.StereoRectifier) the items are
               RAW pairs, rectified on the device, and calib defaults to rectifier.calib
    min_confidence, lr_check   the filters of reproject (the forward runs with confidence / the left-right check)
    max_depth  depths beyond it are dropped, and integration visits only the voxels the frustum can reach
    weight     "peak" = each depth weighted by Confidence.peak of its pixel; None = unit weights
    ply        a path: the extracted surface (min_weight, with normals and, when the volume has colour, colours); a
               TSDFVolume only (an OccupancyGrid writes its map with save_map)
    motion     None (default) = every frame fused as it is; True or a dict of motion.motion's options (tau, tau_rel,
               radius, gate, min_pixels) = each frame is tested against the last frame integrated, at the two
               integration poses, and the pixels of its moving objects get weight 0.  The first frame has no
               reference and is fused as it is
    The colours are the left image of the window (the rectified left image with a rectifier)."""
    if calib is None and rectifier is None:
        raise ValueError("fuse_files needs a calibration (calib=) or a rectifier (rectifier=)")
    if ply is not None and not isinstance(volume, TSDFVolume):
        raise ValueError("ply= writes the surface of a TSDFVolume; an OccupancyGrid writes its map with save_map")
    pipe = FusePipeline(model, calib, volume, mode, crop[0], crop[1], min_confidence, lr_check, lr_threshold,
                        min_depth, max_depth, weight, depth, workers, rectifier, motion)
    pipe.run(items, poses)
    if ply is not None:
        volume.save_ply(ply, min_weight)
    return volume
