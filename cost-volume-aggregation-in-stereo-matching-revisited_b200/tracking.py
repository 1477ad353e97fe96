"""Camera tracking against a fused TSDF volume on the GPU (include/dca_b200.h section 13), so sequences without poses can
be fused: the tracking half of KinectFusion (Newcombe et al., ISMAR 2011).

  Tracker        raycasts the volume at its reference pose (model vertex and normal maps) and aligns a new depth map to
                 them by projective point-to-plane ICP (dca_icp_track: every iteration of a frame in one call, 2 launches
                 per iteration); .track(depth, weight=, init=) -> TrackResult(cam_to_world, ok, inliers, rms)
  track_files    stereo pairs on disk -> Trajectory(poses, ok) and the fused volume: FusePipeline with forward ->
                 reproject -> track -> integrate at the tracked pose, pair after pair
"""
import ctypes
import math
from typing import NamedTuple

import numpy as np
import torch

from . import _lib, engine, fusion
from .fusion import FusePipeline, _bhw, _poses, _window_origin

LEVELS = ((4, 10, 0.4), (2, 5, 0.2), (1, 4, 0.1))   # (pixel stride, iterations, distance gate in metres) per level
MAX_LEVELS = 4                                      # DCA_ICP_MAX_LEVELS
MAX_ITERS = 64                                      # DCA_ICP_MAX_ITERS
MAX_DEPTH = 256.0                                   # DCA_ICP_MAX_DEPTH
MAX_GATE = 16.0                                     # DCA_ICP_MAX_GATE
MAX_PIXELS = 1 << 24                                # DCA_ICP_MAX_PIXELS
TILE, WORKSPACE_ROW = 1024, 32                      # DCA_ICP_TILE, DCA_ICP_WORKSPACE_ROW


def workspace_bytes(h, w):
    """DCA_ICP_WORKSPACE_BYTES(h, w)."""
    return 8 * WORKSPACE_ROW * ((h * w + TILE - 1) // TILE)


class TrackResult(NamedTuple):
    """cam_to_world float64 [4,4] (the prediction when not ok); ok: no ICP iteration failed; inliers int64 [iterations]
    and rms float64 [iterations] (metres, NaN without inliers): the point-to-plane residual of each iteration before its
    update."""
    cam_to_world: np.ndarray
    ok: bool
    inliers: np.ndarray
    rms: np.ndarray


class Trajectory(NamedTuple):
    """poses float64 [N,4,4] camera-to-world of the rectified left camera; ok bool [N] (frame 0: True)."""
    poses: np.ndarray
    ok: np.ndarray


def _icp_kernel(depth, weight, intrinsics, u0, v0, max_depth, model, A0, levels, min_inliers, workspace, pose, stats,
                ok):
    """One dca_icp_track: depth (weight) fp32 [h,w] sharing one layout (unit column stride), model = Rendered maps of the
    window, A0 float64 [12]; pose fp64 [12], stats fp64 [iterations,4], ok int32 [1] on the device."""
    engine._require_cuda(depth, weight, model.vertex, model.normal, workspace)
    h, w = depth.shape
    a0 = np.ascontiguousarray(A0, np.float64)
    n = len(levels)
    stride = (ctypes.c_int * n)(*[lv[0] for lv in levels])
    iters = (ctypes.c_int * n)(*[lv[1] for lv in levels])
    gate = (ctypes.c_float * n)(*[lv[2] for lv in levels])
    _lib.call("dca_icp_track", depth.data_ptr(), 0 if weight is None else weight.data_ptr(), depth.stride(0), h, w,
              *intrinsics, u0, v0, float(max_depth), model.vertex.data_ptr(), 3 * w, model.normal.data_ptr(), 3 * w,
              a0.ctypes.data, n, ctypes.addressof(stride), ctypes.addressof(iters), ctypes.addressof(gate),
              int(min_inliers), workspace.data_ptr(), pose.data_ptr(), stats.data_ptr(), ok.data_ptr(),
              torch.cuda.current_stream(depth.device).cuda_stream)


def _levels(levels):
    out = []
    for lv in levels:
        s, n, g = lv
        if int(s) != s or int(n) != n:
            raise ValueError(f"level {lv!r}: stride and iterations must be integers")
        out.append((int(s), int(n), float(np.float32(g))))
    if not 1 <= len(out) <= MAX_LEVELS:
        raise ValueError(f"levels: 1 to {MAX_LEVELS} (stride, iterations, gate) expected, got {len(out)}")
    for s, n, g in out:
        if s < 1 or not 1 <= n <= MAX_ITERS or not (math.isfinite(g) and 0 < g <= MAX_GATE):
            raise ValueError(f"level {(s, n, g)}: stride >= 1, 1..{MAX_ITERS} iterations, a gate in (0, {MAX_GATE}] m")
    return tuple(out)


class Tracker:
    """Projective point-to-plane ICP of depth maps against a TSDFVolume.

    volume      the TSDFVolume the frames are tracked against (and usually fused into)
    calib       the StereoCalib of the depth maps
    shape       (h, w) of the depth maps; window = reproject's (y0, x0, h, w, v_origin) of them (None = the image)
    pose        the reference pose, camera-to-world float64: where the model is raycast.  A successful track() moves it
                to the tracked pose
    levels      (pixel stride, iterations, gate in metres) per level, coarse to fine, up to 4; strides apply to the
                full-resolution maps (no pyramid images).  The default is KinectFusion's (4, 10), (2, 5), (1, 4)
    max_depth   source depths beyond it are ignored, and the model is raycast up to it; finite, at most 256 m
    min_weight  the raycast's threshold of a known sample
    min_inliers an iteration with fewer pixels kept fails (the pose is left as it was)
    The workspace and the model maps are allocated once, on the volume's device."""

    def __init__(self, volume, calib, shape, window=None, pose=np.eye(4), levels=LEVELS, max_depth=40.0,
                 min_weight=0.5, min_inliers=100):
        self.volume, self.calib = volume, calib
        self.h, self.w = (int(v) for v in shape)
        if self.h <= 0 or self.w <= 0 or self.h * self.w > MAX_PIXELS:
            raise ValueError(f"shape {tuple(shape)}: two sizes > 0, at most {MAX_PIXELS} pixels")
        self.u0, self.v0 = _window_origin(window, self.h, self.w)
        self.levels = _levels(levels)
        if not (math.isfinite(max_depth) and 0 < max_depth <= MAX_DEPTH):
            raise ValueError(f"max_depth must be finite, in (0, {MAX_DEPTH}], got {max_depth!r}")
        if not min_weight == min_weight:
            raise ValueError("min_weight is NaN")
        if int(min_inliers) < 1:
            raise ValueError(f"min_inliers must be >= 1, got {min_inliers!r}")
        self.max_depth, self.min_weight, self.min_inliers = float(max_depth), float(min_weight), int(min_inliers)
        self.intrinsics = (calib.fx, calib.fy, calib.cx, calib.cy)
        self.iterations = sum(n for _, n, _ in self.levels)
        dev = volume.state.device
        self.model = volume._maps(self.h, self.w)
        self.workspace = torch.empty((workspace_bytes(self.h, self.w) // 8,), dtype=torch.int64, device=dev)
        # pose fp64 [12] | stats fp64 [iterations][4] | ok int32: one buffer, so one D2H copy reads them all
        nbytes = 8 * (12 + 4 * self.iterations) + 8
        self._out = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        self._cuda = dev.type == "cuda"
        self._host = torch.empty((nbytes,), dtype=torch.uint8, pin_memory=self._cuda)
        self._done = torch.cuda.Event() if self._cuda else None
        self.pose = pose

    @property
    def pose(self):
        return self._pose

    @pose.setter
    def pose(self, cam_to_world):
        """Setting the reference pose also restarts the constant-velocity prediction from it."""
        self._pose = _poses(cam_to_world, 1)[0]
        self._accepted = [self._pose]

    def predict(self):
        """The constant-velocity guess: P1 (P0^-1 P1) from the last two accepted poses, or the reference pose."""
        if len(self._accepted) < 2:
            return self._accepted[-1].copy()
        p0, p1 = self._accepted[-2:]
        return p1 @ np.linalg.solve(p0, p1)

    def _views(self, buf):
        n = self.iterations
        return (buf[:96].view(torch.float64), buf[96:96 + 32 * n].view(torch.float64).view(n, 4),
                buf[96 + 32 * n:100 + 32 * n].view(torch.int32))

    def _launch(self, depth, weight=None, init=None):
        """The device part of track(): raycast at the reference pose, dca_icp_track and the D2H copy of the results,
        on the current stream, without a host sync.  Returns the guess."""
        depth = _bhw(depth[None] if torch.is_tensor(depth) and depth.dim() == 2 else depth, "depth", torch.float32)
        if tuple(depth.shape) != (1, self.h, self.w) or depth.device != self.volume.state.device:
            raise ValueError(f"depth {tuple(depth.shape)} on {depth.device}: expected [1,{self.h},{self.w}] on "
                             f"{self.volume.state.device}")
        depth = depth[0]
        if weight is not None:
            weight = _bhw(weight[None] if torch.is_tensor(weight) and weight.dim() == 2 else weight, "weight",
                          torch.float32)
            if tuple(weight.shape) != (1, self.h, self.w) or weight.device != depth.device:
                raise ValueError(f"weight {tuple(weight.shape)} on {weight.device}: expected [1,{self.h},{self.w}] "
                                 f"on {depth.device}")
            weight = weight[0]
        if depth.stride(1) != 1 or (weight is not None and weight.stride() != depth.stride()):
            depth = depth.contiguous()
            weight = None if weight is None else weight.contiguous()
        guess = self.predict() if init is None else _poses(init, 1)[0]
        A0 = np.linalg.solve(self._pose, guess)[:3].reshape(12)
        fusion._raycast_kernel(self.volume, self.intrinsics, self.u0, self.v0,
                        self._pose[:3].reshape(12).astype(np.float32), self.min_weight, 0.0, self.max_depth,
                        self.model)
        pose, stats, ok = self._views(self._out)
        _icp_kernel(depth, weight, self.intrinsics, self.u0, self.v0, self.max_depth, self.model, A0, self.levels,
                    self.min_inliers, self.workspace, pose, stats, ok)
        self._host.copy_(self._out, non_blocking=self._cuda)
        if self._cuda:
            self._done.record()
        return guess

    def _collect(self, guess):
        """The host part of track(): the one sync, then the result; a successful frame moves the reference pose."""
        if self._cuda:
            self._done.synchronize()
        pose, stats, ok = (t.numpy() for t in self._views(self._host))
        stats = stats.copy()
        ok = bool(ok[0])
        A = np.eye(4)
        A[:3] = pose.reshape(3, 4)
        with np.errstate(invalid="ignore", divide="ignore"):
            rms = np.sqrt(stats[:, 2] / stats[:, 1])
        result = self._pose @ A if ok else guess
        if ok:
            self._pose = result
            self._accepted = (self._accepted + [result])[-2:]
        return TrackResult(result, ok, stats[:, 0].astype(np.int64), rms)

    def track(self, depth, weight=None, init=None):
        """Track one depth map -> TrackResult.

        depth   fp32 [h,w], [1,h,w] or [1,1,h,w]: PointCloud.depth of reproject on the tracker's window (the left-right
                filter and min_confidence of reproject remove outliers before ICP sees them)
        weight  fp32 map like depth (e.g. the window of Confidence.peak), clamped to [0, 1], NaN = 0; None = 1
        init    a camera-to-world guess (e.g. from an IMU); None = the constant-velocity prediction
        The volume is raycast at tracker.pose, ICP runs from the guess, and cam_to_world = pose . A is composed in
        float64 on the host.  It synchronises once, on purpose: TSDFVolume.integrate computes its voxel box from a host
        pose, and the next raycast takes its pose as launch parameters, so the pose has to reach the host anyway."""
        return self._collect(self._launch(depth, weight, init))


class TrackPipeline(FusePipeline):
    """FusePipeline that tracks each pair before integrating it: the forward and reproject, then (from pair 1 on) the
    raycast, ICP and the D2H copy of the pose on the compute stream; the next pair's H2D copy is queued before the host
    waits for that pose, then the pair is integrated at it.  Pair 0 is integrated at `start`.  A pair that fails to
    track is not integrated; its entry is the prediction."""

    def __init__(self, model, calibs, volume, start, tracker_kw, **kw):
        super().__init__(model, calibs, volume, **kw)
        self.start, self.tracker_kw = _poses(start, 1)[0], tracker_kw
        self.tracker = None
        self.poses, self.ok = [], []

    def _fuse(self, slot, calib, window, pose):
        obs = self._observe(slot, calib, window)
        depth, wmap, _, win = obs
        if self.tracker is None:
            self.tracker = Tracker(self.volume, calib, depth.shape[-2:], win, pose=self.start, **self.tracker_kw)
            self._window = win
            self._integrate(obs, calib, self.start)
            self.poses.append(self.start)
            self.ok.append(True)
            return None
        if tuple(win) != tuple(self._window) or calib is not self.tracker.calib:
            raise ValueError("track_files: every pair must have the window and the calibration of the first")
        return obs, calib, self.tracker._launch(depth, None if wmap is None else wmap[0])

    def _finish(self, pending):
        if pending is None:
            return
        obs, calib, guess = pending
        r = self.tracker._collect(guess)
        self.poses.append(r.cam_to_world)
        self.ok.append(r.ok)
        if r.ok:
            self._integrate(obs, calib, r.cam_to_world)


def track_files(model, items, volume, calib=None, rectifier=None, start=np.eye(4), min_confidence=None,
                lr_check=False, max_depth=40.0, weight="peak", ply=None, min_weight=0.5, levels=LEVELS,
                min_inliers=100, mode="fit", crop=(384, 1248), lr_threshold=1.0, min_depth=0.0, depth=3, workers=2,
                motion=None):
    """Stereo pairs on disk without poses -> Trajectory(poses [N,4,4] float64, ok [N]); the pairs are fused into
    `volume` at their tracked poses.

    items      (left, right) file pairs of one camera, tracked and fused in this order
    volume     a TSDFVolume on the model's device (fused into, not reset); the trajectory must stay inside its grid
    calib      one StereoCalib (or a list aligned with items, all the same object); with a rectifier the items are RAW
               pairs and calib defaults to rectifier.calib
    start      the camera-to-world pose of pair 0, integrated there without tracking
    min_confidence, lr_check   the filters of reproject, applied before ICP and integration
    max_depth  finite: ICP, the raycast and the integration ignore depths beyond it (40 m by default)
    weight     "peak" = Confidence.peak weights both ICP and integration; None = unit weights
    ply        a path: the extracted surface (min_weight), as in fuse_files
    levels, min_inliers   of Tracker; min_weight is also the raycast's
    motion     as in fuse_files: each tracked frame is tested against the last frame integrated, at the tracked poses,
               and its moving objects get weight 0 in the integration (ICP itself is unchanged)
    One host sync per pair, to read the tracked pose (Tracker.track)."""
    if calib is None and rectifier is None:
        raise ValueError("track_files needs a calibration (calib=) or a rectifier (rectifier=)")
    if not (math.isfinite(max_depth) and max_depth > 0):
        raise ValueError(f"max_depth must be finite and > 0, got {max_depth!r}")
    items = list(items)
    pipe = TrackPipeline(model, calib, volume, start,
                         dict(levels=levels, max_depth=max_depth, min_weight=min_weight, min_inliers=min_inliers),
                         mode=mode, crop_height=crop[0], crop_width=crop[1], min_confidence=min_confidence,
                         lr_check=lr_check, lr_threshold=lr_threshold, min_depth=min_depth, max_depth=max_depth,
                         weight=weight, depth=depth, workers=workers, rectifier=rectifier, motion=motion)
    pipe.run(items, np.tile(pipe.start, (len(items), 1, 1)))
    if ply is not None:
        volume.save_ply(ply, min_weight)
    return Trajectory(np.stack(pipe.poses) if pipe.poses else np.zeros((0, 4, 4)), np.array(pipe.ok, bool))
