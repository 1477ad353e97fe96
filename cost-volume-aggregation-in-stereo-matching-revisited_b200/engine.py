"""Host-side driver of the hot path: parameter packing and the kernel sequence.

torch is used for device memory (torch.empty on the current device), the current CUDA stream and
nothing else: every arithmetic step below is a call into libdca_b200.so.  No ATen compute op, no
cuDNN/cuBLAS, no CPU fallback.

Data layout in HBM ("cost planes"): channels-last 16-bit `[planes][B][D][H][W][C]` (fp16 by default, see plane_dtype());
planes=2 ("parity": hi + lo, 22-bit significand) or planes=1 ("fast": a single 16-bit plane).

The forward is written once, as generators (`hot_path_steps`, `cva_steps`, `agg_steps`): unsharded they yield nothing
and `_result` runs them to the end; with `sharded=True` they run on one rank's row slab and yield the `Rows` / `Sum`
requests that hshard.py's drivers fulfil.
"""
from __future__ import annotations

import collections
import os
from dataclasses import dataclass

import torch

from . import _lib

ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
K3S1, K3S2, T3S2, K1, C2D3 = 0, 1, 2, 3, 4
BN_EPS = 1e-5


def plane_dtype():
    """torch dtype of the 16-bit cost planes of the loaded library (fp16 by default, bf16 if built with DCA_F16_PLANES=0)."""
    return torch.float16 if _lib.load().dca_plane_format() == 1 else torch.bfloat16


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _lib.DcaError("dcanet_b200 has no CPU path: tensors must live on a CUDA device")


class Planes:
    """A cost tensor in the kernels' layout."""
    __slots__ = ("t", "B", "D", "H", "W", "C", "planes")

    def __init__(self, B, D, H, W, C, planes, device, t=None):
        self.B, self.D, self.H, self.W, self.C, self.planes = B, D, H, W, C, planes
        self.t = t if t is not None else torch.empty((planes, B, D, H, W, C), dtype=plane_dtype(), device=device)

    @property
    def ptr(self):
        return self.t.data_ptr()

    @classmethod
    def from_ncdhw(cls, x, planes=2, cpad=None, out=None):
        """fp32 [B,C,D,H,W] (or [B,C,H,W]) -> planes (into `out` when given)."""
        _require_cuda(x)
        if x.dim() == 4:
            x = x.unsqueeze(2)
        x = x.contiguous().float()
        B, C, D, H, W = x.shape
        Cp = cpad or ((C + 7) // 8 * 8)
        if out is None:
            out = cls(B, D, H, W, Cp, planes, x.device)
        _lib.call("dca_planes_from_ncdhw", x.data_ptr(), out.ptr, planes, B, C, Cp, D, H, W, _stream())
        return out

    def to_ncdhw(self, channels=None):
        C = channels or self.C
        y = torch.empty((self.B, C, self.D, self.H, self.W), dtype=torch.float32, device=self.t.device)
        _lib.call("dca_planes_to_ncdhw", self.ptr, self.planes, y.data_ptr(), self.B, C, self.C, self.D, self.H,
                  self.W, _stream())
        return y


# --------------------------------------------------------------------------------------------
# parameter packing (load time)
# --------------------------------------------------------------------------------------------
class PackedConv:
    """Conv weight repacked to [taps][Cin][CoutPad] fp32 + folded BN scale/shift (fp32, CoutPad)."""

    def __init__(self, weight, bn=None, transposed=False):
        _require_cuda(weight)
        w = weight.detach().contiguous().float()
        if transposed:
            ci, co = w.shape[0], w.shape[1]
        else:
            co, ci = w.shape[0], w.shape[1]
        taps = int(w[0, 0].numel())
        self.cin, self.cout, self.taps = ci, co, taps
        self.cout_pad = (co + 31) // 32 * 32
        dev = w.device
        self.w = torch.empty((taps, ci, self.cout_pad), dtype=torch.float32, device=dev)
        _lib.call("dca_pack_weights", w.data_ptr(), int(transposed), co, ci, taps, self.w.data_ptr(), self.cout_pad,
                  _stream())
        self.scale = self.shift = None
        if bn is not None:
            self.scale = torch.empty(self.cout_pad, dtype=torch.float32, device=dev)
            self.shift = torch.empty(self.cout_pad, dtype=torch.float32, device=dev)
            g, b = bn.weight.detach().float().contiguous(), bn.bias.detach().float().contiguous()
            m, v = bn.running_mean.detach().float().contiguous(), bn.running_var.detach().float().contiguous()
            _lib.call("dca_fold_bn", g.data_ptr(), b.data_ptr(), m.data_ptr(), v.data_ptr(), float(bn.eps),
                      self.scale.data_ptr(), self.shift.data_ptr(), co, self.cout_pad, _stream())
        self.w_tc = None     # bf16 operand pack for the tcgen05 kernels (filled by pack_tc)
        self.w_march = None  # [kh*3+kw][plane][kd][32][Cin] pack of the depth-marching kernel (k3, Cout == 32)
        self.tc_planes = 0
        self._keep = (w,)

    def pack_tc(self, planes, transposed=False):
        nbytes = _lib.load().dca_pack_weights_tc_bytes(self.cout, self.cin, self.taps, planes)
        if nbytes <= 0:
            return False
        self.w_tc = torch.empty(nbytes, dtype=torch.uint8, device=self.w.device)
        _lib.call("dca_pack_weights_tc", self._keep[0].data_ptr(), int(transposed), self.cout, self.cin, self.taps,
                  self.w_tc.data_ptr(), planes, _stream())
        self.tc_planes = planes
        if not transposed and self.taps == 27 and self.cout == 32 and self.cin in (32, 64):
            nb = _lib.load().dca_pack_weights_tc_march_bytes(self.cin, planes)
            self.w_march = torch.empty(nb, dtype=torch.uint8, device=self.w.device)
            _lib.call("dca_pack_weights_tc_march", self._keep[0].data_ptr(), self.cin, self.w_march.data_ptr(), planes,
                      _stream())
        return True


def pack_convbn(seq, transposed=False):
    """seq = Sequential(Conv3d/ConvTranspose3d/Conv2d, BatchNorm) as built by convbn_3d / convbn."""
    return PackedConv(seq[0].weight, seq[1], transposed)


# --------------------------------------------------------------------------------------------
# operators on planes
# --------------------------------------------------------------------------------------------
class Options:
    use_tc = True                 # route eligible convs to the tcgen05 kernels
    tc_modes = {0, 1, 2, 3}       # conv modes the tcgen05 kernel takes (K3S1, K3S2, T3S2, K1)
    fuse_upsample_in_conv = True  # cva fuse stage: fold the trilinear upsample into the 1x1x1 conv's epilogue
    fuse_redir_in_deconv = True   # Multi_Aggregation: conv3 (transposed) + redir (1x1x1) as one GEMM
    use_march = True              # k3 s1 Cout=32 convs: depth-marching kernel (kd folded into the GEMM N)
    march_min_items = 1184        # ... when there are at least this many (tile column, plane) pairs: 8 per SM.  The kernel
                                  # picks the planes per work item itself (KITTI 1/8 res: 6, 36 -> 31 us vs the halo kernel)
    cout1_on_tc = True            # 32->1 convs: tensor-core per-tap GEMM + shifted sum instead of the CUDA-core kernel
    prop_on_tc = True             # the two 3x3 Conv2d of PropgationNet_4x on the halo-slab tcgen05 kernel
    up2_bilinear = True           # fuse stage: depth interpolation in the attention store, bilinear 4-class GEMM
    # guidance branch of PropgationNet_4x (independent of the cost volume) on a second stream with persistent buffers
    # (+1.5 % pairs/s; with allocator-managed buffers the cross-stream frees stalled single steps for 8-100 ms in 2 of
    # 10 bench runs -- 0 of 16 with persistent buffers).  DCA_SIDE_STREAM=0 disables it.
    prop_side_stream = os.environ.get("DCA_SIDE_STREAM", "1") != "0"
    fp32_stages = frozenset()     # diagnostics: stages whose convs run on the fp32 CUDA-core kernel: {'dres', 'cva', 'cls3'}
    use_up2 = True                # class-wise halo-slab kernel for the transposed conv and the trilinear fuse stage
    fuse_tail = True              # conv(32ch)+BN+ReLU -> Conv3d(32->1): per-tap products from the first conv's epilogue


def conv(x: Planes, pc: PackedConv, mode=K3S1, act=ACT_NONE, res_pre: Planes = None, res_post: Planes = None,
         planes_out=None, out_fp32=False, up: Planes = None, side: Planes = None):
    """y = act(scale*(conv(x) + trilinear_x2(up)) + shift + res_pre) + res_post.  Returns Planes, or an fp32
    channels-last tensor [B,D,H,W,Cout] when out_fp32.  `up` needs the tcgen05 kernel."""
    assert x.C == pc.cin, (x.C, pc.cin)
    if mode == K3S2:
        Do, Ho, Wo = (x.D + 1) // 2, (x.H + 1) // 2, (x.W + 1) // 2
    elif mode == T3S2:
        Do, Ho, Wo = 2 * x.D, 2 * x.H, 2 * x.W
    else:
        Do, Ho, Wo = x.D, x.H, x.W
    planes_out = planes_out or x.planes
    dev = x.t.device
    res = res_pre if res_pre is not None else res_post
    planes_res = res.planes if res is not None else 1
    if res_pre is not None and res_post is not None:
        assert res_pre.planes == res_post.planes
    if out_fp32:
        y = torch.empty((x.B, Do, Ho, Wo, pc.cout), dtype=torch.float32, device=dev)
        yptr = y.data_ptr()
    else:
        y = Planes(x.B, Do, Ho, Wo, pc.cout, planes_out, dev)
        yptr = y.ptr
    if (Options.use_tc and Options.use_march and mode == K3S1 and not out_fp32 and up is None and side is None
            and pc.w_march is not None and pc.tc_planes == x.planes and planes_out == x.planes
            and x.B * x.D * ((x.H + 15) // 16) * ((x.W + 7) // 8) >= Options.march_min_items):
        # depth-marching kernel: enough (tile column x depth chunk) work items to fill the SMs
        _lib.call("dca_conv3d_tc_march", x.ptr, x.planes, pc.w_march.data_ptr(), _ptr(pc.scale), _ptr(pc.shift),
                  res_pre.ptr if res_pre is not None else 0, res_post.ptr if res_post is not None else 0, planes_res,
                  yptr, act, x.B, pc.cin, x.D, x.H, x.W, _stream())
        return y
    if (Options.use_tc and not out_fp32 and pc.w_tc is not None and pc.tc_planes == x.planes
            and tc_supported(mode, pc.cin, pc.cout)):
        _lib.call("dca_conv3d_tc", mode, x.ptr, x.planes, pc.w_tc.data_ptr(), _ptr(pc.scale), _ptr(pc.shift),
                  res_pre.ptr if res_pre is not None else 0, res_post.ptr if res_post is not None else 0, planes_res,
                  up.ptr if up is not None else 0, up.planes if up is not None else 1,
                  side.ptr if side is not None else 0, side.C if side is not None else 0,
                  yptr, planes_out, act, x.B, pc.cin, pc.cout, x.D, x.H, x.W, Do, Ho, Wo, _stream())
        return y
    if up is not None or side is not None:
        raise _lib.DcaError("conv(..., up=/side=) is only implemented by the tcgen05 kernel")
    _lib.call("dca_conv3d_direct", mode, x.ptr, x.planes, pc.w.data_ptr(), _ptr(pc.scale), _ptr(pc.shift),
              res_pre.ptr if res_pre is not None else 0, res_post.ptr if res_post is not None else 0, planes_res,
              yptr, planes_out, 1 if out_fp32 else 0, act, x.B, pc.cin, pc.cout, pc.cout_pad, x.D, x.H, x.W, Do, Ho,
              Wo, _stream())
    return y


class PackedConv2dTc:
    """Conv2d 3x3 (or 1x1, embedded as the centre tap of a 3x3) + optional bias + optional eval-mode BN packed for
    dca_conv2d_tc*: 16-bit hi/lo weights in 64x64 (Cout chunk, Cin slab) tiles; bias and BN folded to fp32 scale/shift
    padded to a multiple of 64 (BN(conv + b) = s*conv + (s*b + t)).  Cin a multiple of 64, at most 320."""

    def __init__(self, weight, bn, planes, bias=None, pad_cout=False):
        w = weight.detach().contiguous().float()
        if w.shape[-1] == 1:                       # 1x1 -> 3x3 with a single non-zero tap (memory plumbing only)
            w3 = torch.zeros((w.shape[0], w.shape[1], 3, 3), dtype=torch.float32, device=w.device)
            w3[:, :, 1, 1] = w[:, :, 0, 0]
            w = w3
        self.cout_valid = w.shape[0]
        if pad_cout and w.shape[0] % 64:           # plane outputs are whole 64-channel rows: zero output channels on top
            assert bn is None and bias is None
            wp = torch.zeros(((w.shape[0] + 63) // 64 * 64,) + tuple(w.shape[1:]), dtype=torch.float32, device=w.device)
            wp[:w.shape[0]] = w
            w = wp
        self.cout, self.cin = w.shape[0], w.shape[1]
        dev = w.device
        nb = _lib.load().dca_pack_weights_tc2d_bytes(self.cout, self.cin, planes)
        if nb <= 0:
            raise _lib.DcaError("dca_conv2d_tc supports Cin = 64, 128, ... 320")
        self.w = torch.empty(nb, dtype=torch.uint8, device=dev)
        _lib.call("dca_pack_weights_tc2d", w.data_ptr(), self.cout, self.cin, self.w.data_ptr(), planes, _stream())
        self.planes = planes
        self.scale = self.shift = None
        cpad = (self.cout + 63) // 64 * 64
        if bn is not None:
            self.scale = torch.empty(cpad, dtype=torch.float32, device=dev)
            self.shift = torch.empty(cpad, dtype=torch.float32, device=dev)
            g, b = bn.weight.detach().float().contiguous(), bn.bias.detach().float().contiguous()
            m, v = bn.running_mean.detach().float().contiguous(), bn.running_var.detach().float().contiguous()
            _lib.call("dca_fold_bn", g.data_ptr(), b.data_ptr(), m.data_ptr(), v.data_ptr(), float(bn.eps),
                      self.scale.data_ptr(), self.shift.data_ptr(), self.cout, cpad, _stream())
        if bias is not None:                       # load-time parameter folding on [Cout] vectors
            b = bias.detach().float()
            if self.scale is None:
                self.scale = torch.ones(cpad, dtype=torch.float32, device=dev)
                self.shift = torch.zeros(cpad, dtype=torch.float32, device=dev)
            self.shift[:self.cout] += self.scale[:self.cout] * b
        torch.cuda.current_stream().synchronize()


def conv2d_tc(x: Planes, pc: PackedConv2dTc, act=ACT_NONE, out_fp32=False, out=None, res: Planes = None, act_post=ACT_NONE,
              dil=1):
    """y = act_post(act(scale * conv3x3(x, dilation dil) + shift) + res) on the halo-slab tcgen05 kernel."""
    assert x.D == 1 and x.C == pc.cin and x.planes == pc.planes
    dev = x.t.device
    if out_fp32:
        y = out if out is not None else torch.empty((x.B, 1, x.H, x.W, pc.cout), dtype=torch.float32, device=dev)
        yptr = y.data_ptr()
    else:
        y = out if out is not None else Planes(x.B, 1, x.H, x.W, pc.cout, x.planes, dev)
        yptr = y.ptr
    if res is None and dil == 1:
        _lib.call("dca_conv2d_tc", x.ptr, x.planes, pc.w.data_ptr(), _ptr(pc.scale), _ptr(pc.shift), yptr, int(out_fp32),
                  act, x.B, pc.cin, pc.cout, x.H, x.W, _stream())
        return y
    if res is not None:
        assert (res.B, res.H, res.W, res.C, res.planes) == (x.B, x.H, x.W, pc.cout, x.planes)
    _lib.call("dca_conv2d_tc_ex", x.ptr, x.planes, pc.w.data_ptr(), _ptr(pc.scale), _ptr(pc.shift),
              res.ptr if res is not None else 0, int(act_post), yptr, int(out_fp32), act, x.B, pc.cin, pc.cout, x.H, x.W,
              int(dil), _stream())
    return y


class PackedStem:
    """Conv2d(3 -> 32, K x K, stride 2) (+ bias) + eval-mode BN for dca_conv2d_stem: fp32 weights in torch layout, BN and bias
    folded to scale/shift."""

    def __init__(self, conv, bn):
        w = conv.weight.detach().contiguous().float()
        if w.shape[0] != 32 or w.shape[1] != 3 or w.shape[2] not in (3, 7) or conv.stride != (2, 2):
            raise _lib.DcaError("dca_conv2d_stem: Conv2d(3 -> 32, 3x3 or 7x7, stride 2) only")
        self.w, self.k = w, int(w.shape[2])
        dev = w.device
        self.scale = torch.ones(32, dtype=torch.float32, device=dev)
        self.shift = torch.zeros(32, dtype=torch.float32, device=dev)
        if bn is not None:
            g, b = bn.weight.detach().float().contiguous(), bn.bias.detach().float().contiguous()
            m, v = bn.running_mean.detach().float().contiguous(), bn.running_var.detach().float().contiguous()
            _lib.call("dca_fold_bn", g.data_ptr(), b.data_ptr(), m.data_ptr(), v.data_ptr(), float(bn.eps),
                      self.scale.data_ptr(), self.shift.data_ptr(), 32, 32, _stream())
        if conv.bias is not None:
            self.shift += self.scale * conv.bias.detach().float()
        torch.cuda.current_stream().synchronize()


def conv2d_stem(x, ps: PackedStem, planes, act=ACT_RELU):
    """fp32 NCHW image [B,3,H,W] -> cost planes [P][B][1][H/2][W/2][32]."""
    _require_cuda(x)
    x = x.contiguous().float()
    B, C, H, W = x.shape
    assert C == 3
    k = ps.k
    y = Planes(B, 1, (H + 2 * (k // 2) - k) // 2 + 1, (W + 2 * (k // 2) - k) // 2 + 1, 32, planes, x.device)
    _lib.call("dca_conv2d_stem", x.data_ptr(), ps.w.data_ptr(), ps.scale.data_ptr(), ps.shift.data_ptr(), y.ptr, planes, act,
              B, H, W, k, _stream())
    return y


def pack_conv2d_s2(conv, bn, planes):
    """A stride-2 Conv2d(32 -> 64) (3x3 pad 1, or 1x1) as the middle depth slice of a 3x3x3 stride-2 Conv3d on a depth-1
    volume: the w-pair slab kernel of Multi_Aggregation.conv1 (K3S2) then IS the 2-D conv (its two outer depth taps read
    the zero padding).  Bias folded into the BN shift."""
    w = conv.weight.detach().float()
    co, ci, k = w.shape[0], w.shape[1], w.shape[2]
    w3 = torch.zeros((co, ci, 3, 3, 3), dtype=torch.float32, device=w.device)
    if k == 3:
        w3[:, :, 1] = w
    elif k == 1:
        w3[:, :, 1, 1, 1] = w[:, :, 0, 0]
    else:
        raise _lib.DcaError("pack_conv2d_s2: 3x3 or 1x1 kernels")
    pc = PackedConv(w3, bn)
    if conv.bias is not None:
        if pc.scale is None:
            pc.scale = torch.ones(pc.cout_pad, dtype=torch.float32, device=w.device)
            pc.shift = torch.zeros(pc.cout_pad, dtype=torch.float32, device=w.device)
        pc.shift[:co] += pc.scale[:co] * conv.bias.detach().float()
    if not pc.pack_tc(planes) or not tc_supported(K3S2, ci, co):
        raise _lib.DcaError("pack_conv2d_s2: the stride-2 tensor-core kernel takes 32 -> 64 channels")
    torch.cuda.current_stream().synchronize()
    return pc


def conv2d_tc_cat(xs, pc: PackedConv2dTc, act=ACT_NONE):
    """conv3x3 over the channel concatenation of up to three plane tensors, without materialising it."""
    x0 = xs[0]
    assert 1 <= len(xs) <= 3 and sum(x.C for x in xs) == pc.cin
    assert all((x.B, x.H, x.W, x.planes) == (x0.B, x0.H, x0.W, x0.planes) for x in xs) and x0.planes == pc.planes
    y = Planes(x0.B, 1, x0.H, x0.W, pc.cout, x0.planes, x0.t.device)
    a = [(x.ptr, x.C) for x in xs] + [(0, 0)] * (3 - len(xs))
    _lib.call("dca_conv2d_tc_cat", a[0][0], a[0][1], a[1][0], a[1][1], a[2][0], a[2][1], x0.planes, pc.w.data_ptr(),
              _ptr(pc.scale), _ptr(pc.shift), y.ptr, 0, act, x0.B, pc.cout, x0.H, x0.W, _stream())
    return y


def planes_to_nchw_slice(x: Planes, out, c0, channels=None):
    """Write x (2-D planes) as channels [c0, c0 + C) of the fp32 NCHW tensor `out` (the torch.cat of the reference)."""
    C = channels or x.C
    assert x.D == 1 and out.is_contiguous() and out.dtype == torch.float32 and out.shape[0] == x.B
    assert out.shape[2:] == (x.H, x.W) and c0 + C <= out.shape[1]
    _lib.call("dca_planes_to_nchw_slice", x.ptr, x.planes, out.data_ptr() + 4 * c0 * x.H * x.W, x.B, C, x.C, x.H, x.W,
              out.shape[1] * x.H * x.W, _stream())


def tc_supported(mode, cin, cout):
    return mode in Options.tc_modes and cin in (32, 64) and cout in (32, 64)


def conv_cout1(x: Planes, w27: torch.Tensor):
    """Conv3d k3 s1 p1 to one channel -> fp32 logits [B,D,H,W]."""
    y = torch.empty((x.B, x.D, x.H, x.W), dtype=torch.float32, device=x.t.device)
    _lib.call("dca_conv3d_cout1", x.ptr, x.planes, w27.data_ptr(), y.data_ptr(), x.B, x.C, x.D, x.H, x.W, _stream())
    return y


class PackedCout1:
    """Conv3d(32 -> 1, k3) packed twice: host [27][32] fp32 for the CUDA-core marching kernel, and a [32][32] 1x1x1
    bf16 operand pack (row = tap) for the tensor-core per-tap GEMM + shifted-sum path."""

    def __init__(self, weight, planes):
        self.host = pack_cout1(weight)
        w = weight.detach().float()
        ci = w.shape[1]
        self.w_tc = None
        if ci == 32:
            wt = torch.zeros((32, ci, 1, 1, 1), dtype=torch.float32, device=w.device)
            wt[:27, :, 0, 0, 0] = w.reshape(ci, 27).t()
            nb = _lib.load().dca_pack_weights_tc_bytes(32, ci, 1, planes)
            self.w_tc = torch.empty(nb, dtype=torch.uint8, device=w.device)
            _lib.call("dca_pack_weights_tc", wt.data_ptr(), 0, 32, ci, 1, self.w_tc.data_ptr(), planes, _stream())
            torch.cuda.current_stream().synchronize()
        self.planes = planes


def conv_cout1_any(x: Planes, pc):
    """32 -> 1 channel 3x3x3 conv: tensor-core per-tap GEMM + 27-tap shifted sum when possible, else the CUDA-core
    marching kernel."""
    nvox = x.B * x.D * x.H * x.W
    if (Options.use_tc and Options.cout1_on_tc and isinstance(pc, PackedCout1) and pc.w_tc is not None
            and pc.planes == x.planes and nvox % 8 == 0):
        P = torch.empty((27, nvox), dtype=torch.float32, device=x.t.device)
        _lib.call("dca_conv1_taps_tc", x.ptr, x.planes, pc.w_tc.data_ptr(), P.data_ptr(), 27, x.B, x.D, x.H, x.W,
                  _stream())
        y = torch.empty((x.B, x.D, x.H, x.W), dtype=torch.float32, device=x.t.device)
        _lib.call("dca_tap_gather3d", P.data_ptr(), y.data_ptr(), x.B, x.D, x.H, x.W, _stream())
        return y
    return conv_cout1(x, pc.host if isinstance(pc, PackedCout1) else pc)


def conv_taps27(x: Planes, pc: PackedConv, pc1: "PackedCout1", act=ACT_RELU):
    """act(BN(conv3x3x3(x)))  ->  per-tap products of the Conv3d(32 -> 1, k3) that follows, straight from the first conv's
    epilogue: fp32 P [27, B, D, H, W] (tap-major), or None when the fused kernel does not apply (the caller then runs the
    two convs separately)."""
    if not (Options.use_tc and Options.fuse_tail and pc.cout == 32 and pc.cin in (32, 64) and pc.taps == 27
            and pc.tc_planes == x.planes and pc1.host.shape == (27, 32)):
        return None
    march = (Options.use_march and pc.w_march is not None
             and x.B * x.D * ((x.H + 15) // 16) * ((x.W + 7) // 8) >= Options.march_min_items)
    w = pc.w_march if march else pc.w_tc
    if w is None:
        return None
    P = torch.empty((27, x.B, x.D, x.H, x.W), dtype=torch.float32, device=x.t.device)
    _lib.call("dca_conv3d_tc_taps27", x.ptr, x.planes, w.data_ptr(), int(march), _ptr(pc.scale), _ptr(pc.shift),
              pc1.host.data_ptr(), P.data_ptr(), act, x.B, pc.cin, x.D, x.H, x.W, _stream())
    return P


def tap_gather(P):
    """27-tap shifted sum: P [27,B,D,H,W] -> logits [B,D,H,W]."""
    _, B, D, H, W = P.shape
    y = torch.empty((B, D, H, W), dtype=torch.float32, device=P.device)
    _lib.call("dca_tap_gather3d", P.data_ptr(), y.data_ptr(), B, D, H, W, _stream())
    return y


def tap_gather_softmax_regress(P, want_logits=False):
    """P [27,B,D,H,W] -> (pred [B,1,H,W], logits [B,D,H,W] or None): shifted sum + softmax + regression in one kernel."""
    _, B, D, H, W = P.shape
    pred = torch.empty((B, 1, H, W), dtype=torch.float32, device=P.device)
    logits = torch.empty((B, D, H, W), dtype=torch.float32, device=P.device) if want_logits else None
    _lib.call("dca_tap_gather_softmax_regress", P.data_ptr(), pred.data_ptr(), _ptr(logits), B, D, H, W, _stream())
    return pred, logits


def pack_cout1(weight):
    """[1,Cin,3,3,3] -> HOST tensor [27][Cin] fp32 (the kernel takes these 864 weights as launch parameters).
    Packed on the device by the generic packer (taps x Cin x CoutPad with CoutPad=1), copied back once at load."""
    w = weight.detach().contiguous().float()
    ci = w.shape[1]
    out = torch.empty((27, ci), dtype=torch.float32, device=w.device)
    _lib.call("dca_pack_weights", w.data_ptr(), 0, 1, ci, 27, out.data_ptr(), 1, _stream())
    return out.cpu().contiguous()


def avgpool(x: Planes):
    y = Planes(x.B, (x.D + 1) // 2, (x.H + 1) // 2, (x.W + 1) // 2, x.C, x.planes, x.t.device)
    _lib.call("dca_avgpool3d", x.ptr, y.ptr, x.planes, x.B, x.C, x.D, x.H, x.W, _stream())
    return y


def class_stats(logits):
    B, D, H, W = logits.shape
    dev = logits.device
    cls = torch.empty((B, H, W), dtype=torch.int32, device=dev)
    e = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    S = torch.empty((B, D), dtype=torch.float32, device=dev)
    scratch = torch.empty(B * D + 1, dtype=torch.int64, device=dev)     # fixed-point sums + ticket (order-independent)
    _lib.call("dca_class_stats", logits.data_ptr(), cls.data_ptr(), e.data_ptr(), S.data_ptr(), scratch.data_ptr(), B, D,
              H, W, _stream())
    return cls, e, S


def disp_attention(x: Planes, cls, e, S, weights, has_wa, pad=0):
    """pad=1: the result gets a replicated 1-voxel border ([D+2][H+2][W+2]) for the up2 (trilinear) GEMM;
    pad=2: the result is already interpolated x2 along depth and border-replicated in h/w ([2D][H+2][W+2])."""
    pad = int(pad)
    if pad == 2:
        y = Planes(x.B, 2 * x.D, x.H + 2, x.W + 2, x.C, x.planes, x.t.device)
    else:
        k = 2 if pad else 0
        y = Planes(x.B, x.D + k, x.H + k, x.W + k, x.C, x.planes, x.t.device)
    _lib.call("dca_disp_attention", x.ptr, cls.data_ptr(), e.data_ptr(), S.data_ptr(), weights.data_ptr(),
              int(has_wa), y.ptr, int(pad), x.planes, x.B, x.C, x.D, x.H, x.W, _stream())
    return y


def up2(kind, x: Planes, side: Planes, w_tc, scale, shift, act, cin, dl, hl, wl, res_post: Planes = None):
    """dca_up2_tc: kind 0 transposed conv (+side 1x1x1), kind 1 trilinear x2 of a padded tensor + side 1x1x1,
    kind 2 bilinear x2 in (h, w) of a depth-interpolated padded tensor + side 1x1x1 (dl = OUTPUT depth)."""
    y = Planes(x.B, dl if kind == 2 else 2 * dl, 2 * hl, 2 * wl, 32, x.planes, x.t.device)
    for name, o in (("side", side), ("res_post", res_post)):
        # both are read at the OUTPUT resolution through tensor maps built from (dl, hl, wl): a mismatch (odd H/4 or W/4)
        # would be silent out-of-bounds reads, where the reference raises at its torch.cat (cva.py:55)
        if o is not None and (o.B, o.D, o.H, o.W) != (y.B, y.D, y.H, y.W):
            raise _lib.DcaError(f"up2: {name} is {(o.B, o.D, o.H, o.W)}, the output is {(y.B, y.D, y.H, y.W)} "
                                "(D/4, H/4 and W/4 must be even)")
    _lib.call("dca_up2_tc", kind, x.ptr, x.planes, side.ptr if side is not None else 0,
              side.C if side is not None else 0, w_tc.data_ptr(), _ptr(scale), _ptr(shift),
              res_post.ptr if res_post is not None else 0, res_post.planes if res_post is not None else 1, y.ptr, act,
              x.B, cin, dl, hl, wl, _stream())
    return y


def upsample_fuse(t: Planes, cost: Planes, wcT, scale, shift):
    assert cost.D == 2 * t.D and cost.H == 2 * t.H and cost.W == 2 * t.W, "cva needs even D/4, H/4, W/4"
    y = Planes(cost.B, cost.D, cost.H, cost.W, cost.C, cost.planes, cost.t.device)
    _lib.call("dca_upsample_fuse", t.ptr, cost.ptr, wcT.data_ptr(), scale.data_ptr(), shift.data_ptr(), y.ptr,
              cost.planes, cost.B, cost.C, t.D, t.H, t.W, _stream())
    return y


def softmax_regress(logits):
    B, D, H, W = logits.shape
    pred = torch.empty((B, 1, H, W), dtype=torch.float32, device=logits.device)
    _lib.call("dca_softmax_regress", logits.data_ptr(), pred.data_ptr(), B, D, H, W, _stream())
    return pred


def regress(x):
    """sum_d d * x[:, d] (the reference's disparity_regression on its own, submodule.py:127-131)."""
    B, D, H, W = x.shape
    pred = torch.empty((B, 1, H, W), dtype=torch.float32, device=x.device)
    _lib.call("dca_regress_f32", x.data_ptr(), pred.data_ptr(), B, D, H, W, _stream())
    return pred


def self_attention(q: Planes, k: Planes, weights):
    """SelfAttentionBlock.forward(query_feats, key_feats) (SelfAttention_bn.py:62-98) on cost planes."""
    assert (q.B, q.D, q.H, q.W, q.C, q.planes) == (k.B, k.D, k.H, k.W, k.C, k.planes)
    y = Planes(q.B, q.D, q.H, q.W, q.C, q.planes, q.t.device)
    _lib.call("dca_self_attention", q.ptr, k.ptr, weights.data_ptr(), y.ptr, q.planes, q.B, q.C, q.D, q.H, q.W, _stream())
    return y


def cached_pack(module, key, build):
    """Pack a module's parameters for the kernels ONCE and reuse the pack until a parameter or buffer of the module is
    replaced, moved or modified in place (data_ptr / _version signature).  The function-level API (cva, Multi_Aggregation,
    hourglass, SemanticLevelContext, PropgationNet_4x, run_convbn_3d) goes through this, so drop-in callers do not
    re-pack every weight on every call."""
    sig = tuple((t.data_ptr(), t._version) for t in list(module.parameters()) + list(module.buffers()))
    cache = module.__dict__.setdefault("_dca_packs", {})
    hit = cache.get(key)
    if hit is None or hit[0] != sig:
        hit = cache[key] = (sig, build())
        torch.cuda.current_stream().synchronize()      # temporaries of the packers die here
    return hit[1]


def convex_upsample(mask, disp):
    B, _, H, W = disp.shape
    out = torch.empty((B, 1, 4 * H, 4 * W), dtype=torch.float32, device=disp.device)
    _lib.call("dca_convex_upsample", mask.data_ptr(), disp.data_ptr(), out.data_ptr(), B, H, W, _stream())
    return out


# Per-pixel confidence of pred4 (include/dca_b200.h section 4): peak = convex-upsampled max_d p(d), in [0, 1]; std =
# convex-upsampled 4 * (standard deviation of the disparity distribution), in full-res px.  fp32 [B,1,H,W] each.
Confidence = collections.namedtuple("Confidence", ["peak", "std"])


def softmax_confidence_upsample(logits, mask, quarter=False):
    """logits [B,D,H,W] + prop-net mask -> (Confidence at 4H x 4W, peak_q, std_q); the 1/4-res maps [B,1,H,W] only when
    `quarter`, else None."""
    B, D, H, W = logits.shape
    dev = logits.device
    peak = torch.empty((B, 1, 4 * H, 4 * W), dtype=torch.float32, device=dev)
    std = torch.empty((B, 1, 4 * H, 4 * W), dtype=torch.float32, device=dev)
    pq = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev) if quarter else None
    sq = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev) if quarter else None
    _lib.call("dca_softmax_confidence_upsample", logits.data_ptr(), mask.data_ptr(), _ptr(pq), _ptr(sq), peak.data_ptr(),
              std.data_ptr(), B, D, H, W, _stream())
    return Confidence(peak, std), pq, sq


# Left-right consistency check (include/dca_b200.h section 8): the right view's disparity, a per-pixel label and the
# background-filled disparity, each shaped like the left disparity.
LRCheck = collections.namedtuple("LRCheck", ["disp_right", "label", "filled"])
LR_CONSISTENT, LR_OCCLUDED, LR_MISMATCH, LR_OUT_OF_VIEW = 0, 1, 2, 3


def lr_consistency(disp_left, disp_right, tau=1.0, mirrored=False, want_right=False):
    """disp_left, disp_right fp32 [B,H,W] or [B,1,H,W] -> (label uint8, filled fp32, right fp32 or None), shaped like
    disp_left.  `mirrored`: disp_right is net(flip(R), flip(L)) as the mirrored forward wrote it, i.e. flip(D_R), and is
    read back to front.  `want_right` also returns D_R in the natural layout, written by the kernel from its staged rows.
    One launch of dca_lr_consistency; W <= 4096 (DCA_LR_MAX_W)."""
    _require_cuda(disp_left, disp_right)
    if disp_left.shape != disp_right.shape or disp_left.dim() not in (3, 4) or \
            (disp_left.dim() == 4 and disp_left.shape[1] != 1):
        raise _lib.DcaError(f"disparities must be two equal [B,H,W] or [B,1,H,W] tensors, got "
                            f"{tuple(disp_left.shape)} / {tuple(disp_right.shape)}")
    if disp_left.dtype != torch.float32 or disp_right.dtype != torch.float32 or disp_left.device != disp_right.device:
        raise _lib.DcaError("disparities must be float32 on one device")
    dl, dr = disp_left.contiguous(), disp_right.contiguous()
    B, H, W = dl.shape[0], dl.shape[-2], dl.shape[-1]
    label = torch.empty(dl.shape, dtype=torch.uint8, device=dl.device)
    filled = torch.empty_like(dl)
    right = torch.empty_like(dl) if want_right else None
    _lib.call("dca_lr_consistency", dl.data_ptr(), dr.data_ptr(), int(bool(mirrored)), label.data_ptr(),
              filled.data_ptr(), _ptr(right), B, H, W, float(tau), _stream())
    return label, filled, right


def fused_volume(gwc_l, gwc_r, cat_l, cat_r, D, G, planes, Cv=None, guide=None):
    """guide = (hq fp32 [B,H,W] contiguous, k, s): the guided volume of include/dca_b200.h section 14."""
    _require_cuda(gwc_l, gwc_r, cat_l, cat_r)
    B, C, H, W = gwc_l.shape
    Cc = 0 if cat_l is None else cat_l.shape[1]
    Cv = Cv or ((G + 2 * Cc + 7) // 8 * 8)
    vol = Planes(B, D, H, W, Cv, planes, gwc_l.device)
    args = (gwc_l.data_ptr(), gwc_r.data_ptr(), _ptr(cat_l), _ptr(cat_r), vol.ptr, B, C, G, Cc, D, H, W, Cv, planes)
    if guide is None:
        _lib.call("dca_volume_gwc_concat", *args, _stream())
    else:
        hq, k, s = guide
        _require_cuda(hq)
        if tuple(hq.shape) != (B, H, W) or hq.dtype != torch.float32 or not hq.is_contiguous():
            raise _lib.DcaError(f"hq: expected contiguous float32 [{B}, {H}, {W}], got {hq.dtype} {tuple(hq.shape)}")
        _lib.call("dca_volume_gwc_concat_guided", *args, hq.data_ptr(), float(k), float(s), _stream())
    return vol


def guide_quarter(hints, maxdisp):
    """Full-res hint map fp32 [B,H,W] (contiguous, H and W multiples of 4) -> hq [B,H/4,W/4]: the largest valid hint
    (finite, 0 < h < maxdisp) of each 4x4 block divided by 4, 0 where there is none (dca_guide_quarter)."""
    _require_cuda(hints)
    B, H, W = hints.shape
    hq = torch.empty((B, H // 4, W // 4), dtype=torch.float32, device=hints.device)
    _lib.call("dca_guide_quarter", hints.data_ptr(), B, H, W, float(maxdisp), hq.data_ptr(), _stream())
    return hq


def _f32c(t):
    return t.contiguous().float()


# --------------------------------------------------------------------------------------------
# requests of the H-sharded sequence (fulfilled by the drivers in hshard.py)
# --------------------------------------------------------------------------------------------
H4_HALO = 2      # halo rows at 1/4 resolution (even: keeps the stride-2 alignment)
H8_HALO = 1      # halo rows at 1/8 resolution
H4_LIVE = 1      # 1/4-res halo rows that are ever read for an owned output (the outer one only keeps the alignment)


@dataclass
class Rows:
    """Refresh the `h` halo rows at both ends of `dim` of `t` (owned rows = [h, n-h)).  Interior side: the neighbour's
    owned rows next to the cut (only if `exchange`).  Image border: `fill` = "zero" | "replicate" | "keep" (all h rows).
    `live`: only that many halo rows, the ones next to the owned rows, are read by any op that produces OWNED output
    (the outer 1/4-res halo row exists for the stride-2 alignment only), so only they travel."""
    t: torch.Tensor
    dim: int
    h: int
    fill: str = "zero"
    exchange: bool = True
    live: int = 0         # rows (next to the owned ones) that actually travel; 0 = all h

    @property
    def nlive(self):
        return self.live or self.h


@dataclass
class Sum:
    """All-reduce (sum) `t` in place over the ranks."""
    t: torch.Tensor


def _result(steps):
    """Run an unsharded sequence generator (it yields no request) and return its result."""
    try:
        next(steps)
    except StopIteration as stop:
        return stop.value
    raise _lib.DcaError("an unsharded sequence yielded a halo request")


# --------------------------------------------------------------------------------------------
# packed parameter sets for the composite blocks
# --------------------------------------------------------------------------------------------
class PackedAttention:
    """7 transposed 32x32 matrices (q0,q1,k0,k1,v,o,Wa) + 6 x (scale,shift), one flat fp32 buffer."""

    def __init__(self, attn, fuse_conv_weight=None):
        convs = [attn.query_project[0], attn.query_project[1], attn.key_project[0], attn.key_project[1],
                 attn.value_project, attn.out_project]
        dev = convs[0][0].weight.device
        self.buf = torch.zeros(7 * 1024 + 6 * 64, dtype=torch.float32, device=dev)
        for i, seq in enumerate(convs):
            pc = PackedConv(seq[0].weight, seq[1])
            assert pc.cin == 32 and pc.cout == 32 and pc.taps == 1
            self.buf[i * 1024:(i + 1) * 1024].copy_(pc.w.view(-1))
            o = 7 * 1024 + i * 64
            self.buf[o:o + 32].copy_(pc.scale[:32])
            self.buf[o + 32:o + 64].copy_(pc.shift[:32])
        self.has_wa = fuse_conv_weight is not None
        if self.has_wa:
            wa = fuse_conv_weight.detach()[:, :32].contiguous()
            pc = PackedConv(wa)
            self.buf[6 * 1024:7 * 1024].copy_(pc.w.view(-1))


class PackedCva:
    def __init__(self, m, planes):
        self.down = pack_convbn(m.downsample[1])
        self.cls0 = pack_convbn(m.classify[0])
        self.cls2 = PackedCout1(m.classify[2].weight, planes)
        fuse_w = m.fuse[0][0].weight                      # [32, 64, 1,1,1]: in = cat(aug, cost)
        self.attn = PackedAttention(m.slc_net.cross_attention, fuse_w)
        pc_c = PackedConv(fuse_w.detach()[:, 32:].contiguous(), m.fuse[0][1])
        pc_c.pack_tc(planes)
        self.fuse_c = pc_c                                # cost half of the fuse conv (+ the fuse BN)
        self.fuse_wcT = pc_c.w.view(32, 32).contiguous()  # [ci][co]
        self.fuse_scale, self.fuse_shift = pc_c.scale, pc_c.shift
        self.agg = PackedAgg(m.cost_agg, planes)
        self.conv1, self.conv2, self.conv3, self.redir = self.agg.conv1, self.agg.conv2, self.agg.conv3, self.agg.redir
        self.conv3_fused = self.agg.conv3_fused
        for pc in (self.down, self.cls0):
            pc.pack_tc(planes)
        # trilinear x2 + cat + fuse as a GEMM: 4 diagonal interpolation taps {27,9,3,1}/64 * I and the cost half Wc
        w5 = torch.zeros((32, 32, 5), dtype=torch.float32, device=fuse_w.device)       # [co][ci][tap]
        eye = torch.eye(32, device=fuse_w.device)
        for i, wv in enumerate((27.0, 9.0, 3.0, 1.0)):
            w5[:, :, i] = eye * (wv / 64.0)
        w5[:, :, 4] = fuse_w.detach().float()[:, 32:, 0, 0, 0]
        nb = _lib.load().dca_pack_weights_tc_bytes(32, 32, 5, planes)
        self.fuse_up2_w = torch.empty(nb, dtype=torch.uint8, device=fuse_w.device)
        _lib.call("dca_pack_weights_tc", w5.data_ptr(), 0, 32, 32, 5, self.fuse_up2_w.data_ptr(), planes, _stream())
        torch.cuda.current_stream().synchronize()
        # same with the depth axis resolved upstream: bilinear taps {9,3,1}/16 * I and Wc
        w4 = torch.zeros((32, 32, 4), dtype=torch.float32, device=fuse_w.device)
        for i, wv in enumerate((9.0, 3.0, 1.0)):
            w4[:, :, i] = eye * (wv / 16.0)
        w4[:, :, 3] = fuse_w.detach().float()[:, 32:, 0, 0, 0]
        nb4 = _lib.load().dca_pack_weights_tc_bytes(32, 32, 4, planes)
        self.fuse_up2b_w = torch.empty(nb4, dtype=torch.uint8, device=fuse_w.device)
        _lib.call("dca_pack_weights_tc", w4.data_ptr(), 0, 32, 32, 4, self.fuse_up2b_w.data_ptr(), planes, _stream())
        torch.cuda.current_stream().synchronize()


FUSED_REDIR_MAX = 1.0e3     # largest |Wr * sr / s3| accepted by the fused deconv + redir pack


class PackedAgg:
    """Multi_Aggregation (cva.py:13-31): conv1 (k3 s2) -> conv2 (k3 s1) -> conv3 (transposed k3 s2) + redir (1x1x1)."""

    def __init__(self, agg, planes):
        self.conv1 = pack_convbn(agg.conv1[0])
        self.conv2 = pack_convbn(agg.conv2[0])
        self.conv3 = PackedConv(agg.conv3[0].weight, agg.conv3[1], transposed=True)
        self.redir = pack_convbn(agg.redir)
        for pc in (self.conv1, self.conv2, self.redir):
            pc.pack_tc(planes)
        self.conv3.pack_tc(planes, transposed=True)
        c = agg.redir[0].weight.shape[0]
        self.conv3_fused = _pack_deconv_with_redir(agg, self.conv3, self.redir, planes) if c == 32 else None


def agg_steps(pk: PackedAgg, x: Planes, res_post: Planes = None, keep=None, sharded=False):
    """Multi_Aggregation.forward (cva.py:26-31): ReLU(BN(conv3(conv2(conv1 x))) + BN(redir x)) (+ res_post).  Generator;
    the result comes back through StopIteration."""
    c1 = conv(x, pk.conv1, K3S2, ACT_RELU)
    if sharded:
        yield Rows(c1.t, 3, H8_HALO)
    c2 = conv(c1, pk.conv2, K3S1, ACT_RELU)
    if sharded:
        yield Rows(c2.t, 3, H8_HALO)
    fd = pk.conv3_fused
    if Options.use_tc and Options.use_up2 and fd is not None and fd.tc_planes == c2.planes:
        out = up2(0, c2, x, fd.w_tc, fd.scale, fd.shift, ACT_RELU, 64, c2.D, c2.H, c2.W, res_post=res_post)
    elif Options.use_tc and Options.fuse_redir_in_deconv and fd is not None and fd.tc_planes == c2.planes \
            and tc_supported(T3S2, 64, 32):
        # ReLU(BN(deconv(c2)) + BN(redir(x))) (+ res_post) as one tcgen05 GEMM with a 28th, 1x1x1 tap
        out = Planes(c2.B, 2 * c2.D, 2 * c2.H, 2 * c2.W, 32, c2.planes, c2.t.device)
        _lib.call("dca_conv3d_tc", T3S2, c2.ptr, c2.planes, fd.w_tc.data_ptr(), fd.scale.data_ptr(),
                  fd.shift.data_ptr(), 0, res_post.ptr if res_post is not None else 0,
                  res_post.planes if res_post is not None else 1, 0, 1, x.ptr, x.C, out.ptr, c2.planes,
                  ACT_RELU, c2.B, 64, 32, c2.D, c2.H, c2.W, out.D, out.H, out.W, _stream())
    else:
        # also taken when the fused deconv + redir pack was declined (a tiny BN gamma of conv3, _pack_deconv_with_redir):
        # redir is per voxel, so valid halo rows stay valid
        redir = conv(x, pk.redir, K1, ACT_NONE)
        out = conv(c2, pk.conv3, T3S2, ACT_RELU, res_pre=redir, res_post=res_post)
    if sharded:
        yield Rows(out.t, 3, H4_HALO, live=H4_LIVE)
    if keep is not None:
        keep.update(c1=c1, c2=c2)
    return out


class _FusedDeconv:
    """conv3 (ConvTranspose3d 64->32 + BN) and redir (1x1x1 32->32 + BN) of Multi_Aggregation as ONE GEMM:
    s3*deconv + b3 + sr*(Wr x) + br = s3*(deconv + (diag(sr/s3) Wr) x) + (b3 + br): 27 deconv taps + a 28th
    tap holding diag(sr/s3) Wr zero-padded from 32 to 64 input channels."""

    def __init__(self, w_tc, scale, shift, planes):
        self.w_tc, self.scale, self.shift, self.tc_planes = w_tc, scale, shift, planes
        self.cin, self.cout = 64, 32


def _pack_deconv_with_redir(agg, pc3, pcr, planes):
    s3, sr = pc3.scale[:32], pcr.scale[:32]
    if pc3.w_tc is None or bool((s3.abs() < 1e-12).any()):
        return None                                   # a zero BN scale cannot be divided out: keep the two kernels
    # the rescaled redir weights go into fp16 hi/lo planes (saturating at 65504, and hi*lo products in fp32): decline when
    # a decayed / dead BN gamma of conv3 would blow them up (real checkpoints have gammas down to 1e-8); the two-kernel
    # route (redir as its own 1x1x1 conv, added as res_pre) has no such division
    wr_scaled = agg.redir[0].weight.detach().float().view(32, 32) * (sr / s3).view(32, 1)
    if not bool(torch.isfinite(wr_scaled).all()) or float(wr_scaled.abs().max()) > FUSED_REDIR_MAX:
        return None
    lib = _lib.load()
    per_tap = lib.dca_pack_weights_tc_bytes(32, 64, 1, planes)
    buf = torch.empty(28 * per_tap, dtype=torch.uint8, device=pc3.w.device)
    buf[:27 * per_tap].copy_(pc3.w_tc)
    wr = agg.redir[0].weight.detach().float().view(32, 32) * (sr / s3).view(32, 1)      # [co][ci]
    wr64 = torch.zeros((32, 64, 1, 1, 1), dtype=torch.float32, device=wr.device)
    wr64[:, :32, 0, 0, 0] = wr
    _lib.call("dca_pack_weights_tc", wr64.data_ptr(), 0, 32, 64, 1, buf[27 * per_tap:].data_ptr(), planes, _stream())
    torch.cuda.current_stream().synchronize()        # wr64 is a temporary
    return _FusedDeconv(buf, pc3.scale, (pc3.shift + pcr.shift).contiguous(), planes)


def cva_steps(pk: PackedCva, cost: Planes, res_post: Planes = None, keep=None, sharded=False):
    """cva.forward(downsample=True) (cva.py:59-72).  Generator; returns (logits fp32 [B,D8,H8,W8], augmented cost Planes)
    through StopIteration.  Sharded, `cost` arrives with refreshed halo rows and `out` leaves with them."""
    pooled = avgpool(cost)
    if sharded:
        yield Rows(pooled.t, 3, H8_HALO)
    cost_down = conv(pooled, pk.down, K3S1, ACT_RELU)
    if sharded:
        yield Rows(cost_down.t, 3, H8_HALO)
    P27 = conv_taps27(cost_down, pk.cls0, pk.cls2)
    if P27 is not None:
        if sharded:        # the per-tap products are a per-voxel function of the conv's output rows
            yield Rows(P27, 3, H8_HALO)
        logits = tap_gather(P27)
    else:
        h = conv(cost_down, pk.cls0, K3S1, ACT_RELU)
        if sharded:
            yield Rows(h.t, 3, H8_HALO)
        logits = conv_cout1_any(h, pk.cls2)
    if sharded:
        yield Rows(logits, 2, H8_HALO)
    cls, e, S = class_stats(logits)
    if sharded:            # S[b,k] over the OWNED pixels, summed over the ranks = over the image
        _, _, S = class_stats(logits[:, :, H8_HALO:logits.shape[2] - H8_HALO].contiguous())
        yield Sum(S)
    use_up2 = Options.use_tc and Options.use_up2 and pk.attn.has_wa
    bil = use_up2 and Options.up2_bilinear
    t = disp_attention(cost_down, cls, e, S, pk.attn.buf, pk.attn.has_wa, pad=(2 if bil else (1 if use_up2 else 0)))
    if sharded:
        # t: [2*D8][Hb8+2][W8+2], replicated 1-voxel border in h/w.  Interior cuts need nothing (the halo row is a valid
        # per-pixel result); at the image border the clamp of the trilinear must start at the border row, not outside it.
        yield Rows(t.t, 3, H8_HALO + 1, fill="replicate", exchange=False)
    if bil:
        # depth axis of the trilinear already resolved by the attention kernel's store; 4-class bilinear GEMM here
        fused = up2(2, t, cost, pk.fuse_up2b_w, pk.fuse_scale, pk.fuse_shift, ACT_NONE, 32, cost.D, cost_down.H,
                    cost_down.W)
    elif use_up2:
        # trilinear x2 + cat + 1x1x1 fuse + BN as ONE class-wise GEMM over halo slabs of the padded low-res tensor
        fused = up2(1, t, cost, pk.fuse_up2_w, pk.fuse_scale, pk.fuse_shift, ACT_NONE, 32, cost_down.D, cost_down.H,
                    cost_down.W)
    elif Options.use_tc and Options.fuse_upsample_in_conv and tc_supported(K1, 32, 32):
        # trilinear x2 + cat + 1x1x1 fuse + BN as ONE tcgen05 conv: Wc.cost by MMA, up(t) added in the epilogue
        fused = conv(cost, pk.fuse_c, K1, ACT_NONE, up=t)
    else:
        fused = upsample_fuse(t, cost, pk.fuse_wcT, pk.fuse_scale, pk.fuse_shift)
    if sharded:
        yield Rows(fused.t, 3, H4_HALO, live=H4_LIVE)
    out = yield from agg_steps(pk.agg, fused, res_post=res_post, sharded=sharded)
    if keep is not None:
        keep.update(pooled=pooled, cost_down=cost_down, logits=logits, class_map=cls, e=e, S=S, t=t, fused=fused, out=out)
    return logits, out


class PackedHotPath:
    """All hot-path parameters of a GwcNet, packed for the kernels."""

    def __init__(self, net, planes):
        self.planes = planes
        self.maxdisp = net.maxdisp
        self.num_groups = net.num_groups
        self.dres0_0 = pack_convbn(net.dres0[0]); self.dres0_2 = pack_convbn(net.dres0[2])
        self.dres1_0 = pack_convbn(net.dres1[0]); self.dres1_2 = pack_convbn(net.dres1[2])
        # stage-count variants (gwcnet_dca{0,1,2,4}_g.py): N cva stages, head = classif<N>, returned class logits = stage pv_stage
        self.num_cva = getattr(net, "num_cva", 3)
        self.pv_stage = getattr(net, "pv_stage", 2)
        self.cva = [PackedCva(getattr(net, f"cva{i + 1}"), planes) for i in range(self.num_cva)]
        head = getattr(net, f"classif{self.num_cva}")
        self.cls3_0 = pack_convbn(head[0])
        self.cls3_2 = PackedCout1(head[2].weight, planes)
        self.prop0 = pack_convbn(net.prop.conv[0])
        self.prop2 = PackedConv(net.prop.conv[2].weight)
        self.prop0_tc = PackedConv2dTc(net.prop.conv[0][0].weight, net.prop.conv[0][1], planes)
        self.prop2_tc = PackedConv2dTc(net.prop.conv[2].weight, None, planes)
        for pc in (self.dres0_0, self.dres0_2, self.dres1_0, self.dres1_2, self.cls3_0):
            pc.pack_tc(planes)


_SIDE_STREAMS = {}


def _prop_mask_steps(pk, g, P, sharded=False):
    """PropgationNet_4x.conv on the guidance features (gwcnet_dca_g.py:112-115,119): fp32 channels-last mask logits.
    Generator; the mask comes back through StopIteration."""
    gp = Planes.from_ncdhw(g, planes=P)
    if Options.use_tc and Options.prop_on_tc:
        m1 = conv2d_tc(gp, pk.prop0_tc, ACT_RELU)
        if sharded:
            yield Rows(m1.t, 3, H4_HALO, live=H4_LIVE)
        return conv2d_tc(m1, pk.prop2_tc, ACT_NONE, out_fp32=True)
    m1 = conv(gp, pk.prop0, C2D3, ACT_RELU)
    return conv(m1, pk.prop2, C2D3, ACT_NONE, out_fp32=True)


def _prop_mask_start(pk, g, P):
    """The mask branch only depends on the guidance features, so it is issued on a second stream at the start of the
    forward: its 5 short launches (234 tiles each) fill SMs that the cost-volume kernels leave idle at their tails."""
    main = torch.cuda.current_stream()
    dev = (g.device.index, main.cuda_stream)   # one side stream AND one buffer set per calling stream: forwards issued
    side = _SIDE_STREAMS.get(dev)              # concurrently on several streams must not share the mask buffers
    if side is None:
        side = _SIDE_STREAMS[dev] = torch.cuda.Stream(device=g.device)
    side.wait_stream(main)                 # g is ready, and the previous forward no longer reads the buffers below
    capturing = torch.cuda.is_current_stream_capturing()
    if not capturing:
        g.record_stream(side)
    # persistent buffers per shape: no caching-allocator traffic on the side stream (cross-stream frees made single
    # steps stall for 8-100 ms in 2 of 10 bench runs)
    B, Cg, H, W = g.shape
    key = (g.device.index, main.cuda_stream, B, Cg, H, W, P)
    # (under CUDA-graph capture the buffers come from the graph's own pool instead: every graph bakes in its own set)
    bufs = None if capturing else pk.__dict__.setdefault("_side_bufs", {}).get(key)
    if bufs is None and not capturing and Options.use_tc and Options.prop_on_tc:
        gp = Planes(B, 1, H, W, (Cg + 7) // 8 * 8, P, g.device)
        m1 = Planes(B, 1, H, W, pk.prop0_tc.cout, P, g.device)
        mask = torch.empty((B, 1, H, W, pk.prop2_tc.cout), dtype=torch.float32, device=g.device)
        bufs = pk._side_bufs[key] = (gp, m1, mask)
    with torch.cuda.stream(side):
        if bufs is not None:
            gp, m1, mask = bufs
            Planes.from_ncdhw(g, planes=P, out=gp)
            conv2d_tc(gp, pk.prop0_tc, ACT_RELU, out=m1)
            conv2d_tc(m1, pk.prop2_tc, ACT_NONE, out_fp32=True, out=mask)
        else:
            mask = _result(_prop_mask_steps(pk, g, P))
    return (side, mask, main, bufs)


def _prop_mask_wait(job):
    side, mask, main, bufs = job
    main.wait_stream(side)
    if bufs is None and not torch.cuda.is_current_stream_capturing():
        mask.record_stream(main)
    return mask


def check_feature_shapes(pk, gwc_l, gwc_r, cat_l, cat_r, g):
    """The five feature maps must agree in (B, H/4, W/4); with cva stages D/4, H/4 and W/4 must be even (the reference
    raises at `torch.cat` in cva.py:55 otherwise; here the up2 tensor maps would be built with the wrong pitches)."""
    if gwc_l.dim() != 4 or gwc_l.shape != gwc_r.shape:
        raise _lib.DcaError(f"gwc features must be two equal [B,C,H/4,W/4] tensors, got {tuple(gwc_l.shape)} / {tuple(gwc_r.shape)}")
    B, _, H4, W4 = gwc_l.shape
    if (cat_l is None) != (cat_r is None):
        raise _lib.DcaError("concat features: both or none")
    for name, t in (("cat_l", cat_l), ("cat_r", cat_r), ("guidance", g)):
        if t is not None and (t.dim() != 4 or (t.shape[0], t.shape[2], t.shape[3]) != (B, H4, W4)):
            raise _lib.DcaError(f"{name} is {tuple(t.shape)}, expected [{B}, C, {H4}, {W4}]")
    if cat_l is not None and cat_l.shape != cat_r.shape:
        raise _lib.DcaError("concat features differ in shape")
    if pk.cva and (H4 % 2 or W4 % 2 or (pk.maxdisp // 4) % 2):
        raise _lib.DcaError(f"cva needs even D/4, H/4, W/4 (got {pk.maxdisp // 4}, {H4}, {W4}): pad the images to a "
                            "multiple of 8 (the reference's callers pad to 16, main_dca.py:153-166)")


def hot_path_forward(pk: PackedHotPath, gwc_l, gwc_r, cat_l, cat_r, g, keep=None, confidence=False, guide=None):
    """Feature maps -> (pred4 [B,1,H,W], prob_volume2 logits [B,D8,H8,W8]), plus a third item Confidence(peak, std)
    (fp32 [B,1,H,W] each) when `confidence`.  Mirrors GwcNet.forward (eval) of the reference,
    models/gwcnet_dca_g.py:216-240,282; the confidence is this library's addition (one more launch after the upsampling,
    pred4 and prob_volume2 unchanged bit for bit).  guide = (hints fp32 [B, 4 H/4, 4 W/4] contiguous, k, s) runs the
    LiDAR-guided volume (include/dca_b200.h section 14)."""
    _require_cuda(gwc_l, gwc_r, cat_l, cat_r, g)
    check_feature_shapes(pk, gwc_l, gwc_r, cat_l, cat_r, g)
    if guide is not None:
        B, _, H4, W4 = gwc_l.shape
        hints = guide[0]
        _require_cuda(hints)
        if tuple(hints.shape) != (B, 4 * H4, 4 * W4) or hints.dtype != torch.float32 or not hints.is_contiguous():
            raise _lib.DcaError(f"hints: expected contiguous float32 [{B}, {4 * H4}, {4 * W4}], got {hints.dtype} "
                                f"{tuple(hints.shape)}")
    tc0 = Options.use_tc
    try:
        return _result(hot_path_steps(pk, gwc_l, gwc_r, cat_l, cat_r, g, keep, confidence, guide=guide))
    finally:
        Options.use_tc = tc0          # fp32_stages (diagnostics) toggles it per stage; never leak that into later calls


def hot_path_steps(pk: PackedHotPath, gwc_l, gwc_r, cat_l, cat_r, g, keep=None, confidence=False, sharded=False,
                   guide=None):
    """The launches of `hot_path_forward`, as a generator returning its result through StopIteration.  Sharded, the
    feature maps are one rank's row slab with H4_HALO refreshed halo rows per side (hshard.py), a `Rows` request follows
    every layer whose halo rows need a refresh and a `Sum` request the per-class sums S[b,k]; the results keep their
    halo rows.  Unsharded, nothing is yielded.  guide = (full-res hints [B,H,W], k, s): dca_guide_quarter, then the
    guided volume (unsharded only)."""
    P = pk.planes
    D4 = pk.maxdisp // 4
    g = _f32c(g)
    if guide is not None and sharded:
        raise _lib.DcaError("LiDAR guidance is not available in the H-sharded forward")
    hq = guide_quarter(guide[0], pk.maxdisp) if guide is not None else None
    side_job = _prop_mask_start(pk, g, P) if Options.prop_side_stream and not sharded else None
    vol = fused_volume(_f32c(gwc_l), _f32c(gwc_r), _f32c(cat_l) if cat_l is not None else None,
                       _f32c(cat_r) if cat_r is not None else None, D4, pk.num_groups, P,
                       guide=(hq, guide[1], guide[2]) if guide is not None else None)
    tc0 = Options.use_tc
    Options.use_tc = tc0 and "dres" not in Options.fp32_stages
    c = conv(vol, pk.dres0_0, K3S1, ACT_RELU)
    if sharded:
        yield Rows(c.t, 3, H4_HALO, live=H4_LIVE)
    c = conv(c, pk.dres0_2, K3S1, ACT_RELU)
    if sharded:
        yield Rows(c.t, 3, H4_HALO, live=H4_LIVE)
    r = conv(c, pk.dres1_0, K3S1, ACT_RELU)
    if sharded:
        yield Rows(r.t, 3, H4_HALO, live=H4_LIVE)
    cost0 = conv(r, pk.dres1_2, K3S1, ACT_NONE, res_post=c)
    if sharded:
        yield Rows(cost0.t, 3, H4_HALO, live=H4_LIVE)
    Options.use_tc = tc0 and "cva" not in Options.fp32_stages
    kept = [{} if keep is not None else None for _ in pk.cva]
    cur, out1, logits2 = cost0, None, None
    for i, stage in enumerate(pk.cva):      # cva1 adds cost0 back (gwcnet_dca_g.py:229), the others chain
        lg, cur = yield from cva_steps(stage, cur, res_post=cost0 if i == 0 else None, keep=kept[i], sharded=sharded)
        if i == 0:
            out1 = cur
        if i + 1 == pk.pv_stage:
            logits2 = lg
    Options.use_tc = tc0 and "cls3" not in Options.fp32_stages
    P27 = conv_taps27(cur, pk.cls3_0, pk.cls3_2)
    if P27 is not None:
        if sharded:
            yield Rows(P27, 3, H4_HALO, live=H4_LIVE)
        # the head's logits are only an OUTPUT when there is no cva stage (gwcnet_dca0_g.py:190), when a caller keeps them
        # or when the confidence is wanted
        pred_q, logits = tap_gather_softmax_regress(P27, want_logits=(not pk.cva) or keep is not None or confidence)
    else:
        h = conv(cur, pk.cls3_0, K3S1, ACT_RELU)
        if sharded:         # only one halo row of h is live: the logits are valid on the owned rows
            yield Rows(h.t, 3, H4_HALO, live=H4_LIVE)
        logits = conv_cout1_any(h, pk.cls3_2)
        pred_q = softmax_regress(logits)
    Options.use_tc = tc0
    if side_job is not None:
        mask = _prop_mask_wait(side_job)
    else:
        mask = yield from _prop_mask_steps(pk, g, P, sharded)
    if sharded:
        # the convex upsampling reads the 3x3 neighbourhood of the regressed disparity: one row from each neighbour, and
        # zero DISPARITY outside the image (F.unfold(padding=1) of the reference)
        yield Rows(pred_q, 2, H4_HALO, fill="zero", live=H4_LIVE)
    pred4 = convex_upsample(mask, pred_q)
    if confidence:
        conf, peak_q, std_q = softmax_confidence_upsample(logits, mask, quarter=keep is not None)
    if keep is not None:
        keep.update(volume=vol, dres0=c, cost0=cost0, out1=out1, classif3_logits=logits, pred_quarter=pred_q, mask=mask)
        keep.update({f"cva{i + 1}": k for i, k in enumerate(kept)})
        if confidence:
            keep.update(peak_quarter=peak_q, std_quarter=std_q)
        if hq is not None:
            keep.update(hint_quarter=hq)
    pv = logits if not pk.cva else logits2     # no cva stage (gwcnet_dca0_g.py:190): the head's own logits
    return (pred4, pv, conf) if confidence else (pred4, pv)


# --------------------------------------------------------------------------------------------
# the forward as ONE CUDA graph
# --------------------------------------------------------------------------------------------
class GraphedHotPath:
    """`hot_path_forward` captured once per (input buffers, shapes) into a CUDA graph and replayed: the ~46 launches of
    a forward (programmatic-dependent-launch edges included) become one `cudaGraphLaunch`, so the host cost per pair
    drops from ~0.9 ms of ctypes calls to ~10 us and the launch-bound small shapes stop being launch bound.

    The graph reads the caller's input tensors IN PLACE (their addresses are baked in): calling again with the same
    tensors (new contents) replays; other tensors capture another graph (a small LRU of them, all sharing one memory
    pool -- their replays are ordered on the calling stream, so they may reuse each other's activations).  Results are
    returned as copies, so they survive the next replay.  `confidence` is part of the graph key: the forward with the
    confidence maps is a graph of its own.  So are the LiDAR hint map's address and shape, k and s: the hint map is read
    in place like the other inputs.  Weights are baked in as well: `GwcNet` drops its graphs
    whenever it drops its packed parameters."""
    MAX_GRAPHS = 8

    def __init__(self, pk: "PackedHotPath"):
        self.pk = pk
        self.graphs = {}          # key -> (graph, static outputs, input tensors kept alive)
        self.pool = None
        self.replays = 0

    @staticmethod
    def _key(tensors):
        return tuple((0, ()) if t is None else (t.data_ptr(), tuple(t.shape)) for t in tensors)

    def _capture(self, ins, confidence=False, guide=None):
        s = torch.cuda.Stream(device=ins[0].device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):                 # warm-up outside the capture: lazy module loads, persistent side buffers
            for _ in range(2):
                hot_path_forward(self.pk, *ins, confidence=confidence, guide=guide)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize(ins[0].device)
        g = torch.cuda.CUDAGraph()
        if self.pool is None:
            self.pool = torch.cuda.graph_pool_handle()
        with torch.cuda.graph(g, pool=self.pool):
            out = hot_path_forward(self.pk, *ins, confidence=confidence, guide=guide)
        return g, out

    def __call__(self, gwc_l, gwc_r, cat_l, cat_r, g, confidence=False, guide=None):
        ins = (gwc_l, gwc_r, cat_l, cat_r, g)
        _require_cuda(*ins)
        for t in ins + ((guide[0],) if guide is not None else ()):
            if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
                raise _lib.DcaError("the graphed forward reads its inputs in place: contiguous fp32 tensors only")
        confidence = bool(confidence)
        key = self._key(ins) + (confidence,)
        if guide is not None:
            guide = (guide[0], float(guide[1]), float(guide[2]))
            key += self._key(guide[:1]) + guide[1:]
        hit = self.graphs.pop(key, None)
        if hit is None:
            if len(self.graphs) >= self.MAX_GRAPHS:
                self.graphs.pop(next(iter(self.graphs)))
            graph, out = self._capture(ins, confidence) if guide is None else self._capture(ins, confidence, guide)
            hit = (graph, out, ins + (guide,))
        self.graphs[key] = hit                     # most recently used last
        hit[0].replay()
        self.replays += 1
        return tuple(o.clone() if torch.is_tensor(o) else type(o)(*(t.clone() for t in o)) for o in hit[1])
