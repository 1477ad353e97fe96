"""H-sharded single-pair mode (BASELINE.json configs[4], SURVEY.md section 8e): ONE stereo pair, its 1/4-resolution
rows split into contiguous slabs over the ranks of one box, with a halo-row exchange between neighbours after every
layer that looks at neighbouring rows and one [B, D/8] sum all-reduce per cva stage.

STATUS: host logic and exchange plan are covered on CPU (tests/test_hshard_plan.py: the drivers below run the same
plan over the CPU checker's ATen ops, in-process with 2/3/4 virtual ranks and over gloo with world_size 2, against
the un-sharded CPU result; tests/test_host_sequence.py: the launches and requests of a rank, by a dry run).  The kernel
sequence `hot_path_steps` is covered on the GPU by tests/test_gpu_hshard.py (virtual ranks on one device, and one
process per GPU over both transports when >= 2 GPUs are visible).

Frame of one rank.  The rank owns the 1/4-res rows [r0, r1) (both even, so its 1/8-res rows [r0/2, r1/2) align).
Every local tensor carries halo rows: 2 at 1/4 res (buffer = global rows [r0-2, r1+2)), 1 at 1/8 res (global rows
[r0/2-1, r1/2+1)).  With an EVEN 1/4-res halo the stride-2 ops (AvgPool3d k3 s2 p1 `cva.py:39`, conv1 `cva.py:17`),
the transposed conv (`cva.py:21`) and the trilinear x2 (`cva.py:64`) keep their row alignment in the local frame, so
the single-GPU kernels run unchanged on the slab.  A k3 kernel computes garbage in the outermost halo row (it sees the
buffer's zero padding instead of the neighbour's rows); after each such layer the halo rows are refreshed:
  * interior side: the neighbour's owned rows (only the ONE row next to the cut travels, `live`: <= 6.3 MB per side and exchange at Middlebury = 2 planes x 96 x 512 x 32 ch x 2 B),
  * image border: zeros -- exactly the zero padding of the reference's convs / AvgPool3d(count_include_pad) /
    F.unfold(padding=1) -- or, for the trilinear input only, a copy of the border row (align_corners=False clamps).
Per-pixel ops (1x1x1 convs, attention over the disparity axis, softmax + regression) keep valid halos valid.
The only quantity that spans the image is S[b,k] = sum over the pixels of class k of exp(P) (`semantic_level.py:112-116`):
each rank sums its OWNED rows and the [B, D/8] vectors are all-reduced.

The layer sequence is the single-GPU one: `engine.hot_path_steps(..., sharded=True)` yields a `Rows` request after
every layer whose halo rows need a refresh and a `Sum` request for S[b,k].  This module keeps what is specific to
slabs: the row partition, the padding and exchange of the five feature maps, the crop of the results to the owned rows,
and the drivers that fulfil the requests -- `drive_distributed` (one process per GPU, torch.distributed) and
`drive_lockstep` (N virtual ranks in one process, for single-device verification).  Every rank issues the same
sequence of requests, so the exchanges stay in lockstep.
"""
from __future__ import annotations

import os

import torch

from . import _lib
from . import engine as E
from .engine import H4_HALO, H4_LIVE, H8_HALO, Rows, Sum

FUSED_EXCHANGE = os.environ.get("DCA_HALO_FUSED", "1") != "0"   # one launch per exchange instead of push + wait/unpack


# --------------------------------------------------------------------------------------------
# partition
# --------------------------------------------------------------------------------------------
def row_partition(H4, world):
    """Contiguous even-aligned 1/4-res row ranges [(r0, r1)] per rank: the 1/8-res rows are dealt out as evenly as
    possible (SURVEY 8e: Middlebury H4 = 384 over 8 ranks = 48 rows each)."""
    if H4 % 2:
        raise _lib.DcaError("H-sharding needs an even number of 1/4-resolution rows")
    H8 = H4 // 2
    if world < 1 or H8 < 2 * world:
        # >= 2 owned 1/8-res rows per rank keeps every halo inside the DIRECT neighbour's owned rows
        raise _lib.DcaError(f"cannot split {H4} quarter-res rows over {world} ranks (need >= 4 rows per rank)")
    base, extra = divmod(H8, world)
    out, a = [], 0
    for r in range(world):
        b = a + base + (1 if r < extra else 0)
        out.append((2 * a, 2 * b))
        a = b
    return out


def owned_rows(t, world, rank, dim=2, scale=1):
    """The slab of a full-image tensor that `rank` owns (`scale` = 4 for full-res rows, 1 for 1/4 res)."""
    H4 = t.shape[dim] // scale
    r0, r1 = row_partition(H4, world)[rank]
    return t.narrow(dim, r0 * scale, (r1 - r0) * scale).contiguous()


# --------------------------------------------------------------------------------------------
# drivers of the exchange requests (engine.Rows / engine.Sum)
# --------------------------------------------------------------------------------------------
def _fill_border(req: Rows, top: bool):
    t, d, h = req.t, req.dim, req.h
    n = t.shape[d]
    halo = t.narrow(d, 0 if top else n - h, h)
    if req.fill == "zero":
        halo.zero_()
    elif req.fill == "replicate":
        halo.copy_(t.narrow(d, h if top else n - h - 1, 1).expand_as(halo))
    elif req.fill != "keep":
        raise _lib.DcaError(f"unknown halo fill {req.fill!r}")


def _send_rows(req: Rows, to_upper: bool):
    """The owned rows a neighbour needs: the first `live` owned rows go up, the last `live` owned rows go down."""
    n, k = req.t.shape[req.dim], req.nlive
    return req.t.narrow(req.dim, req.h if to_upper else n - req.h - k, k)


def _halo_rows(req: Rows, top: bool):
    """The `live` halo rows next to the owned ones."""
    n, k = req.t.shape[req.dim], req.nlive
    return req.t.narrow(req.dim, req.h - k if top else n - req.h, k)


def drive_lockstep(gens):
    """Run N rank generators in one process (virtual ranks 0..N-1 on one device), fulfilling their requests by plain
    copies between the ranks' buffers.  Returns the list of generator results."""
    n = len(gens)
    results = [None] * n
    while True:
        reqs = []
        for i, g in enumerate(gens):
            try:
                reqs.append(next(g))
            except StopIteration as stop:
                results[i] = stop.value
                reqs.append(None)
        if all(r is None for r in reqs):
            return results
        if any(r is None for r in reqs) or len({type(r) for r in reqs}) != 1:
            raise _lib.DcaError("H-shard ranks fell out of step")
        if isinstance(reqs[0], Sum):
            total = reqs[0].t.clone()
            for r in reqs[1:]:
                total += r.t
            for r in reqs:
                r.t.copy_(total)
            continue
        for i, r in enumerate(reqs):            # halos never overlap owned rows, so the order of the copies is free
            if i == 0:
                _fill_border(r, True)
            elif r.exchange:
                _halo_rows(r, True).copy_(_send_rows(reqs[i - 1], False))
            if i == n - 1:
                _fill_border(r, False)
            elif r.exchange:
                _halo_rows(r, False).copy_(_send_rows(reqs[i + 1], True))


class PeerHalo:
    """Halo rows over NVLink peer memory (csrc/halo_p2p.cu) instead of NCCL send/recv: two launches per exchange on the
    compute stream, no host round trip.  Every rank owns one symmetric buffer (torch symmetric memory, peer-mapped by
    all ranks of the box): 2 parities x 2 directions of staging slots, two 64-bit arrival counters and an error word.
    Slot / counter index 0 = "arrives from ABOVE" (written by rank-1), 1 = "arrives from BELOW" (written by rank+1).
    Opt-in (`transport="p2p"`)."""

    def __init__(self, rank, world, device, group=None, slot_bytes=16 << 20):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        self.rank, self.world, self.slot = rank, world, int(slot_bytes)
        self.buf = symm.empty(4 * self.slot + 64, dtype=torch.uint8, device=device)
        self.hdl = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.buf.zero_()
        torch.cuda.current_stream().synchronize()
        self.hdl.barrier()
        self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        self.ctas = _lib.load().dca_halo_push_ctas()
        self.epoch = 0
        ms = int(os.environ.get("DCA_HALO_TIMEOUT_MS", "10000"))
        _lib.call("dca_halo_set_timeout_ms", ms)
        # the error word of the arrival waits is copied to pinned host memory at the end of every forward and looked at
        # at the start of the next one (and by check()): a timed-out wait raises instead of yielding stale halo rows
        self._err_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self._err_event = None

    def _slot(self, r, parity, direction):
        return self.ptrs[r] + (2 * parity + direction) * self.slot

    def _flag(self, r, direction):
        return self.ptrs[r] + 4 * self.slot + 8 * direction

    def supports(self, req: Rows):
        t = req.t
        inner = t.element_size()
        for d in range(req.dim + 1, t.dim()):
            inner *= t.shape[d]
        outer = 1
        for d in range(req.dim):
            outer *= t.shape[d]
        return (t.is_cuda and t.is_contiguous() and inner % 16 == 0 and t.data_ptr() % 16 == 0
                and outer * req.nlive * inner <= self.slot)

    def refresh(self, req: Rows):
        """Interior sides of one exchange (the caller fills the image-border side).  Every rank must call this for the
        same sequence of requests: the arrival counters count exchanges."""
        t, r = req.t, self.rank
        inner = t.element_size()
        for d in range(req.dim + 1, t.dim()):
            inner *= t.shape[d]
        outer = 1
        for d in range(req.dim):
            outer *= t.shape[d]
        rows = t.shape[req.dim]
        self.epoch += 1
        par = self.epoch & 1
        up, down = r - 1, r + 1
        has_up, has_down = up >= 0, down < self.world
        st = E._stream()
        push = (self._slot(up, par, 1) if has_up else 0, self._slot(down, par, 0) if has_down else 0,
                self._flag(up, 1) if has_up else 0, self._flag(down, 0) if has_down else 0)
        wait = (self._slot(r, par, 0) if has_up else 0, self._slot(r, par, 1) if has_down else 0,
                self._flag(r, 0) if has_up else 0, self._flag(r, 1) if has_down else 0,
                self.epoch * self.ctas, self.ptrs[r] + 4 * self.slot + 16)
        if FUSED_EXCHANGE:       # push + wait/unpack in one launch (halo_exchange_kernel)
            _lib.call("dca_halo_exchange", t.data_ptr(), outer, rows, inner, req.h, req.nlive, *push, *wait, st)
        else:
            _lib.call("dca_halo_push", t.data_ptr(), outer, rows, inner, req.h, req.nlive, *push, st)
            _lib.call("dca_halo_wait_unpack", t.data_ptr(), outer, rows, inner, req.h, req.nlive, *wait, st)

    def _err_word(self):
        return self.buf[4 * self.slot + 16:4 * self.slot + 20].view(torch.int32)

    def end_forward(self):
        """Queue the copy of the error word (no synchronisation); `begin_forward` / `check` look at it."""
        self._err_host.copy_(self._err_word(), non_blocking=True)
        self._err_event = torch.cuda.Event()
        self._err_event.record()

    def begin_forward(self):
        """Raises if a wait of an EARLIER forward timed out (its results were invalid).  Never blocks: the error word is
        sticky on the device (a timed-out wait sets it, nothing clears it), so the copy queued by the latest finished
        forward is enough; when that copy has not landed yet (forwards issued back to back) the look is skipped and the
        next call -- or `check()` -- sees it.  A blocking wait here cost 1.5 ms per Middlebury pair at 8 ranks: every
        forward's issue started on an idle device."""
        if self._err_event is not None and self._err_event.query():
            self._err_event = None
            if int(self._err_host[0]) != 0:
                raise _lib.DcaError("H-shard peer-memory halo exchange timed out waiting for a neighbour: an earlier "
                                    "forward's results were invalid")

    def check(self):
        """Raises if a wait timed out (a neighbour never pushed).  Synchronises; call after the forward."""
        torch.cuda.current_stream().synchronize()
        self._err_event = None
        if int(self._err_word().item()) != 0:
            raise _lib.DcaError("H-shard peer-memory halo exchange timed out waiting for a neighbour")


def drive_distributed(gen, rank, world, group=None, peer: "PeerHalo" = None):
    """Run one rank's generator under torch.distributed (nccl on the GPU box, gloo in the CPU tests): halo rows travel
    as grouped point-to-point sends/receives with the two neighbours (or, with `peer`, as direct NVLink stores into the
    neighbours' staging buffers), S[b,k] as an all-reduce."""
    import torch.distributed as dist
    try:
        req = next(gen)
        while True:
            if isinstance(req, Sum):
                dist.all_reduce(req.t, op=dist.ReduceOp.SUM, group=group)
            elif peer is not None and req.exchange and peer.supports(req):
                if rank == 0:
                    _fill_border(req, True)
                if rank == world - 1:
                    _fill_border(req, False)
                peer.refresh(req)
            else:
                ops, landing = [], []
                for top, nb in ((True, rank - 1), (False, rank + 1)):
                    if nb < 0 or nb >= world:
                        _fill_border(req, top)
                        continue
                    if not req.exchange:
                        continue
                    out = _send_rows(req, top).contiguous()
                    buf = torch.empty_like(out)
                    gpeer = nb if group is None else dist.get_global_rank(group, nb)
                    ops.append(dist.P2POp(dist.isend, out, gpeer, group))
                    ops.append(dist.P2POp(dist.irecv, buf, gpeer, group))
                    landing.append((top, buf))
                if ops:
                    for w in dist.batch_isend_irecv(ops):
                        w.wait()
                    for top, buf in landing:
                        _halo_rows(req, top).copy_(buf)
            req = gen.send(None)
    except StopIteration as stop:
        return stop.value


# --------------------------------------------------------------------------------------------
# the kernel sequence of one rank
# --------------------------------------------------------------------------------------------
def _pad_rows(x, h):
    """fp32 [B,C,Hl,W] -> [B,C,Hl+2h,W] with zeroed halo rows (device memory plumbing, no arithmetic)."""
    B, C, H, W = x.shape
    y = torch.zeros((B, C, H + 2 * h, W), dtype=torch.float32, device=x.device)
    y[:, :, h:h + H].copy_(x)
    return y


def _require_default_route(pk):
    o = E.Options
    if not (o.use_tc and o.use_up2 and o.up2_bilinear and o.prop_on_tc and not o.fp32_stages):
        raise _lib.DcaError("the H-sharded mode runs the default tcgen05 route only (engine.Options at defaults)")
    for c in pk.cva:
        if not c.attn.has_wa:
            raise _lib.DcaError("the H-sharded mode needs the fuse conv folded into the attention pack")


def hot_path_steps(pk: E.PackedHotPath, gwc_l, gwc_r, cat_l, cat_r, g):
    """GwcNet.forward (eval, `gwcnet_dca_g.py:216-240,282`) for the rows this rank owns.  Inputs: the rank's OWNED rows
    of the fp32 feature maps [B,C,Hl,W4].  Result: (pred4 [B,1,4*Hl,4*W4], prob_volume2 [B,D8,Hl/2,W8])."""
    E._require_cuda(gwc_l, gwc_r, cat_l, cat_r, g)
    _require_default_route(pk)
    E.check_feature_shapes(pk, gwc_l, gwc_r, cat_l, cat_r, g)
    if gwc_l.shape[2] % 2 or gwc_l.shape[2] < 4:
        raise _lib.DcaError("a rank must own an even number (>= 4) of 1/4-resolution rows")
    feats = []
    for f in (gwc_l, gwc_r, cat_l, cat_r, g):
        if f is None:
            feats.append(None)
            continue
        fp = _pad_rows(E._f32c(f), H4_HALO)
        yield Rows(fp, 2, H4_HALO, live=H4_LIVE)
        feats.append(fp)
    pred4, pv = yield from E.hot_path_steps(pk, *feats, sharded=True)
    pred4 = pred4[:, :, 4 * H4_HALO:pred4.shape[2] - 4 * H4_HALO].contiguous()
    h = H8_HALO if pk.cva else H4_HALO       # no cva stage: prob_volume2 is the head's own 1/4-res logits
    return pred4, pv[:, :, h:pv.shape[2] - h].contiguous()


_PEERS = {}


def hot_path_forward_hsharded(pk, gwc_l, gwc_r, cat_l, cat_r, g, rank, world, group=None, transport="nccl"):
    """One rank of the H-sharded forward under torch.distributed (inputs and outputs: this rank's owned rows).
    transport: "nccl" (grouped send/recv) or "p2p" (peer-memory stores, csrc/halo_p2p.cu)."""
    peer = None
    if transport == "p2p":
        key = (gwc_l.device.index, rank, world, id(group))
        peer = _PEERS.get(key)
        if peer is None:
            # created AFTER the weights are packed (pk exists); its rendezvous ends with a barrier over the ranks, so the
            # first exchange starts with every rank ready
            peer = _PEERS[key] = PeerHalo(rank, world, gwc_l.device, group)
        peer.begin_forward()
    elif transport != "nccl":
        raise _lib.DcaError(f"unknown H-shard transport {transport!r}")
    res = drive_distributed(hot_path_steps(pk, gwc_l, gwc_r, cat_l, cat_r, g), rank, world, group, peer)
    if peer is not None:
        peer.end_forward()
    return res


def hot_path_forward_virtual(pk, gwc_l, gwc_r, cat_l, cat_r, g, world):
    """The same plan with `world` virtual ranks on ONE device (verification of the plan against the un-sharded
    forward): full-image feature maps in, full-image (pred4, prob_volume2) out."""
    gens = []
    for rank in range(world):
        sl = [None if f is None else owned_rows(f, world, rank) for f in (gwc_l, gwc_r, cat_l, cat_r, g)]
        gens.append(hot_path_steps(pk, *sl))
    res = drive_lockstep(gens)
    return torch.cat([r[0] for r in res], dim=2), torch.cat([r[1] for r in res], dim=2)
