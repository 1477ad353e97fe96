"""CPU-only host-logic tests: the ordered list of C-ABI entry points (with their shape/mode arguments) that one forward
launches, recorded by a dry run (tests/_dryrun.py: `_lib.call` replaced by a recorder, nothing is computed)."""
import collections
import json
import os

import torch

import _dryrun

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _gold(name):
    return [tuple(t) for t in json.load(open(os.path.join(GOLD, name)))]


def test_default_forward_launches_the_recorded_kernel_sequence():
    """KITTI 384x1248 / maxdisp 192: 41 launches per pair (= bench.py's gpu_launches / steps), in the order recorded when
    the GPU parity suite was last green (tests/golden/make_host_sequences.py)."""
    import dcanet_b200 as d
    tr, (pred4, pv) = _dryrun.forward_trace(d.GwcNet(192).eval(), 96, 312)
    assert pred4.shape == (1, 1, 384, 1248) and pv.shape == (1, 24, 48, 156)
    assert len(tr) == 41
    assert tr == _gold("kernel_sequence_kitti.json")
    tr, _ = _dryrun.forward_trace(d.GwcNet(48).eval(), 16, 32)
    assert tr == _gold("kernel_sequence_tiny.json")


def test_hsharded_forward_host_flow():
    """hshard.hot_path_steps with 3 virtual ranks: every rank launches the un-sharded sequence at its slab shape
    (owned rows + 2 halo rows per side) plus one extra dca_class_stats per cva (S over the owned rows), the stitched
    outputs have the full-image shapes, and a rank issues the recorded number of halo and sum requests."""
    import dcanet_b200 as d
    hs = d.hshard
    H4, W4, world = 24, 40, 3
    feats = [torch.zeros(1, c, H4, W4) for c in (320, 320, 12, 12, 64)]
    net = d.GwcNet(48).eval()
    with _dryrun.recording() as trace:
        pk = net.packed()
        n0 = len(trace)
        with torch.no_grad():
            pred4, pv = hs.hot_path_forward_virtual(pk, *feats, world=world)
        sharded = trace[n0:]
    assert pred4.shape == (1, 1, 4 * H4, 4 * W4) and pv.shape == (1, 6, H4 // 2, W4 // 2)
    # un-sharded forward on ONE slab shape (all three ranks own 8 rows -> 12-row buffers)
    slab, _ = _dryrun.forward_trace(d.GwcNet(48).eval(), 8 + 2 * hs.H4_HALO, W4)
    want = collections.Counter(slab)
    want.update({("dca_class_stats", 1, 6, 4, W4 // 2, 0): 3})          # S[b,k] over the 4 owned 1/8-res rows, per cva
    got = collections.Counter(sharded)
    assert got == collections.Counter({k: v * world for k, v in want.items()})
    # the requests of one rank: 5 feature maps + mask + 4 dres + 3 x (6 at 1/8 res + fused + out) + head + pred_q
    # exchanged, one live row each; the attention output's border-only replicate fill and the S all-reduce once per cva
    with _dryrun.recording():
        with torch.no_grad():
            reqs = list(hs.hot_path_steps(pk, *[hs.owned_rows(f, world, 1) for f in feats]))
    rows = [r for r in reqs if isinstance(r, hs.Rows)]
    assert len(reqs) == 42 and sum(isinstance(r, hs.Sum) for r in reqs) == 3
    assert all(r.nlive == 1 for r in rows if r.exchange)
    assert collections.Counter(r.h for r in rows if r.exchange) == {2: 18, 1: 18}
    assert [(r.h, r.fill) for r in rows if not r.exchange] == [(2, "replicate")] * 3


def test_default_forward_buffer_dataflow():
    """Same launches AND the same buffer wiring between them (pointer arguments normalised to first-appearance ids) as
    recorded from the engine that passed the GPU parity suite: guards host refactors that cannot be run on a GPU."""
    import dcanet_b200 as d
    got = _dryrun.dataflow_trace(d.GwcNet(48).eval(), 16, 32)
    assert got == _gold("kernel_dataflow_tiny.json")
