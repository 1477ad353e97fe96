"""CPU-only: the H-sharded single-pair plan (BASELINE.json configs[4], SURVEY 8e) and its two drivers.

The product's kernel sequence (`hshard.hot_path_steps`) needs a GPU; what runs here is the SAME plan -- halo widths
(2 rows at 1/4 res, 1 at 1/8), refresh after every layer that reads neighbouring rows, zero / replicate fills at the
image border, S[b,k] summed over the owned rows and all-reduced -- restated over the oracle's ATen ops (`_oracle_steps`
mirrors `hot_path_steps` step for step), driven by the product's own `drive_lockstep` (2/3/4 virtual ranks) and
`drive_distributed` (gloo, world_size 2), and compared with the un-sharded oracle.
"""
import importlib
import os
import socket

import pytest
import torch
import torch.nn.functional as F

from oracle import dcanet_oracle as O

hs = importlib.import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.hshard")
Rows, Sum = hs.Rows, hs.Sum

MAXDISP = 32


def _cva_oracle_steps(ctx, p, cost, res=None):
    pooled = F.avg_pool3d(cost, 3, stride=2, padding=1)
    yield Rows(pooled, 3, 1)
    cost_down = ctx.convbn3d(pooled, p + ".downsample.1", 1, 1, "relu")
    yield Rows(cost_down, 3, 1)
    h = ctx.convbn3d(cost_down, p + ".classify.0", 1, 1, "relu")
    yield Rows(h, 3, 1)
    logits = ctx.conv3d(h, p + ".classify.2.weight", 1, 1).squeeze(1).contiguous()
    yield Rows(logits, 2, 1)
    _, k, e, _, _ = O.class_stats(logits)
    S = O.class_stats(logits[:, :, 1:-1].contiguous())[3]
    yield Sum(S)
    B, C, D, H, W = cost_down.shape
    w = e / S.gather(1, k.view(B, -1)).view(B, H, W)
    onehot = F.one_hot(k, D).permute(0, 3, 1, 2).to(cost_down.dtype)
    key = cost_down * (1.0 + onehot * w.unsqueeze(1)).unsqueeze(1)
    aug_down = O.disparity_attention(ctx, p + ".slc_net.cross_attention", cost_down, key).contiguous()
    yield Rows(aug_down, 3, 1, fill="replicate", exchange=False)
    aug = F.interpolate(aug_down, scale_factor=(2, 2, 2), mode="trilinear")
    fused = ctx.convbn3d(torch.cat([aug, cost], dim=1), p + ".fuse.0", 1, 0, None)
    yield Rows(fused, 3, 2, live=1)
    c1 = ctx.convbn3d(fused, p + ".cost_agg.conv1.0", 2, 1, "relu")
    yield Rows(c1, 3, 1)
    c2 = ctx.convbn3d(c1, p + ".cost_agg.conv2.0", 1, 1, "relu")
    yield Rows(c2, 3, 1)
    c3 = ctx.bn(ctx.deconv3d(c2, p + ".cost_agg.conv3.0.weight"), p + ".cost_agg.conv3.1")
    out = F.relu(c3 + ctx.convbn3d(fused, p + ".cost_agg.redir", 1, 0, None))
    if res is not None:
        out = out + res
    out = out.contiguous()
    yield Rows(out, 3, 2, live=1)
    return logits, out


def _oracle_steps(sd, gl, gr, cl, cr, g):
    ctx = O._Ctx(sd)
    D4 = MAXDISP // 4
    feats = []
    for f in (gl, gr, cl, cr, g):
        fp = F.pad(f, (0, 0, 2, 2)).contiguous()
        yield Rows(fp, 2, 2, live=1)
        feats.append(fp)
    gl, gr, cl, cr, g = feats
    vol = torch.cat([O.build_gwc_volume(gl, gr, D4, 40), O.build_concat_volume(cl, cr, D4)], dim=1)
    c = ctx.convbn3d(vol, "dres0.0", 1, 1, "relu")
    yield Rows(c, 3, 2, live=1)
    c = ctx.convbn3d(c, "dres0.2", 1, 1, "relu")
    yield Rows(c, 3, 2, live=1)
    r = ctx.convbn3d(c, "dres1.0", 1, 1, "relu")
    yield Rows(r, 3, 2, live=1)
    cost0 = (ctx.convbn3d(r, "dres1.2", 1, 1, None) + c).contiguous()
    yield Rows(cost0, 3, 2, live=1)
    _, out1 = yield from _cva_oracle_steps(ctx, "cva1", cost0, res=cost0)
    logits2, out2 = yield from _cva_oracle_steps(ctx, "cva2", out1)
    _, out3 = yield from _cva_oracle_steps(ctx, "cva3", out2)
    h = ctx.convbn3d(out3, "classif3.0", 1, 1, "relu")
    yield Rows(h, 3, 2, live=1)
    logits = ctx.conv3d(h, "classif3.2.weight", 1, 1).squeeze(1)
    pred_q = O.disparity_regression(F.softmax(logits, dim=1), D4).contiguous()
    m1 = F.relu(ctx.bn(ctx.conv2d(g, "prop.conv.0.0.weight"), "prop.conv.0.1")).contiguous()
    yield Rows(m1, 2, 2, live=1)
    mlog = ctx.conv2d(m1, "prop.conv.2.weight")
    yield Rows(pred_q, 2, 2, fill="zero", live=1)
    B, _, H, W = pred_q.shape
    m = F.softmax(mlog.view(B, 9, 4, 4, H, W), dim=1)
    dp = F.pad(4.0 * pred_q[:, 0], (1, 1, 1, 1))
    up = pred_q.new_zeros(B, 4, 4, H, W)
    for n in range(9):
        dy, dx = n // 3, n % 3
        up = up + m[:, n] * dp[:, None, None, dy:dy + H, dx:dx + W]
    pred4 = up.permute(0, 3, 1, 4, 2).reshape(B, 1, 4 * H, 4 * W)
    return pred4[:, :, 8:4 * H - 8].contiguous(), logits2[:, :, 1:-1].contiguous()


def _case(H4, W4, seed=0):
    feats = O.synth_features(seed, 1, H4, W4, shift=2)
    sd = O.calibrate_state_dict(O.synth_state_dict(seed), feats, MAXDISP)
    with torch.no_grad():
        ref4, refpv = O.hot_path(sd, *feats, maxdisp=MAXDISP)
    return feats, sd, ref4, refpv


def _check(pred4, pv, ref4, refpv):
    assert pred4.shape == ref4.shape and pv.shape == refpv.shape
    # same ATen ops on row slabs: only the blocking of the conv loops differs (measured: 1e-4 px / 1.4e-5)
    assert float((pred4 - ref4).abs().max()) < 5e-4, float((pred4 - ref4).abs().max())
    assert float((pv - refpv).abs().max()) < 1e-4, float((pv - refpv).abs().max())


def test_row_partition_is_even_aligned_and_covers_the_image():
    assert hs.row_partition(384, 8) == [(48 * r, 48 * (r + 1)) for r in range(8)]     # Middlebury config
    for H4, world in ((20, 3), (16, 4), (96, 8), (136, 8), (12, 1)):
        parts = hs.row_partition(H4, world)
        assert parts[0][0] == 0 and parts[-1][1] == H4
        for (a, b), (c, _) in zip(parts, parts[1:] + [(H4, H4)]):
            assert a % 2 == 0 and b % 2 == 0 and b - a >= 4 and b == c
    with pytest.raises(hs._lib.DcaError):
        hs.row_partition(12, 4)          # fewer than 4 quarter-res rows per rank
    with pytest.raises(hs._lib.DcaError):
        hs.row_partition(13, 2)


def test_rows_request_semantics_in_lockstep():
    # 3 virtual ranks, 4 owned rows + 2 halo rows each side; value = 100*rank + local row
    ts = [torch.arange(8.0).view(1, 8, 1) + 100 * r for r in range(3)]

    def gen(t, fill):
        yield Rows(t, 1, 2, fill=fill)
        return t

    out = hs.drive_lockstep([gen(t.clone(), "zero") for t in ts])
    assert out[0][0, :, 0].tolist() == [0, 0, 2, 3, 4, 5, 102, 103]
    assert out[1][0, :, 0].tolist() == [4, 5, 102, 103, 104, 105, 202, 203]
    assert out[2][0, :, 0].tolist() == [104, 105, 202, 203, 204, 205, 0, 0]
    out = hs.drive_lockstep([gen(t.clone(), "replicate") for t in ts])
    assert out[0][0, :2, 0].tolist() == [2, 2] and out[2][0, 6:, 0].tolist() == [205, 205]

    def gen_border_only(t):
        yield Rows(t, 1, 2, fill="zero", exchange=False)
        return t

    out = hs.drive_lockstep([gen_border_only(t.clone()) for t in ts])
    assert out[1][0, :, 0].tolist() == ts[1][0, :, 0].tolist()          # interior rank untouched
    assert out[0][0, :, 0].tolist() == [0, 0, 2, 3, 4, 5, 6, 7]


def _poison_dead_rows(gen):
    """Before every exchange, NaN the halo rows that do NOT travel (h - live outer rows): the result may not depend on
    them.  (The image-border fill then zeroes them again on the outside; at interior cuts they stay NaN.)"""
    try:
        req = next(gen)
        while True:
            if isinstance(req, Rows) and req.nlive < req.h:
                n, dead = req.t.shape[req.dim], req.h - req.nlive
                req.t.narrow(req.dim, 0, dead).fill_(float("nan"))
                req.t.narrow(req.dim, n - dead, dead).fill_(float("nan"))
            x = yield req
            req = gen.send(x)
    except StopIteration as stop:
        return stop.value


@pytest.mark.parametrize("H4,world", [(16, 2), (20, 3), (16, 4)])
def test_hsharded_plan_matches_unsharded_oracle_virtual_ranks(H4, world):
    feats, sd, ref4, refpv = _case(H4, 24)
    with torch.no_grad():
        gens = [_poison_dead_rows(_oracle_steps(sd, *[hs.owned_rows(f, world, r) for f in feats]))
                for r in range(world)]
        res = hs.drive_lockstep(gens)
    _check(torch.cat([r[0] for r in res], 2), torch.cat([r[1] for r in res], 2), ref4, refpv)


def test_dropping_the_halo_refresh_is_detected():
    """The comparison has teeth: without the interior exchanges the result moves by far more than the tolerance."""
    feats, sd, ref4, _ = _case(16, 24)

    def no_exchange(gen):
        try:
            req = next(gen)
            while True:
                if isinstance(req, Rows):
                    req.exchange = False
                x = yield req
                req = gen.send(x)
        except StopIteration as stop:
            return stop.value

    with torch.no_grad():
        gens = [no_exchange(_oracle_steps(sd, *[hs.owned_rows(f, 2, r) for f in feats])) for r in range(2)]
        res = hs.drive_lockstep(gens)
    err = float((torch.cat([r[0] for r in res], 2) - ref4).abs().max())
    assert not err < 0.05, err          # (a NaN from an emptied class also counts as detected)


def _worker(rank, world, port, q, H4=16):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    feats, sd, ref4, refpv = _case(H4, 24)
    with torch.no_grad():
        gen = _oracle_steps(sd, *[hs.owned_rows(f, world, rank) for f in feats])
        pred4, pv = hs.drive_distributed(gen, rank, world)
    q.put((rank, pred4.numpy(), pv.numpy()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,H4", [(2, 16), (3, 20)])
def test_hsharded_plan_over_gloo(world, H4):
    """world 3: the middle rank exchanges with both neighbours in one grouped send/recv."""
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, H4)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    _, _, ref4, refpv = _case(H4, 24)
    _check(torch.cat([torch.from_numpy(r[1]) for r in res], 2), torch.cat([torch.from_numpy(r[2]) for r in res], 2),
           ref4, refpv)
