"""Module-level (function-level API) forwards on the GPU against the SAME torch modules evaluated on the CPU in fp32:
the mirror classes are parameter containers built from ordinary torch layers, so calling those layers the way the
reference's forward does (gwcnet_dca_g.py:94-124, cva.py:26-31, SelfAttention_bn.py:62-98, submodule.py:121-131) is the
reference computation.  Also the op-level tests of the kernels the default route actually ships (dca_up2_tc kinds 0/1/2,
dca_conv1_taps_tc + dca_tap_gather3d) at odd shapes."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _mods():
    import dcanet_b200 as d
    return d, d.engine


def _init(mod, seed):
    """Unit-scale random weights and non-trivial BN statistics (eval mode)."""
    g = torch.Generator().manual_seed(seed)
    for m in mod.modules():
        if isinstance(m, (torch.nn.Conv3d, torch.nn.Conv2d, torch.nn.ConvTranspose3d)):
            fan = m.weight[0].numel() if not isinstance(m, torch.nn.ConvTranspose3d) else m.weight.shape[0] * 27 / 8
            m.weight.data.copy_(torch.randn(m.weight.shape, generator=g) / fan ** 0.5)
        elif isinstance(m, (torch.nn.BatchNorm3d, torch.nn.BatchNorm2d)):
            m.weight.data.copy_(torch.rand(m.weight.shape, generator=g) * 0.5 + 0.75)
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) * 0.5 + 0.75)
    return mod.eval()


def close(got, ref, rel, what):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err = float((got - ref).abs().max())
    scale = float(ref.abs().max()) + 1e-12
    assert err <= rel * scale + 1e-7, f"{what}: max err {err:.3e} vs scale {scale:.3e}"


def rnd(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


# ---------------------------------------------------------------------------------------------------------
def test_self_attention_block_two_input_forward():
    """SelfAttentionBlock.forward(query_feats, key_feats), SelfAttention_bn.py:62-98, on un-related query / key tensors."""
    d, E = _mods()
    blk = _init(d.SemanticLevelContext(32, 32).cross_attention, 3)
    for (B, D, H, W) in ((1, 24, 5, 7), (2, 6, 3, 5), (1, 30, 2, 9), (1, 48, 2, 3)):
        q, k = rnd(B, 32, D, H, W, seed=D), rnd(B, 32, D, H, W, seed=D + 1)
        with torch.no_grad():
            def proj(seq, x):
                return seq(x)
            qq = proj(blk.query_project, q).reshape(B, 4, 8, D, H * W).permute(0, 4, 1, 3, 2)      # [B,P,head,D,8]
            kk = proj(blk.key_project, k).reshape(B, 4, 8, D, H * W).permute(0, 4, 1, 2, 3)        # [B,P,head,8,D]
            vv = proj(blk.value_project, k).reshape(B, 4, 8, D, H * W).permute(0, 4, 1, 3, 2)
            sim = torch.softmax(torch.matmul(qq, kk) * (8 ** -0.5), dim=-1)
            ctx = torch.matmul(sim, vv)                                                             # [B,P,head,D,8]
            ctx = ctx.permute(0, 2, 4, 3, 1).reshape(B, 32, D, H, W)
            ref = blk.out_project(ctx)
            got = blk.cuda()(q.cuda(), k.cuda())
        blk.cpu()
        close(got, ref, 3e-4, f"self attention D={D}")


def test_self_attention_block_matches_oracle_attention():
    """Same entry point against the oracle's disparity_attention (the pinned restatement of the reference)."""
    d, E = _mods()
    from oracle import dcanet_oracle as O
    sd = O.synth_state_dict(5)
    pref = "cva1.slc_net.cross_attention."
    blk = d.SemanticLevelContext(32, 32).cross_attention
    blk.load_state_dict({k[len(pref):]: v for k, v in sd.items() if k.startswith(pref)})
    q, k = rnd(1, 32, 24, 4, 6, seed=1), rnd(1, 32, 24, 4, 6, seed=2)
    with torch.no_grad():
        ref = O.disparity_attention(O._Ctx(sd), pref[:-1], q, k)
        got = blk.cuda().eval()(q.cuda(), k.cuda())
    close(got, ref, 3e-4, "attention vs oracle")


def test_disparity_regression_is_plain_weighted_sum():
    """submodule.py:127-131: sum_d d * x[d]; un-normalised (even negative) input is NOT renormalised."""
    d, E = _mods()
    x = rnd(2, 12, 5, 9, seed=4)
    ref = torch.sum(x * torch.arange(12, dtype=x.dtype).view(1, 12, 1, 1), 1, keepdim=True)
    close(d.disparity_regression(x.cuda(), 12), ref, 1e-6, "disparity_regression")
    p = torch.softmax(x, 1)
    ref = torch.sum(p * torch.arange(12, dtype=x.dtype).view(1, 12, 1, 1), 1, keepdim=True)
    close(d.disparity_regression(p.cuda(), 12), ref, 1e-6, "disparity_regression(prob)")
    close(d.softmax_disparity_regression(x.cuda(), 12), ref, 1e-5, "softmax_disparity_regression")


@pytest.mark.parametrize("shape", [(1, 8, 12, 16), (2, 4, 8, 24), (1, 12, 20, 8)])
def test_multi_aggregation_module_forward(shape):
    d, E = _mods()
    B, D, H, W = shape
    m = _init(d.Multi_Aggregation(32), 7)
    x = rnd(B, 32, D, H, W, seed=1)
    with torch.no_grad():
        c2 = m.conv2(m.conv1(x))
        ref = F.relu(m.conv3(c2) + m.redir(x))
        got = m.cuda()(x.cuda())
        got2 = m(x.cuda())                      # second call: cached pack
    close(got, ref, 3e-4, "Multi_Aggregation")
    assert torch.equal(got, got2)
    assert len(m._dca_packs) == 1


def test_multi_aggregation_repacks_after_weight_change():
    d, E = _mods()
    m = _init(d.Multi_Aggregation(32), 8).cuda()
    x = rnd(1, 32, 4, 8, 8, seed=1).cuda()
    with torch.no_grad():
        a = m(x)
        m.redir[0].weight.mul_(2.0)             # in-place change bumps the version -> repack
        b = m(x)
        ref = F.relu(m.conv3(m.conv2(m.conv1(x))) + m.redir(x))
    assert not torch.equal(a, b)
    close(b, ref, 3e-4, "Multi_Aggregation after in-place weight change")


def test_hourglass_module_forward():
    d, E = _mods()
    m = _init(d.hourglass(32), 9)
    x = rnd(1, 32, 8, 16, 24, seed=2)
    with torch.no_grad():
        c1 = m.conv1(x); c2 = m.conv2(c1); c3 = m.conv3(c2); c4 = m.conv4(c3)
        c5 = F.relu(m.conv5(c4) + m.redir2(c2))
        ref = F.relu(m.conv6(c5) + m.redir1(x))
        got = m.cuda()(x.cuda())
    close(got, ref, 5e-4, "hourglass")


def test_propagation_net_module_forward():
    """PropgationNet_4x.forward (gwcnet_dca_g.py:117-124) through the tcgen05 2-D convs + convex upsample."""
    d, E = _mods()
    m = _init(d.PropgationNet_4x(64), 10)
    B, H, W = 2, 12, 20
    g, disp = rnd(B, 64, H, W, seed=3), rnd(B, 1, H, W, seed=4).abs() * 10
    with torch.no_grad():
        mask = m.conv(g).view(B, 1, 9, 4, 4, H, W)
        mask = torch.softmax(mask, dim=2)
        up = F.unfold(4 * disp, [3, 3], padding=1).view(B, 1, 9, 1, 1, H, W)
        ref = torch.sum(mask * up, dim=2).permute(0, 1, 4, 2, 5, 3).reshape(B, 1, 4 * H, 4 * W)
        got = m.cuda()(g.cuda(), disp.cuda())
    close(got, ref, 3e-4, "PropgationNet_4x")


@pytest.mark.parametrize("cin,cout,k,s", [(32, 32, 3, 1), (64, 32, 3, 1), (32, 64, 3, 2), (64, 64, 3, 1), (32, 32, 1, 1)])
def test_run_convbn_3d(cin, cout, k, s):
    d, E = _mods()
    from importlib import import_module
    sub = import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.submodule")
    seq = _init(sub.convbn_3d(cin, cout, k, s, 1 if k == 3 else 0), 11)
    x = rnd(1, cin, 6, 10, 12, seed=5)
    with torch.no_grad():
        ref = F.relu(seq(x))
        got = sub.run_convbn_3d(seq.cuda(), x.cuda(), act=E.ACT_RELU)
    close(got, ref, 3e-4, f"convbn_3d {cin}->{cout} k{k} s{s}")


# --------------------------------------------------------------------------------------------------------- op level
@pytest.mark.parametrize("pair", [1, 0])
@pytest.mark.parametrize("B,Dl,Hl,Wl,with_res", [(1, 3, 5, 7, False), (2, 2, 17, 9, True), (1, 5, 16, 8, True), (1, 1, 1, 1, False),
                                                 (1, 6, 40, 30, True)])
def test_up2_kind0_transposed_conv_plus_redir(B, Dl, Hl, Wl, with_res, pair):
    """dca_up2_tc kind 0 = ReLU(BN(ConvTranspose3d(x)) + BN(redir(side))) + res_post (cva.py:20-31), the kernel
    cva_steps ships, at shapes that are not multiples of the 8x16 tile."""
    d, E = _mods()
    m = _init(d.Multi_Aggregation(32), 12)
    x, side = rnd(B, 64, Dl, Hl, Wl, seed=1), rnd(B, 32, 2 * Dl, 2 * Hl, 2 * Wl, seed=2)
    res = rnd(B, 32, 2 * Dl, 2 * Hl, 2 * Wl, seed=3) if with_res else None
    with torch.no_grad():
        ref = F.relu(m.conv3(x) + m.redir(side))
        if res is not None:
            ref = ref + res
        m.cuda()
        pk = E.PackedAgg(m, 2)
        assert pk.conv3_fused is not None
        fd = pk.conv3_fused
        d._lib.call("dca_tc_set_deconv_pair", pair)       # 1: two depth-adjacent tiles per weight fetch, 0: the up2 kernel
        try:
            got = E.up2(0, E.Planes.from_ncdhw(x.cuda(), 2), E.Planes.from_ncdhw(side.cuda(), 2), fd.w_tc, fd.scale, fd.shift,
                        E.ACT_RELU, 64, Dl, Hl, Wl, res_post=E.Planes.from_ncdhw(res.cuda(), 2) if with_res else None)
            torch.cuda.synchronize()
        finally:
            d._lib.call("dca_tc_set_deconv_pair", 1)
    close(got.to_ncdhw(), ref, 3e-4, "up2 kind 0")


@pytest.mark.parametrize("B,Dl,Hl,Wl", [(1, 3, 5, 7), (2, 2, 17, 9), (1, 6, 16, 8)])
@pytest.mark.parametrize("bilinear", [False, True])
def test_up2_kinds_1_2_trilinear_cat_fuse(B, Dl, Hl, Wl, bilinear):
    """dca_up2_tc kind 1 / kind 2 = BN(fuse(cat(trilinear_x2(t), cost))) (cva.py:64,55,69) with t = Wa . aug as the
    attention kernel hands it over (padded / depth-interpolated layouts built here with torch)."""
    d, E = _mods()
    c = _init(d.cva(192, 32), 13).cuda()
    pk = E.PackedCva(c, 2)
    aug, cost = rnd(B, 32, Dl, Hl, Wl, seed=1), rnd(B, 32, 2 * Dl, 2 * Hl, 2 * Wl, seed=2)
    with torch.no_grad():
        c.cpu()
        up = F.interpolate(aug, scale_factor=(2, 2, 2), mode="trilinear")
        ref = c.fuse(torch.cat((up, cost), 1))
        wa = c.fuse[0][0].weight[:, :32, 0, 0, 0]                        # t = Wa . aug (linear: commutes with the upsampling)
        t = torch.einsum("oc,bcdhw->bodhw", wa, aug)
        if bilinear:
            tz = F.interpolate(t, scale_factor=(2, 1, 1), mode="trilinear")   # depth axis resolved upstream
            tp = F.pad(tz, (1, 1, 1, 1, 0, 0), mode="replicate")
            got = E.up2(2, E.Planes.from_ncdhw(tp.cuda(), 2), E.Planes.from_ncdhw(cost.cuda(), 2), pk.fuse_up2b_w,
                        pk.fuse_scale, pk.fuse_shift, E.ACT_NONE, 32, 2 * Dl, Hl, Wl)
        else:
            tp = F.pad(t, (1, 1, 1, 1, 1, 1), mode="replicate")
            got = E.up2(1, E.Planes.from_ncdhw(tp.cuda(), 2), E.Planes.from_ncdhw(cost.cuda(), 2), pk.fuse_up2_w,
                        pk.fuse_scale, pk.fuse_shift, E.ACT_NONE, 32, Dl, Hl, Wl)
    close(got.to_ncdhw(), ref, 3e-4, "up2 kind %d" % (2 if bilinear else 1))


def test_up2_rejects_mismatched_side():
    d, E = _mods()
    m = _init(d.Multi_Aggregation(32), 12).cuda()
    fd = E.PackedAgg(m, 2).conv3_fused
    x = E.Planes.from_ncdhw(rnd(1, 64, 2, 3, 4).cuda(), 2)
    side = E.Planes.from_ncdhw(rnd(1, 32, 4, 7, 8).cuda(), 2)            # 7 rows instead of 6
    with pytest.raises(d._lib.DcaError):
        E.up2(0, x, side, fd.w_tc, fd.scale, fd.shift, E.ACT_RELU, 64, 2, 3, 4)


@pytest.mark.parametrize("B,D,H,W", [(1, 6, 8, 12), (2, 4, 6, 8), (1, 24, 12, 10), (1, 3, 16, 8)])
def test_cout1_conv_tensor_core_route(B, D, H, W):
    """Conv3d(32 -> 1, k3, p1) as dca_conv1_taps_tc + dca_tap_gather3d (the route engine.conv_cout1_any takes when
    B*D*H*W % 8 == 0) against torch and against the CUDA-core kernel."""
    d, E = _mods()
    assert (B * D * H * W) % 8 == 0
    w = rnd(1, 32, 3, 3, 3, seed=6) * 0.1
    x = rnd(B, 32, D, H, W, seed=7)
    ref = F.conv3d(x, w, padding=1)[:, 0]
    xp = E.Planes.from_ncdhw(x.cuda(), 2)
    pc = E.PackedCout1(w.cuda(), 2)
    assert pc.w_tc is not None
    got = E.conv_cout1_any(xp, pc)
    close(got, ref, 2e-5, "32->1 tensor-core route")
    close(E.conv_cout1(xp, pc.host), ref, 2e-5, "32->1 CUDA-core route")


@pytest.mark.parametrize("cin,B,D,H,W,march", [(32, 1, 6, 8, 12, False), (32, 1, 24, 40, 72, True), (64, 1, 9, 17, 21, False),
                                               (32, 2, 5, 33, 9, False), (32, 1, 17, 48, 104, True), (64, 1, 20, 36, 100, True)])
def test_fused_tail_conv_taps27(cin, B, D, H, W, march):
    """dca_conv3d_tc_taps27 + dca_tap_gather3d == Conv3d(32->1,k3)(ReLU(BN(Conv3d(cin->32,k3)(x)))) (classif3
    gwcnet_dca_g.py:166-168, cva.classify cva.py:51-53) on both kernels (halo-slab and depth-marching), ragged shapes;
    and the fused gather + softmax + regression against torch on the same logits."""
    d, E = _mods()
    from importlib import import_module
    sub = import_module("cost-volume-aggregation-in-stereo-matching-revisited_b200.submodule")
    head = _init(torch.nn.Sequential(sub.convbn_3d(cin, 32, 3, 1, 1), torch.nn.ReLU(),
                                     torch.nn.Conv3d(32, 1, 3, padding=1, bias=False)), 21)
    x = rnd(B, cin, D, H, W, seed=8)
    with torch.no_grad():
        ref = head(x)[:, 0]
        ref_pred = torch.sum(torch.softmax(ref, 1) * torch.arange(D, dtype=ref.dtype).view(1, D, 1, 1), 1, keepdim=True)
    head.cuda()
    pc = E.pack_convbn(head[0])
    assert pc.pack_tc(2)
    pc1 = E.PackedCout1(head[2].weight, 2)
    xp = E.Planes.from_ncdhw(x.cuda(), 2)
    saved = E.Options.march_min_items
    E.Options.march_min_items = 0 if march else 1 << 30          # pick the kernel under test regardless of the size
    try:
        P = E.conv_taps27(xp, pc, pc1)
    finally:
        E.Options.march_min_items = saved
    assert P is not None and P.shape == (27, B, D, H, W)
    close(E.tap_gather(P), ref, 3e-5, "fused tail logits")
    pred, lg = E.tap_gather_softmax_regress(P, want_logits=True)
    close(lg, ref, 3e-5, "fused tail logits (fused gather)")
    close(pred, ref_pred, 1e-4, "fused tail regression")
    pred2, none = E.tap_gather_softmax_regress(P)
    assert none is None and torch.equal(pred, pred2)
