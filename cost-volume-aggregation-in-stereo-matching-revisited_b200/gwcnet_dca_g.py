"""GwcNet (DCANet, 3 cva stages) mirror of the reference's models/gwcnet_dca_g.py: same ctor, same
forward signature, same 726-key state_dict layout, so reference checkpoints load unchanged.
The hot path (feature maps -> disparity) runs entirely in the sm_100a kernels; the 2-D front end
(feature_extraction, Guidance) is ordinary torch (out of scope, SURVEY.md section 2)."""
import torch
import torch.nn as nn

from . import engine
from .cva import cva
from .submodule import BasicBlock, Guidance, PropgationNet_4x, convbn, convbn_3d


class feature_extraction(nn.Module):
    def __init__(self, concat_feature=False, concat_feature_channel=12):
        super().__init__()
        self.concat_feature = concat_feature
        self.inplanes = 32
        self.firstconv = nn.Sequential(convbn(3, 32, 3, 2, 1, 1), nn.ReLU(inplace=True),
                                       convbn(32, 32, 3, 1, 1, 1), nn.ReLU(inplace=True),
                                       convbn(32, 32, 3, 1, 1, 1), nn.ReLU(inplace=True))
        self.layer1 = self._make_layer(BasicBlock, 32, 3, 1, 1, 1)
        self.layer2 = self._make_layer(BasicBlock, 64, 16, 2, 1, 1)
        self.layer3 = self._make_layer(BasicBlock, 128, 3, 1, 1, 1)
        self.layer4 = self._make_layer(BasicBlock, 128, 3, 1, 1, 2)
        if self.concat_feature:
            self.lastconv = nn.Sequential(convbn(320, 128, 3, 1, 1, 1), nn.ReLU(inplace=True),
                                          nn.Conv2d(128, concat_feature_channel, kernel_size=1, padding=0, stride=1,
                                                    bias=False))
        self.frontend_planes = 2        # the front end always runs hi+lo planes (GwcNet.set_precision governs the hot path only)

    def _make_layer(self, block, planes, blocks, stride, pad, dilation):
        downsample = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            downsample = nn.Sequential(nn.Conv2d(self.inplanes, planes * block.expansion, kernel_size=1,
                                                 stride=stride, bias=False),
                                       nn.BatchNorm2d(planes * block.expansion))
        layers = [block(self.inplanes, planes, stride, downsample, pad, dilation)]
        self.inplanes = planes * block.expansion
        layers += [block(self.inplanes, planes, 1, None, pad, dilation) for _ in range(1, blocks)]
        return nn.Sequential(*layers)

    def forward(self, x):
        from . import frontend
        if frontend.use_kernels(self, x) and x.shape[2] % 8 == 0 and x.shape[3] % 8 == 0:
            # CUDA + eval: the 1/4-resolution layers (layer2[1:], layer3, layer4, lastconv) on the tcgen05 2-D conv kernel
            return frontend.feature_extraction_forward(self, x, self.frontend_planes)
        x = self.layer1(self.firstconv(x))
        l2 = self.layer2(x)
        l3 = self.layer3(l2)
        l4 = self.layer4(l3)
        gwc_feature = torch.cat((l2, l3, l4), dim=1)
        if not self.concat_feature:
            return {"gwc_feature": gwc_feature}
        return {"gwc_feature": gwc_feature, "concat_feature": self.lastconv(gwc_feature)}


class hourglass(nn.Module):
    """Full GwcNet hourglass (reference gwcnet_dca_g.py:69-106): defined but never instantiated by
    GwcNet, so it adds no state_dict keys.  Runs on the same conv kernels."""

    def __init__(self, in_channels):
        super().__init__()
        c = in_channels
        self.conv1 = nn.Sequential(convbn_3d(c, c * 2, 3, 2, 1), nn.ReLU(inplace=True))
        self.conv2 = nn.Sequential(convbn_3d(c * 2, c * 2, 3, 1, 1), nn.ReLU(inplace=True))
        self.conv3 = nn.Sequential(convbn_3d(c * 2, c * 4, 3, 2, 1), nn.ReLU(inplace=True))
        self.conv4 = nn.Sequential(convbn_3d(c * 4, c * 4, 3, 1, 1), nn.ReLU(inplace=True))
        self.conv5 = nn.Sequential(nn.ConvTranspose3d(c * 4, c * 2, 3, padding=1, output_padding=1, stride=2,
                                                      bias=False), nn.BatchNorm3d(c * 2))
        self.conv6 = nn.Sequential(nn.ConvTranspose3d(c * 2, c, 3, padding=1, output_padding=1, stride=2,
                                                      bias=False), nn.BatchNorm3d(c))
        self.redir1 = convbn_3d(c, c, kernel_size=1, stride=1, pad=0)
        self.redir2 = convbn_3d(c * 2, c * 2, kernel_size=1, stride=1, pad=0)
        self.precision_planes = 2

    def _pack(self, planes):
        E = engine
        pk = {n: E.pack_convbn(getattr(self, n)[0]) for n in ("conv1", "conv2", "conv3", "conv4")}
        pk["redir1"], pk["redir2"] = E.pack_convbn(self.redir1), E.pack_convbn(self.redir2)
        pk["conv5"] = E.PackedConv(self.conv5[0].weight, self.conv5[1], True)
        pk["conv6"] = E.PackedConv(self.conv6[0].weight, self.conv6[1], True)
        for n, pc in pk.items():      # tcgen05 operand packs where the kernels take the channel counts (32/64)
            pc.pack_tc(planes, transposed=n in ("conv5", "conv6"))
        return pk

    def forward(self, x):
        """x fp32 [B,C,D,H,W] (D, H, W multiples of 4) -> [B,C,D,H,W]; reference gwcnet_dca_g.py:94-106."""
        E = engine
        E._require_cuda(x)
        P = self.precision_planes
        pk = E.cached_pack(self, ("hourglass", P), lambda: self._pack(P))
        return self.forward_planes(E.Planes.from_ncdhw(x, P), pk).to_ncdhw()

    @staticmethod
    def forward_planes(xp, pk):
        """The same on cost planes (used by the plain-GwcNet baseline, gwcnet.py, which chains three of these)."""
        E = engine
        c1 = E.conv(xp, pk["conv1"], E.K3S2, E.ACT_RELU)
        c2 = E.conv(c1, pk["conv2"], E.K3S1, E.ACT_RELU)
        c3 = E.conv(c2, pk["conv3"], E.K3S2, E.ACT_RELU)
        c4 = E.conv(c3, pk["conv4"], E.K3S1, E.ACT_RELU)
        r2 = E.conv(c2, pk["redir2"], E.K1, E.ACT_NONE)
        c5 = E.conv(c4, pk["conv5"], E.T3S2, E.ACT_RELU, res_pre=r2)
        r1 = E.conv(xp, pk["redir1"], E.K1, E.ACT_NONE)
        return E.conv(c5, pk["conv6"], E.T3S2, E.ACT_RELU, res_pre=r1)


class GwcNet(nn.Module):
    """precision: "parity" (hi+lo 16-bit planes, meets |d disp| <= 0.05 px) or "fast" (single 16-bit plane).

    The class constants describe the stage graph; the reference's stage-count variants (gwcnet_dca{0,1,2,4}_g.py)
    subclass this with other values and run the same kernels."""
    NUM_CVA = 3           # cva stages; the head is classif<NUM_CVA>, the heads below it are training-only
    PV_STAGE = 2          # eval returns the class logits of this stage (`prob_volume2`, gwcnet_dca_g.py:282)
    SQUEEZE_PRED = False  # eval returns pred4 [B,1,H,W]; the 0/1/2-stage variants return pred.squeeze(1)

    def __init__(self, maxdisp, use_concat_volume=True, precision="parity"):
        super().__init__()
        self.num_cva, self.pv_stage = self.NUM_CVA, self.PV_STAGE
        assert maxdisp % 8 == 0, "maxdisp must be a multiple of 8 (1/4 volume, 1/8 DCA stage)"
        self.maxdisp = maxdisp
        self.use_concat_volume = use_concat_volume
        self.num_groups = 40
        if self.use_concat_volume:
            self.concat_channels = 12
            self.feature_extraction = feature_extraction(concat_feature=True,
                                                         concat_feature_channel=self.concat_channels)
        else:
            self.concat_channels = 0
            self.feature_extraction = feature_extraction(concat_feature=False)
        self.dres0 = nn.Sequential(convbn_3d(self.num_groups + self.concat_channels * 2, 32, 3, 1, 1),
                                   nn.ReLU(inplace=True), convbn_3d(32, 32, 3, 1, 1), nn.ReLU(inplace=True))
        self.dres1 = nn.Sequential(convbn_3d(32, 32, 3, 1, 1), nn.ReLU(inplace=True), convbn_3d(32, 32, 3, 1, 1))
        for i in range(self.num_cva):
            setattr(self, f"cva{i + 1}", cva(self.maxdisp, 32, downsample=True))
        for i in range(self.num_cva + 1):   # the heads below classif<N> are training-only; kept for the state_dict layout
            setattr(self, f"classif{i}", nn.Sequential(
                convbn_3d(32, 32, 3, 1, 1), nn.ReLU(inplace=True),
                nn.Conv3d(32, 1, kernel_size=3, padding=1, stride=1, bias=False)))
        self.guidance = Guidance(64)
        self.prop = PropgationNet_4x(64)
        self._graphed = None
        self.set_precision(precision)
        self._packed = None

    # ---- precision / packing -------------------------------------------------------------
    def set_precision(self, precision):
        assert precision in ("parity", "fast")
        self.precision = precision
        self._planes = 2 if precision == "parity" else 1
        for m in self.modules():
            if hasattr(m, "precision_planes"):
                m.precision_planes = self._planes
        self._packed = None

    def invalidate(self):
        """Drop the packed kernel parameters (call after mutating weights in place)."""
        self._packed = None

    def _apply(self, fn, *a, **kw):        # .cuda() / .to() / .float() move the weights -> repack
        self._packed = None
        return super()._apply(fn, *a, **kw)

    def packed(self):
        """Pack (once per load) every hot-path parameter for the kernels: BN folded to fp32 scale/shift,
        conv weights to [tap][Cin][Cout] (+ the bf16 operand packs of the tcgen05 kernels)."""
        if self._packed is None or self._packed.planes != self._planes:
            self._packed = engine.PackedHotPath(self, self._planes)
        return self._packed

    def load_state_dict(self, state_dict, strict=True, **kw):
        """Accepts reference checkpoints as saved from nn.DataParallel (`module.` prefix, main_dca.py:277-281)
        and the {'state_dict': ...} wrapper."""
        if "state_dict" in state_dict and not any(k.startswith(("dres0", "module.dres0")) for k in state_dict):
            state_dict = state_dict["state_dict"]
        if any(k.startswith("module.") for k in state_dict):
            state_dict = {(k[7:] if k.startswith("module.") else k): v for k, v in state_dict.items()}
        self._packed = None
        return super().load_state_dict(state_dict, strict=strict, **kw)

    # ---- forward -------------------------------------------------------------------------
    def hot_path(self, gwc_l, gwc_r, cat_l, cat_r, g, keep=None, confidence=False):
        """feature maps -> (pred4 [B,1,H,W], prob_volume2 [B,D8,H8,W8]); the graded path.  confidence=True adds a third
        item, `Confidence(peak, std)` (fp32 [B,1,H,W] each, include/dca_b200.h section 4); pred4 and prob_volume2 stay
        bit-identical."""
        return engine.hot_path_forward(self.packed(), gwc_l, gwc_r, cat_l, cat_r, g, keep, confidence)

    def hot_path_graphed(self, gwc_l, gwc_r, cat_l, cat_r, g, confidence=False):
        """`hot_path` as one CUDA graph per set of input buffers (captured on first use, replayed afterwards; the inputs
        are read in place, results are returned as copies).  Same kernels, same results, one launch.  Graphs (and their
        shared activation pool) are kept per CALLING stream, so forwards replayed concurrently on several streams do not
        share buffers.  With and without `confidence` are two graphs."""
        return self.graphed()(gwc_l, gwc_r, cat_l, cat_r, g, confidence)

    def graphed(self):
        """The `engine.GraphedHotPath` of the current stream (created on first use; dropped with the packed parameters)."""
        pk = self.packed()
        if self._graphed is None or self._graphed[0] is not pk:
            self._graphed = (pk, {})
        sid = torch.cuda.current_stream().cuda_stream
        gh = self._graphed[1].get(sid)
        if gh is None:
            gh = self._graphed[1][sid] = engine.GraphedHotPath(pk)
        return gh

    def hot_path_hsharded(self, gwc_l, gwc_r, cat_l, cat_r, g, rank, world, group=None, transport="nccl"):
        """One rank of the H-sharded single-pair mode (BASELINE configs[4]): this rank's OWNED 1/4-res rows of the
        feature maps in (`hshard.owned_rows`), its rows of (pred4, prob_volume2) out; halo rows and the per-class sums
        travel over torch.distributed.  See hshard.py for the plan and its verification status."""
        from . import hshard
        return hshard.hot_path_forward_hsharded(self.packed(), gwc_l, gwc_r, cat_l, cat_r, g, rank, world, group,
                                                transport)

    def forward(self, left, right, disp_true=None, *, confidence=False, lr_check=False, lr_threshold=1.0):
        """(pred, prob_volume) as the reference's eval forward; confidence=True adds `Confidence(peak, std)`, shaped like
        pred (squeezed with it in the 0/1/2-stage variants).  lr_check=True appends, last, `LRCheck(disp_right, label,
        filled)` of the left-right consistency check with threshold `lr_threshold` px (include/dca_b200.h section 8),
        each shaped like pred: the right view runs in the same forward as the mirrored pair (flip(R), flip(L)), at twice
        the batch, and pred / prob_volume / Confidence are those of the forward without the flag."""
        if self.training:
            raise NotImplementedError("dcanet_b200 is an inference engine: call .eval() (training-mode heads "
                                      "classif0-2 exist only so checkpoints load)")
        from . import frontend
        B = left.shape[0]
        nb = 2 * B if lr_check else B       # pairs through the hot path
        with frontend._no_tf32():          # whatever part of the front end runs on cuDNN runs in true fp32
            if lr_check:                   # left references (L, flip(R)), right images (R, flip(L)): one 4B front end
                imgs = torch.cat((left, right.flip(-1), right, left.flip(-1)), dim=0)
                f = self.feature_extraction(imgs)
                g = self.guidance(imgs[:nb])["g"]
            else:
                f = self.feature_extraction(torch.cat((left, right), dim=0))      # eval-mode BN: batching changes nothing
                g = self.guidance(left)["g"]
        gwc, cat = f["gwc_feature"], f.get("concat_feature")
        out = self.hot_path(gwc[:nb], gwc[nb:], None if cat is None else cat[:nb], None if cat is None else cat[nb:], g,
                            confidence=confidence)
        sq = (lambda t: t.squeeze(1)) if self.SQUEEZE_PRED else (lambda t: t)
        left_view = (lambda t: t[:B]) if lr_check else (lambda t: t)
        pred, pv = out[0], out[1]
        res = [sq(left_view(pred)), left_view(pv)]
        if confidence:
            conf = out[2]
            res.append(engine.Confidence(sq(left_view(conf.peak)), sq(left_view(conf.std))))
        if lr_check:
            label, filled, right_disp = engine.lr_consistency(pred[:B], pred[B:], lr_threshold, mirrored=True,
                                                              want_right=True)
            res.append(engine.LRCheck(sq(right_disp), sq(label), sq(filled)))
        return tuple(res)
