"""cva / Multi_Aggregation mirror (reference models/augment/cva.py:13-72)."""
import torch.nn as nn

from . import engine
from .semantic_level import SemanticLevelContext
from .submodule import convbn_3d


class Multi_Aggregation(nn.Module):
    def __init__(self, in_channels):
        super().__init__()
        self.conv1 = nn.Sequential(convbn_3d(in_channels, in_channels * 2, 3, 2, 1), nn.ReLU(inplace=True))
        self.conv2 = nn.Sequential(convbn_3d(in_channels * 2, in_channels * 2, 3, 1, 1), nn.ReLU(inplace=True))
        self.conv3 = nn.Sequential(
            nn.ConvTranspose3d(in_channels * 2, in_channels, 3, padding=1, output_padding=1, stride=2, bias=False),
            nn.BatchNorm3d(in_channels))
        self.redir = convbn_3d(in_channels, in_channels, kernel_size=1, stride=1, pad=0)
        self.precision_planes = 2

    def forward(self, x):
        """x fp32 [B,C,D,H,W] (even D, H, W) -> ReLU(BN(deconv(conv2(conv1 x))) + BN(redir x)) (cva.py:26-31)."""
        engine._require_cuda(x)
        P = self.precision_planes
        pk = engine.cached_pack(self, ("agg", P), lambda: engine.PackedAgg(self, P))
        return engine._result(engine.agg_steps(pk, engine.Planes.from_ncdhw(x, P))).to_ncdhw()


class cva(nn.Module):
    def __init__(self, max_disp, in_channel, downsample=True):
        super().__init__()
        if in_channel != 32:
            raise NotImplementedError("kernels are built for the 32-channel cva DCANet instantiates")
        self.max_disp = max_disp
        self.channel = in_channel
        if downsample:
            self.downsample = nn.Sequential(nn.AvgPool3d((3, 3, 3), stride=2, padding=1),
                                            convbn_3d(32, 32, 3, 1, 1), nn.ReLU(inplace=True))
        self.slc_net = SemanticLevelContext(feats_channels=self.channel, transform_channels=self.channel,
                                            concat_input=True)
        self.classify = nn.Sequential(convbn_3d(self.channel, self.channel, 3, 1, 1), nn.ReLU(inplace=True),
                                      nn.Conv3d(self.channel, 1, kernel_size=3, padding=1, stride=1, bias=False))
        self.fuse = nn.Sequential(convbn_3d(64, 32, 1, 1, 0), )
        self.cost_agg = Multi_Aggregation(self.channel)
        self.precision_planes = 2
        self.last = None

    def forward(self, cost_volume, downsample=True):
        """cost_volume fp32 [B,32,D4,H4,W4] -> (class logits [B,1,D8,H8,W8], augmented cost [B,32,D4,H4,W4])."""
        if not downsample:
            raise NotImplementedError("DCANet always calls cva with downsample=True (gwcnet_dca_g.py:228-232)")
        engine._require_cuda(cost_volume)
        pk = engine.cached_pack(self, ("cva", self.precision_planes),
                                lambda: engine.PackedCva(self, self.precision_planes))
        keep = {}
        cost = engine.Planes.from_ncdhw(cost_volume, self.precision_planes)
        logits, out = engine._result(engine.cva_steps(pk, cost, keep=keep))
        self.last = keep
        return logits.unsqueeze(1), out.to_ncdhw()
