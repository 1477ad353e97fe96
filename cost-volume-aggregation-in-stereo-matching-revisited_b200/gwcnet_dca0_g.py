"""Mirror of the reference's models/gwcnet_dca0_g.py:107-190: no cva stage: dres0/dres1 -> classif0 -> regression -> prop; eval returns (pred0.squeeze(1), the classif0 logits [B,D/4,H/4,W/4]).
Same ctor and 2-argument forward as the reference, same state_dict key layout (tests/golden/state_dict_keys_dca0.txt),
same kernels as the 3-stage model: only the stage graph differs (engine.PackedHotPath reads num_cva / pv_stage)."""
from .gwcnet_dca_g import GwcNet as _GwcNet3
from .gwcnet_dca_g import feature_extraction, hourglass  # noqa: F401  (the reference module defines them too)


class GwcNet(_GwcNet3):
    NUM_CVA = 0
    PV_STAGE = 0
    SQUEEZE_PRED = True

    def forward(self, left, right, disp_true=None, *, confidence=False, lr_check=False, lr_threshold=1.0):
        # reference signature: forward(left, right)
        return super().forward(left, right, confidence=confidence, lr_check=lr_check, lr_threshold=lr_threshold)


def GwcNet_G(d):
    return GwcNet(d, use_concat_volume=False)


def GwcNet_GC(d):
    return GwcNet(d, use_concat_volume=True)
