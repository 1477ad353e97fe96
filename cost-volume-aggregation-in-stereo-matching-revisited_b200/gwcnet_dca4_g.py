"""Mirror of the reference's models/gwcnet_dca4_g.py:146-302: four cva stages (built there from cva_bn / submodule_bn, which differ from cva / submodule only in importing the SyncBN names), head classif4; eval returns (pred4 [B,1,H,W], prob_volume4).
Same ctor and 2-argument forward as the reference, same state_dict key layout (tests/golden/state_dict_keys_dca4.txt),
same kernels as the 3-stage model: only the stage graph differs (engine.PackedHotPath reads num_cva / pv_stage)."""
from .gwcnet_dca_g import GwcNet as _GwcNet3
from .gwcnet_dca_g import feature_extraction, hourglass  # noqa: F401  (the reference module defines them too)


class GwcNet(_GwcNet3):
    NUM_CVA = 4
    PV_STAGE = 4
    SQUEEZE_PRED = False

    def forward(self, left, right, disp_true=None, *, confidence=False, lr_check=False, lr_threshold=1.0, hints=None,
                hints_right=None, hint_k=10.0, hint_c=1.0):
        # reference signature: forward(left, right)
        return super().forward(left, right, confidence=confidence, lr_check=lr_check, lr_threshold=lr_threshold,
                               hints=hints, hints_right=hints_right, hint_k=hint_k, hint_c=hint_c)


def GwcNet_G(d):
    return GwcNet(d, use_concat_volume=False)


def GwcNet_GC(d):
    return GwcNet(d, use_concat_volume=True)
