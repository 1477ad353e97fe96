"""Mirror of the reference's models/gwcnet_dca2_g.py:110-235: two cva stages, head classif2; eval returns (pred2.squeeze(1), prob_volume2).
Same ctor and 2-argument forward as the reference, same state_dict key layout (tests/golden/state_dict_keys_dca2.txt),
same kernels as the 3-stage model: only the stage graph differs (engine.PackedHotPath reads num_cva / pv_stage)."""
from .gwcnet_dca_g import GwcNet as _GwcNet3
from .gwcnet_dca_g import feature_extraction, hourglass  # noqa: F401  (the reference module defines them too)


class GwcNet(_GwcNet3):
    NUM_CVA = 2
    PV_STAGE = 2
    SQUEEZE_PRED = True

    def forward(self, left, right, disp_true=None, *, confidence=False, lr_check=False, lr_threshold=1.0, hints=None,
                hints_right=None, hint_k=10.0, hint_c=1.0):
        # reference signature: forward(left, right)
        return super().forward(left, right, confidence=confidence, lr_check=lr_check, lr_threshold=lr_threshold,
                               hints=hints, hints_right=hints_right, hint_k=hint_k, hint_c=hint_c)


def GwcNet_G(d):
    return GwcNet(d, use_concat_volume=False)


def GwcNet_GC(d):
    return GwcNet(d, use_concat_volume=True)
