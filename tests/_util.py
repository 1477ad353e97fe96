"""Shared helpers for the tests (fixture loading)."""
import glob
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def load_e2e():
    """Reference-generated 64x128 / maxdisp 48 fixture + the seeded hot-path state_dict it was made with.  The fixture is
    e2e_64x128_d48.npz plus one e2e_64x128_d48.<key>.npz per large array (make_golden.save_split), merged into one dict."""
    from oracle import dcanet_oracle as O
    z = {}
    for fn in sorted(glob.glob(os.path.join(GOLD, "e2e_64x128_d48*.npz"))):
        with np.load(fn) as part:
            z.update({k: part[k] for k in part.files})
    H, W, maxdisp, seed = [int(v) for v in z["meta"]]
    sd = O.synth_state_dict(seed)
    csum = sum(float(v.double().abs().sum()) for v in sd.values() if v.dim() >= 4)
    assert abs(csum - float(z["conv_weight_abs_sum"])) < 1e-6 * csum, "seeded weights differ from fixture"
    for k in z:
        if k.startswith("bn:"):
            sd[k[3:]] = _t(z[k])
    return z, sd, maxdisp
