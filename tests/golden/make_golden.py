"""Generate golden vectors for the hot path FROM THE REFERENCE ITSELF (build container only).

    python tests/golden/make_golden.py            # writes tests/golden/*.npz

Imports /root/reference/models/gwcnet_dca_g.py with the two shims of SURVEY.md section 8c (stub
`models` package because models/__init__.py imports a missing file; stub matplotlib), loads the
repo's seeded synthetic hot-path weights into it, calibrates every BatchNorm with ONE reference
train-mode forward (momentum=1.0), then records the reference's eval forward at every boundary of
SURVEY section 8a.  /root/reference does not exist on the GPU box, so only the resulting fixtures
travel.  Conv weights are not stored (they are regenerated from the seed by
oracle.dcanet_oracle.synth_state_dict; a checksum guards that), BN tensors and the front-end
outputs are.
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference"


def import_reference():
    sys.dont_write_bytecode = True
    pkg = types.ModuleType("models")
    pkg.__path__ = [os.path.join(REF, "models")]
    sys.modules["models"] = pkg
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.image"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.path.insert(0, REF)
    import models.gwcnet_dca_g as ref_model  # noqa
    import models.submodule as ref_sub  # noqa
    return ref_model, ref_sub


def synthetic_pair(seed, H, W, shift):
    g = torch.Generator().manual_seed(seed)
    lo = torch.randn(1, 3, H // 8, W // 8, generator=g)
    left = F.interpolate(lo, size=(H, W), mode="bilinear", align_corners=False)
    left = left + 0.1 * torch.randn(1, 3, H, W, generator=g)
    right = torch.roll(left, -shift, dims=3) + 0.05 * torch.randn(1, 3, H, W, generator=g)
    return left, right


def save_split(stem, arrays, limit=256 * 1024):
    """np.savez_compressed to `<stem>.npz`, except that every array over `limit` bytes goes to its own
    `<stem>.<key>.npz`, so that no fixture file comes near 1 MB (tests/_util.load_e2e merges them)."""
    big = {k: v for k, v in arrays.items() if v.nbytes > limit}
    np.savez_compressed(stem + ".npz", **{k: v for k, v in arrays.items() if k not in big})
    for k, v in big.items():
        np.savez_compressed(f"{stem}.{k}.npz", **{k: v})


def main():
    from oracle import dcanet_oracle as O
    ref_model, ref_sub = import_reference()
    torch.manual_seed(0)
    torch.set_num_threads(8)

    # ---------------- op-level vectors (odd shapes, edge cases) ----------------
    g = torch.Generator().manual_seed(11)
    ops = {}
    for tag, (B, C, G, H, W, D) in {"a": (2, 24, 8, 5, 13, 6), "b": (1, 40, 40, 3, 16, 12),
                                    "c": (1, 320, 40, 4, 20, 7)}.items():
        L = torch.randn(B, C, H, W, generator=g)
        R = torch.randn(B, C, H, W, generator=g)
        if D <= W:  # the reference's slice-assign only works for D <= W
            ops[f"gwc_{tag}_L"], ops[f"gwc_{tag}_R"] = L.numpy(), R.numpy()
            ops[f"gwc_{tag}_meta"] = np.array([D, G])
            ops[f"gwc_{tag}_out"] = ref_sub.build_gwc_volume(L, R, D, G).numpy()
            ops[f"cat_{tag}_out"] = ref_sub.build_concat_volume(L[:, :12], R[:, :12], D).numpy()
    x = torch.randn(2, 12, 6, 10, generator=g)
    ops["regress_in"] = x.numpy()
    ops["regress_out"] = ref_sub.disparity_regression(F.softmax(x, dim=1), 12).numpy()
    np.savez_compressed(os.path.join(HERE, "ops_small.npz"), **ops)

    # ---------------- end-to-end, 64x128 pair, maxdisp 48 ----------------
    H, W, maxdisp, seed = 64, 128, 48, 0
    model = ref_model.GwcNet(maxdisp)
    sd_syn = O.synth_state_dict(seed)
    msd = model.state_dict()
    for k, v in sd_syn.items():
        assert msd[k].shape == v.shape, (k, msd[k].shape, v.shape)
    missing = [k for k in msd if k not in sd_syn and not k.startswith(("feature_extraction.", "guidance."))]
    assert not missing, missing
    model.load_state_dict(sd_syn, strict=False)
    # front end: keep the reference init but give its BNs non-trivial affine params too
    gen = torch.Generator().manual_seed(123)
    for name, m in model.named_modules():
        if isinstance(m, (nn.BatchNorm2d, nn.BatchNorm3d)):
            m.momentum = 1.0
            if name.startswith(("feature_extraction", "guidance")):
                m.weight.data.copy_(torch.rand(m.weight.shape, generator=gen) * 0.5 + 0.75)
                m.bias.data.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)
    left, right = synthetic_pair(seed, H, W, shift=12)
    model.train()
    with torch.no_grad():
        model(left, right, None)            # calibration pass: running stats := batch stats
    model.eval()

    cap = {}

    def hook(name):
        def fn(mod, inp, out):
            cap.setdefault(name, []).append(out)
        return fn

    model.feature_extraction.register_forward_hook(hook("fe"))
    model.guidance.register_forward_hook(hook("guidance"))
    model.dres0.register_forward_hook(hook("dres0"))
    model.classif3.register_forward_hook(hook("classif3"))
    for s in (1, 2, 3):
        c = getattr(model, f"cva{s}")
        c.register_forward_hook(hook(f"cva{s}"))
        c.downsample.register_forward_hook(hook(f"cva{s}.cost_down"))
        c.slc_net.register_forward_hook(hook(f"cva{s}.aug_down"))
        c.fuse.register_forward_hook(hook(f"cva{s}.fused"))
    with torch.no_grad():
        pred4, pv2 = model(left, right, None)

    out = {"meta": np.array([H, W, maxdisp, seed])}
    feL, feR = cap["fe"]
    out["gwc_l"], out["gwc_r"] = feL["gwc_feature"].numpy(), feR["gwc_feature"].numpy()
    out["cat_l"], out["cat_r"] = feL["concat_feature"].numpy(), feR["concat_feature"].numpy()
    out["g"] = cap["guidance"][0]["g"].numpy()
    out["left"], out["right"] = left.numpy(), right.numpy()
    out["dres0"] = cap["dres0"][0].numpy()
    for s in (1, 2, 3):
        logits, aug = cap[f"cva{s}"][0]
        out[f"cva{s}.logits"] = logits.squeeze(1).numpy()
        out[f"cva{s}.class_map"] = F.softmax(logits.squeeze(1), dim=1).argmax(1).numpy().astype(np.int32)
        out[f"cva{s}.out"] = aug.numpy()
        out[f"cva{s}.cost_down"] = cap[f"cva{s}.cost_down"][0].numpy()
        out[f"cva{s}.aug_down"] = cap[f"cva{s}.aug_down"][0].numpy()
        out[f"cva{s}.fused"] = cap[f"cva{s}.fused"][0].numpy()
    out["classif3_logits"] = cap["classif3"][0].squeeze(1).numpy()
    out["pred4"], out["prob_volume2"] = pred4.numpy(), pv2.numpy()
    # BN tensors of the hot path (calibrated by the reference) + conv-weight checksum
    msd = model.state_dict()
    csum = 0.0
    for k in sd_syn:
        leaf = k.rsplit(".", 1)[1]
        if msd[k].dim() >= 4:
            csum += float(msd[k].double().abs().sum())
        elif leaf in ("running_mean", "running_var"):
            out["bn:" + k] = msd[k].numpy()
    out["conv_weight_abs_sum"] = np.array(csum)
    # (front-end weights are NOT stored: 13 MB, out of scope; its outputs above are the inputs)
    save_split(os.path.join(HERE, "e2e_64x128_d48"), out)
    keys = sorted(msd.keys())
    with open(os.path.join(HERE, "state_dict_keys.txt"), "w") as f:
        for k in keys:
            f.write(f"{k} {tuple(msd[k].shape)}\n")
    print("pred4 range", float(pred4.min()), float(pred4.max()), "keys", len(keys))
    for s in (1, 2, 3):
        cm = out[f"cva{s}.class_map"]
        print(f"cva{s} classes used", len(np.unique(cm)), "of", maxdisp // 8)
    for f_ in sorted(os.listdir(HERE)):
        if f_.endswith((".npz", ".txt")):
            print(f_, os.path.getsize(os.path.join(HERE, f_)) // 1024, "KiB")


if __name__ == "__main__":
    main()
