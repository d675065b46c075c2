"""Shared helpers for the test-suite (test infrastructure; may import oracle/)."""
import os
import time

import numpy as np
import torch

from oracle import configs, restate

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_MIRRORS = {}


def load_golden(case):
    path = os.path.join(GOLDEN_DIR, case + ".npz")
    z = np.load(path, allow_pickle=False)
    T, B, H, W = [int(v) for v in z["meta"]]
    return dict(z=z, family=str(z["family"]), T=T, B=B, H=H, W=W)


def build_mirror(family, steps, trained=False):
    """The product's plugin model under the golden weight seed (cached per (family, trained); steps is mutable).
    trained=True: the trained-like regime of oracle.configs.trainedify (the `*_trained` goldens).
    Always returned on the CPU: GPU tests move the shared model with .to(device), the CPU tests that follow need it
    back on the host (the head re-packs its engines' weights when their storage changes)."""
    from diffusiondepth_b200.model import get
    if (family, trained) not in _MIRRORS:
        args = configs.make_args(family, steps)
        torch.manual_seed(configs.SEED_WEIGHTS)
        m = get(args)(args).eval()
        _MIRRORS[(family, trained)] = configs.trainedify(m) if trained else m
    m = _MIRRORS[(family, trained)]
    m.depth_head.diffusion_inference_steps = steps
    return m.cpu()


def is_trained_case(case):
    return case in configs.GOLDEN_TRAINED


def weight_checksum(sd):
    keys = sorted(k for k in sd if k.startswith("depth_head.model.") or "conv_inv_transform" in k
                  or k.startswith("depth_head.conv_lateral") or k.endswith("relative_position_bias_table"))
    return float(sum(sd[k].double().abs().sum() for k in keys if sd[k].is_floating_point()))


def golden_view(g, name, full):
    """Sub-sample a full tensor the way make_golden.subsample stored `name`."""
    s = int(g["z"][name + "_stride"])
    if name == "cond":
        return full[:, ::32, ::s, ::s]
    return full[..., ::s, ::s]


def inputs_for(g):
    sample = restate.synthetic_sample(g["B"], g["H"], g["W"], configs.SEED_INPUTS)
    noise = restate.synthetic_noise(g["B"], g["H"], g["W"], configs.SEED_NOISE)
    return sample, noise
