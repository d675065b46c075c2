"""Stochastic DDIM (eta > 0) and the heads' `pipeline` entry point, CPU side: the scheduler's coefficients against the
reference's `DDIMScheduler.step`, the eta restatement against goldens from the reference's own pipeline, the pipeline's
signature and draw order."""
import inspect
import json
import os

import numpy as np
import pytest
import torch

from oracle import configs, restate
import dd_helpers as helpers
import eta_oracle

from diffusiondepth_b200 import EngineError
from diffusiondepth_b200.model.diffusers.schedulers.scheduling_ddim import DDIMScheduler
from diffusiondepth_b200.model.head._pipeline import draw_pipeline_noise
from diffusiondepth_b200.model.registry import HEADS

TOL_Z = 5e-5  # as tests/test_oracle_golden.py
HEAD_TYPES = ["DDIMDepthEstimate_Res", "DDIMDepthEstimate_ResVis", "DDIMDepthEstimate_Swin_ADD",
              "DDIMDepthEstimate_Swin_ADDHAHI", "DDIMDepthEstimate_Swin_ADDHAHIVis", "DDIMDepthEstimate_MPVIT_ADDHAHI"]


def _head(name, steps=5):
    return HEADS.build(dict(type=name, in_channels=[64, 128, 256, 512], inference_steps=steps, num_train_timesteps=1000,
                            depth_feature_dim=16, loss_cfgs=[], init_cfg=None)).eval()


@pytest.mark.parametrize("eta", [0.3, 1.0])
@pytest.mark.parametrize("T", [5, 20, 50])
def test_stochastic_coefficients_reproduce_reference_step(eta, T):
    ref = np.load(os.path.join(helpers.GOLDEN_DIR, "ref_scheduler_eta.npz"), allow_pickle=False)
    k = f"eta{eta}_T{T}_"
    x, eps, z, prev = (torch.from_numpy(ref[k + n]) for n in ("x", "eps", "z", "prev"))
    ts, cx, ce, sg = DDIMScheduler(num_train_timesteps=1000, clip_sample=False).stochastic_coefficients(T, eta)
    assert len(ts) == T and sg[-1] == 0.0 and all(s > 0 for s in sg[:-1])
    for i in range(T):
        got = cx[i] * x[i].double() + ce[i] * eps[i].double() + sg[i] * z[i].double()
        scale = max(1.0, float(prev[i].abs().max()))
        assert (got - prev[i].double()).abs().max().item() < 2e-6 * scale, (i, ts[i])


@pytest.mark.parametrize("T", [5, 20, 50])
def test_stochastic_coefficients_at_eta_zero_are_the_fused_ones(T):
    s = DDIMScheduler(num_train_timesteps=1000, clip_sample=False)
    ts, cx, ce, sg = s.stochastic_coefficients(T, 0.0)
    assert (ts, cx, ce) == tuple(s.fused_coefficients(T))
    assert sg == [0.0] * T


def test_invalid_eta_rejected():
    s = DDIMScheduler(num_train_timesteps=1000, clip_sample=False)
    with pytest.raises(ValueError):
        s.stochastic_coefficients(20, -0.1)
    with pytest.raises(ValueError):
        s.stochastic_coefficients(20, float("nan"))
    with pytest.raises(ValueError):  # 1 - a_prev - sigma^2 < 0: the reference would produce NaN
        s.stochastic_coefficients(20, 3.0)


@pytest.mark.parametrize("case", sorted(eta_oracle.GOLDEN_ETA))
def test_eta_restatement_reproduces_reference_golden(case):
    family, T, B, H, W, eta = eta_oracle.GOLDEN_ETA[case]
    g = helpers.load_golden(case)
    assert float(g["z"]["eta"]) == eta
    m = helpers.build_mirror(family, T)
    sd = m.state_dict()
    ck = helpers.weight_checksum(sd)
    assert abs(ck - float(g["z"]["weight_checksum"])) <= 1e-6 * ck, "weights were not regenerated identically"
    sample, noise = helpers.inputs_for(g)
    z_steps = eta_oracle.synthetic_step_noise(T, B, H, W)
    out = eta_oracle.forward(sd, sample, configs.FAMILIES[family]["backbone_name"], T, noise, eta, z_steps)
    assert (helpers.golden_view(g, "logits", out["logits"]) - torch.from_numpy(g["z"]["logits"])).abs().max().item() < TOL_Z
    lat = helpers.golden_view(g, "latent", out["latent"])
    assert (lat - torch.from_numpy(g["z"]["latent"])).abs().max().item() < 1e-5 * max(1.0, float(g["z"]["latent_absmax"]))
    if "image_list" in g["z"].files:
        s = int(g["z"]["image_list_stride"])
        steps = torch.stack(out["trace"])[..., ::s, ::s]
        ref = torch.from_numpy(g["z"]["image_list"])
        assert ref.shape == steps.shape
        assert (steps - ref).abs().max().item() < 1e-5 * max(1.0, float(ref.abs().max()))
    # the noise matters: the same case without it is far away
    det = restate.ddim_loop(sd, out["cond"], noise, T, "swin" if "swin" in family else "res")
    assert (det - out["latent"]).abs().max().item() > 1e-2


def test_synthetic_step_noise_shards():
    full = eta_oracle.synthetic_step_noise(4, 3, 10, 14)
    assert full.shape == (4, 3, 16, 5, 7)
    assert torch.equal(full[:, 1:], eta_oracle.synthetic_step_noise(4, 2, 10, 14, first=1))


@pytest.mark.parametrize("name", HEAD_TYPES)
def test_every_head_has_the_reference_pipeline(name):
    sig = json.load(open(os.path.join(helpers.GOLDEN_DIR, "ref_pipeline_signature.json")))
    head = _head(name)
    assert str(inspect.signature(type(head.pipeline).__call__)) == sig["vis" if name.endswith("Vis") else "plain"]
    assert head.ddim_eta == 0.0
    cond = torch.randn(1, 256, 4, 6)
    with pytest.raises(EngineError):
        head.pipeline(batch_size=1, device=cond.device, dtype=cond.dtype, shape=(16, 4, 6),
                      input_args=(cond, None, None, None), num_inference_steps=5, return_dict=False)


def test_pipeline_rejects_a_generator_on_another_device():
    head = _head("DDIMDepthEstimate_Res")
    cond = torch.randn(1, 256, 4, 6)
    with pytest.raises(ValueError):
        head.pipeline(1, torch.device("cuda"), torch.float32, (16, 4, 6), (cond, None, None, None),
                      generator=torch.Generator(), num_inference_steps=5)


def test_pipeline_rejects_negative_eta():
    head = _head("DDIMDepthEstimate_Res")
    with pytest.raises(ValueError):
        head.pipeline(1, torch.device("cpu"), torch.float32, (16, 4, 6), (torch.randn(1, 256, 4, 6),), eta=-1.0)


@pytest.mark.parametrize("T", [1, 5])
def test_draw_order_is_the_reference_pipelines(T):
    shape = (2, 16, 3, 5)
    torch.manual_seed(123)
    want = [torch.randn(shape) for _ in range(T + 1)]
    torch.manual_seed(123)
    x_T, steps = draw_pipeline_noise(T, shape, "cpu")
    assert torch.equal(x_T, want[0])
    assert steps.shape == (T, *shape)
    for i in range(T):
        assert torch.equal(steps[i], want[i + 1])
    torch.manual_seed(123)
    x_T0, none = draw_pipeline_noise(T, shape, "cpu", stochastic=False)
    assert none is None and torch.equal(x_T0, want[0])
