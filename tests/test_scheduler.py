"""DDIM scheduler mirror: tables, timesteps, step and the collapsed coefficients the CUDA loop uses
(reference src/model/diffusers/schedulers/scheduling_ddim.py; probe values from SURVEY.md §3.3)."""
import math
import os

import numpy as np
import pytest
import torch

from diffusiondepth_b200 import ddim_coefficients
from diffusiondepth_b200.model.diffusers.schedulers.scheduling_ddim import DDIMScheduler
from oracle import make_golden, restate
import dd_helpers as helpers


def test_tables_and_timesteps():
    s = DDIMScheduler(num_train_timesteps=1000, clip_sample=False)
    assert torch.equal(s.alphas_cumprod, restate.ddim_tables())
    for T, first in ((20, 950), (5, 800), (50, 980)):
        s.set_timesteps(T)
        assert s.timesteps.tolist() == restate.ddim_timesteps(T)
        assert s.timesteps[0].item() == first and s.timesteps[-1].item() == 0
    assert s.config.num_train_timesteps == 1000 and s.num_train_timesteps == 1000


def test_survey_probe_values():
    s = DDIMScheduler()
    ts, cx, ce = s.fused_coefficients(20)
    assert abs(float(s.alphas_cumprod[950]) - 1.06e-4) < 2e-6
    assert abs(cx[0] - 1.5964) < 1e-3 and abs(ce[0] + 0.5964) < 1e-3
    assert abs(cx[-1] - 1.00005) < 1e-5 and abs(ce[-1] + 0.010001) < 1e-5
    ts5, cx5, ce5 = s.fused_coefficients(5)
    assert abs(cx5[0] - 4.118) < 2e-3 and abs(ce5[0] + 3.128) < 2e-3
    assert ddim_coefficients(s.alphas_cumprod, 20, 1000)[1] == pytest.approx(cx)


@pytest.mark.parametrize("T", [5, 20, 50])
def test_collapsed_update_equals_three_expression_step(T):
    """x_{t-1} = c_x x + c_eps eps reproduces DDIMScheduler.step (eta=0) to fp32 rounding."""
    s = DDIMScheduler()
    ts, cx, ce = s.fused_coefficients(T)
    g = torch.Generator().manual_seed(T)
    x = torch.randn(2, 16, 12, 20, generator=g, dtype=torch.float64) * 30
    acp = restate.ddim_tables()
    for t, a, b in zip(ts, cx, ce):
        eps = torch.rand(x.shape, generator=g, dtype=torch.float64) * 3
        full = s.step(eps, t, x, eta=0.0, use_clipped_model_output=True)["prev_sample"]
        oracle = restate.ddim_step(eps, t, x, acp, T)
        fused = a * x + b * eps
        scale = full.abs().max().item()
        assert (full - oracle).abs().max().item() <= 1e-6 * scale  # fp32 vs fp64 sqrt of the table entries
        x32, e32 = x.float(), eps.float()
        assert torch.equal(s.step(e32, t, x32, eta=0.0, use_clipped_model_output=True)["prev_sample"],
                           restate.ddim_step(e32, t, x32, acp, T))  # identical in the reference's own fp32
        assert (full - fused).abs().max().item() <= 1e-6 * scale  # table is fp32, algebra exact
        x = full


def test_add_noise_and_sample_prediction():
    s = DDIMScheduler()
    x0 = torch.randn(3, 16, 4, 4)
    n = torch.randn(3, 16, 4, 4)
    t = torch.tensor([0, 500, 999])
    y = s.add_noise(x0, n, t)
    a = restate.ddim_tables()[t].view(3, 1, 1, 1)
    assert torch.allclose(y, a.sqrt() * x0 + (1 - a).sqrt() * n, atol=1e-6)
    with pytest.raises(ValueError):
        DDIMScheduler().step(n, 10, x0)


def test_against_reference_scheduler():
    """Bit for bit against the reference's DDIMScheduler on the seeded chain of oracle.make_golden.fixture_scheduler
    (tests/golden/ref_scheduler.npz: every step as a sha256 of its float32 bytes, the last step in full)."""
    ref = np.load(os.path.join(helpers.GOLDEN_DIR, "ref_scheduler.npz"), allow_pickle=False)
    mine = DDIMScheduler(num_train_timesteps=1000, clip_sample=False)
    assert torch.equal(torch.from_numpy(ref["alphas_cumprod"]), mine.alphas_cumprod)
    g = torch.Generator().manual_seed(3)
    for T in (5, 20, 50):
        mine.set_timesteps(T)
        assert torch.equal(torch.from_numpy(ref[f"T{T}_timesteps"]), mine.timesteps)
        x = torch.randn(1, 16, 6, 10, generator=g)
        for i, t in enumerate(mine.timesteps):
            eps = torch.rand(x.shape, generator=g)
            b = mine.step(eps, t, x, eta=0.0, use_clipped_model_output=True)
            assert make_golden.digest(b["prev_sample"]) == ref[f"T{T}_prev_sample_sha256"][i], (T, i)
            assert make_golden.digest(b["pred_original_sample"]) == ref[f"T{T}_pred_original_sha256"][i], (T, i)
            x = b["prev_sample"]
        assert torch.equal(x, torch.from_numpy(ref[f"T{T}_last_prev_sample"]))
        assert torch.equal(b["pred_original_sample"], torch.from_numpy(ref[f"T{T}_last_pred_original"]))
    t = torch.tensor([7, 300])
    x0, n = torch.randn(2, 16, 3, 3, generator=g), torch.randn(2, 16, 3, 3, generator=g)
    assert torch.equal(mine.add_noise(x0, n, t), torch.from_numpy(ref["add_noise"]))
