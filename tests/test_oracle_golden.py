"""Pin the CPU restatement (oracle/restate.py) and the mirror's step-invariant producers against golden
vectors generated from the REAL reference (oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import configs, make_golden, restate
import dd_helpers as helpers

TOL_Z = 5e-5  # fp32-vs-fp32 re-association noise on the logits (SURVEY.md §7.2: 3e-5 vs fp64 over 20 steps)


@pytest.mark.parametrize("case", ["g_res18_c1", "g_res18_ragged", "g_mpvit_small", "g_mpvit_trained", "g_res18_trained",
                                  "g_swinl_small_trained", "g_swinl_odd_trained", "g_res18_vis_trained"])
def test_oracle_reproduces_reference_golden(case):
    """`*_trained`: the trained-like regime (oracle.configs.trainedify: random non-zero Swin relative-position tables,
    non-trivial BatchNorm running statistics, LayerNorm / GroupNorm affines) — what released checkpoints look like."""
    g = helpers.load_golden(case)
    m = helpers.build_mirror(g["family"], g["T"], helpers.is_trained_case(case))
    sd = m.state_dict()
    ck = helpers.weight_checksum(sd)
    assert abs(ck - float(g["z"]["weight_checksum"])) <= 1e-6 * ck, "weights were not regenerated identically"
    sample, noise = helpers.inputs_for(g)
    out = restate.forward(sd, sample, configs.FAMILIES[g["family"]]["backbone_name"], g["T"], noise)
    z_ref = torch.from_numpy(g["z"]["logits"])
    assert (helpers.golden_view(g, "logits", out["logits"]) - z_ref).abs().max().item() < TOL_Z
    lat_ref = torch.from_numpy(g["z"]["latent"])
    lat = helpers.golden_view(g, "latent", out["latent"])
    assert (lat - lat_ref).abs().max().item() < 1e-5 * max(1.0, float(g["z"]["latent_absmax"]))
    cond_ref = torch.from_numpy(g["z"]["cond"])
    assert (helpers.golden_view(g, "cond", out["cond"]) - cond_ref).abs().max().item() < 1e-5 * float(g["z"]["cond_absmax"])
    # depth itself, where exp(-z) is well conditioned
    pm = restate.parity_metrics(helpers.golden_view(g, "logits", out["logits"]), z_ref,
                                helpers.golden_view(g, "pred", out["pred"]), torch.from_numpy(g["z"]["pred"]))
    assert pm["max_rel_depth_wellcond"] < 1e-3
    assert sorted(str(k) for k in g["z"]["output_keys"]) == sorted([
        'aff', 'blur_depth_t', 'confidence', 'ddim_loss', 'gamma', 'gt_map_t', 'guidance', 'offset', 'pred',
        'pred_init', 'pred_inter', 'pred_uncertainty', 'weight_map'])


@pytest.mark.parametrize("case", ["g_res18_c1", "g_res18_ragged", "g_mpvit_small", "g_mpvit_trained", "g_res18_trained",
                                  "g_swinl_small_trained", "g_swinl_odd_trained"])
def test_mirror_producers_match_reference_condition(case):
    """backbone + FPN of the product mirror (torch ops, once per image) reproduce the reference's cond map."""
    g = helpers.load_golden(case)
    m = helpers.build_mirror(g["family"], g["T"], helpers.is_trained_case(case))
    sample, _ = helpers.inputs_for(g)
    with torch.no_grad():
        fp = m.depth_backbone(sample["rgb"])
        cond = m.depth_head._condition(m.depth_head._neck(fp))
        enc = m.depth_head.depth_transform.t(sample["gt"])
    ref = torch.from_numpy(g["z"]["cond"])
    assert (helpers.golden_view(g, "cond", cond) - ref).abs().max().item() < 1e-5 * float(g["z"]["cond_absmax"])
    assert enc.shape == (g["B"], 16, (g["H"] + 1) // 2, (g["W"] + 1) // 2)


def test_oracle_fp64_budget():
    """fp32 restatement vs its own fp64 evaluation: the error floor parity numbers are read against."""
    g = helpers.load_golden("g_res18_ragged")
    m = helpers.build_mirror(g["family"], g["T"])
    sd = m.state_dict()
    sample, noise = helpers.inputs_for(g)
    bb = configs.FAMILIES[g["family"]]["backbone_name"]
    o32 = restate.forward(sd, sample, bb, g["T"], noise, dtype=torch.float32)
    o64 = restate.forward(sd, sample, bb, g["T"], noise, dtype=torch.float64)
    assert (o32["logits"].double() - o64["logits"]).abs().max().item() < 1e-4


def test_denoiser_is_nonnegative_and_batch_independent():
    g = helpers.load_golden("g_res18_ragged")
    sd = helpers.build_mirror(g["family"], g["T"]).state_dict()
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(2, 16, 9, 11, generator=gen)
    cond = torch.randn(2, 256, 9, 11, generator=gen)
    e2 = restate.denoiser(sd, x, torch.tensor([10, 700]), cond, "res")
    e0 = restate.denoiser(sd, x[:1], 10, cond[:1], "res")
    assert (e2 >= 0).all()          # post-ReLU "noise" (SURVEY.md §3.2)
    assert torch.allclose(e2[:1], e0, atol=1e-6)


def test_oracle_against_reference_swin_head():
    """Swin *head* path (HAHI neck + FPN + upsample_fuse loop + decoder) against the reference's head, fed with
    synthetic Swin-shaped feature maps so the (slow) Swin-L backbone is not needed on CPU (tests/golden/ref_swin_head.npz:
    the reference's decoder logits and depth under the mirror head's seeded weights, oracle.make_golden.fixture_swin_head)."""
    ref = np.load(os.path.join(helpers.GOLDEN_DIR, "ref_swin_head.npz"), allow_pickle=False)
    head = make_golden.swin_head_mirror()
    sd = {"depth_head." + k: v for k, v in head.state_dict().items()}
    ck = float(sum(v.double().abs().sum() for v in sd.values() if v.is_floating_point()))
    assert abs(ck - float(ref["weight_checksum"])) <= 1e-9 * ck, "weights were not regenerated identically"
    fp, gt, noise = make_golden.swin_head_inputs()
    with torch.no_grad():
        cond = restate.fpn_condition(sd, restate.hahi_neck(sd, fp))
        lat = restate.ddim_loop(sd, cond, noise, 3, "swin")
        z = restate.decode_logits(sd, lat)
    assert (z - torch.from_numpy(ref["logits"])).abs().max().item() < TOL_Z
    assert torch.allclose(restate.decode(sd, lat), torch.from_numpy(ref["pred"]), rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("case", range(len(make_golden.WINDOW_MSA_CASES)),
                         ids=[f"{h}x{w}-shift{s}" for (h, w), s in make_golden.WINDOW_MSA_CASES])
def test_window_msa_against_reference_trained_regime(case):
    """The reference's own ShiftWindowMSA / WindowMSA modules (backbone/swin.py:150-189, 250-325) with NON-ZERO
    relative-position tables, padded (24x40 -> 28x42, 13x9 -> 14x14) and shifted windows, against (a) the
    restatement and (b) the mirror's module — the bias / mask / roll path that the `nopretrain` factory leaves at zero.
    tests/golden/ref_window_msa.npz holds a seeded sample of the reference's output tokens per case; the mirror's module
    under the same seed has the reference module's weights (checked by checksum)."""
    ref = np.load(os.path.join(helpers.GOLDEN_DIR, "ref_window_msa.npz"), allow_pickle=False)
    hw, shift = make_golden.WINDOW_MSA_CASES[case]
    C, heads = 96, 3
    from diffusiondepth_b200.model.backbone import swin as mirror_swin
    torch.manual_seed(5)
    mine = mirror_swin.ShiftWindowMSA(C, heads, 7, shift).eval()
    table, x = make_golden.window_msa_inputs(hw, heads, C)
    with torch.no_grad():
        mine.w_msa.relative_position_bias_table.copy_(table)
    sd = mine.state_dict()
    ck = float(sum(v.double().abs().sum() for v in sd.values() if v.is_floating_point()))
    assert abs(ck - float(ref[f"c{case}_weight_checksum"])) <= 1e-9 * ck, "weights were not regenerated identically"
    rows = torch.from_numpy(ref[f"c{case}_rows"])
    want = torch.from_numpy(ref[f"c{case}_out"])
    tol = 2e-6 * float(ref[f"c{case}_out_absmax"]) + 1e-6
    got = restate._shift_window_msa({"a." + k: v for k, v in sd.items()}, x, hw, "a.", heads, 7, shift)
    assert (got[:, rows] - want).abs().max().item() < tol
    with torch.no_grad():
        assert (mine(x, hw)[:, rows] - want).abs().max().item() < tol
        # the bias really matters in this regime
        mine.w_msa.relative_position_bias_table.zero_()
        assert (mine(x, hw)[:, rows] - want).abs().max().item() > 1e-3
