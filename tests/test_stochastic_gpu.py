"""Stochastic DDIM (eta > 0) and `head.pipeline` on the B200: bit-identity with the deterministic loop at sigma = 0,
parity with the reference's own pipeline (goldens), the Vis `image_list`, the CUDA draw order, graph staging of the
step noise, sharding and generator handling.  Tolerance: 1e-3 on the decoder logit z, as tests/test_gpu_parity.py."""
import pytest
import torch

import diffusiondepth_b200 as dd
from oracle import configs, restate
import dd_helpers as helpers
import eta_oracle
from diffusiondepth_b200.model.head._pipeline import draw_pipeline_noise
from diffusiondepth_b200.model.registry import HEADS

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOL = 1e-3


def _head(name, steps, seed=7):
    torch.manual_seed(seed)
    return HEADS.build(dict(type=name, in_channels=[64, 128, 256, 512], inference_steps=steps, num_train_timesteps=1000,
                            depth_feature_dim=16, loss_cfgs=[], init_cfg=None)).eval().to(DEV)


def _engine_tensors(head):
    return {k: v.detach() for k, v in head._engine_tensors().items()}


@pytest.mark.parametrize("variant,fp8", [("res", False), ("swin", False), ("swin", True)])
def test_sigma_zero_is_bit_identical_to_the_deterministic_loop(variant, fp8):
    T, B, (h, w) = 4, 2, (20, 28)
    chw = (h, w) if variant == "res" else (h // 2, w // 2)
    head = _head("DDIMDepthEstimate_Res" if variant == "res" else "DDIMDepthEstimate_Swin_ADDHAHI", T)
    g = torch.Generator().manual_seed(3)
    cond = torch.randn(B, 256, *chw, generator=g).abs().to(DEV)
    noise = torch.randn(B, 16, h, w, generator=g).to(DEV)
    z = torch.randn(T, B, 16, h, w, generator=g).to(DEV)
    ts, cx, ce = head.scheduler.fused_coefficients(T)
    outs = []
    for stoch in (False, True):
        eng = dd.DenoiseEngine(variant, B, (h, w), chw, T, DEV, fp8_corr=fp8, stochastic=stoch)
        eng.load_weights(_engine_tensors(head))
        eng.set_schedule(ts, cx, ce, [0.0] * T if stoch else None)
        if stoch:
            with pytest.raises(dd.EngineError):
                eng.denoise_decode(cond, noise)
            d, lat, _, zl, _ = eng.denoise_decode_stochastic(cond, noise, z, want_latent=True, want_logits=True)
        else:
            with pytest.raises(dd.EngineError):
                eng.denoise_decode_stochastic(cond, noise, z)
            d, lat, zl = eng.denoise_decode(cond, noise, want_latent=True, want_logits=True)
        eng.poll_status()
        outs.append((d, lat, zl))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def _run_case(case, fp8=True, batch=None):
    family, T, B, H, W, eta = eta_oracle.GOLDEN_ETA[case]
    g = helpers.load_golden(case)
    B = batch or B
    m = helpers.build_mirror(family, T).to(DEV)
    head = m.depth_head
    head.fp8_corrections = fp8
    head.capture_logits = True
    sample = restate.synthetic_sample(B, H, W, configs.SEED_INPUTS)
    sample["noise"] = restate.synthetic_noise(B, H, W, configs.SEED_NOISE)
    sample["step_noise"] = eta_oracle.synthetic_step_noise(T, B, H, W)
    sample = {k: v.to(DEV) for k, v in sample.items()}
    head.ddim_eta = eta
    try:
        with torch.no_grad():
            out = m(sample)
    finally:
        head.ddim_eta = 0.0
    return g, m, sample, out


@pytest.mark.parametrize("case,fp8", [("g_res18_eta", False), ("g_swinl_small_eta", True), ("g_swinl_small_eta", False),
                                      ("g_swinl_c3_eta", True), ("g_swinl_c3_eta", False)])
def test_forward_with_eta_matches_reference_golden(case, fp8, parity_log):
    g, m, sample, out = _run_case(case, fp8)
    z = m.depth_head.last_logits.cpu()
    dz = (helpers.golden_view(g, "logits", z) - torch.from_numpy(g["z"]["logits"])).abs()
    parity_log(case + ("" if fp8 else " [exact 3-pass split]"),
               "reference golden, eta=%g (logits sub-sampled x%d)" % (float(g["z"]["eta"]), int(g["z"]["logits_stride"])), dz)
    assert dz.max().item() < TOL, f"{case}: max|dz| {dz.max().item():.3e}"
    if case == "g_swinl_c3_eta":  # every pixel against the restatement
        family, T, B, H, W, eta = eta_oracle.GOLDEN_ETA[case]
        sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
        s = {k: v.cpu() for k, v in sample.items()}
        ref = eta_oracle.forward(sd, s, configs.FAMILIES[family]["backbone_name"], T, s["noise"], eta, s["step_noise"])
        dz = (z - ref["logits"]).abs()
        parity_log(case + ("" if fp8 else " [exact 3-pass split]"), "fp32 restatement, all %d pixels" % dz.numel(), dz)
        assert dz.max().item() < TOL


@pytest.mark.parametrize("case", ["g_res18_eta", "g_swinl_small_eta"])
def test_pipeline_with_eta_matches_reference_golden(case, parity_log):
    """`head.pipeline(..., eta=)` on the condition map, with x_T and the step draws injected through torch.randn's
    CUDA default generator state."""
    family, T, B, H, W, eta = eta_oracle.GOLDEN_ETA[case]
    g, m, sample, _ = _run_case(case)  # also leaves the condition map the forward built
    head = m.depth_head
    head.capture_cond = True
    with torch.no_grad():
        m(sample)
    cond = head.last_cond
    ts_shape = (B, 16, (H + 1) // 2, (W + 1) // 2)
    torch.cuda.manual_seed(11)
    x_T, steps = draw_pipeline_noise(T, ts_shape, DEV)
    torch.cuda.manual_seed(11)
    with torch.no_grad():
        (lat,) = head.pipeline(B, DEV, torch.float32, ts_shape[1:], (cond, None, None, None), eta=eta,
                               num_inference_steps=T, return_dict=False)
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    ref = eta_oracle.ddim_loop(sd, cond.cpu(), x_T.cpu(), T, head.variant, eta, steps.cpu())
    dz = (restate.decode_logits(sd, lat.cpu()) - restate.decode_logits(sd, ref)).abs()
    parity_log(case + " pipeline", "fp32 restatement on its draws, eta=%g" % eta, dz)
    assert dz.max().item() < TOL
    # injected x_T = the golden's: the pipeline then reproduces the reference's latent
    x_T = sample["noise"]
    with torch.no_grad():
        lat2, = head.sample_latents(cond, x_T, sample["step_noise"], eta, T)[:1]
    dz = (helpers.golden_view(g, "logits", restate.decode_logits(sd, lat2.cpu())) - torch.from_numpy(g["z"]["logits"])).abs()
    parity_log(case + " pipeline", "reference golden, eta=%g" % eta, dz)
    assert dz.max().item() < TOL


def test_vis_pipeline_image_list_and_pred_inter():
    case = "g_swinl_vis_eta"
    family, T, B, H, W, eta = eta_oracle.GOLDEN_ETA[case]
    g, m, sample, out = _run_case(case)
    head = m.depth_head
    si = int(g["z"]["pred_inter_stride"])
    inter = torch.stack([p.cpu() for p in out["pred_inter"]])[..., ::si, ::si]
    ref_inter = torch.from_numpy(g["z"]["pred_inter"])
    rel = ((inter - ref_inter).abs() / ref_inter.abs().clamp_min(1e-6))[ref_inter < 1e5]
    assert rel.max().item() < TOL
    head.capture_cond = True
    with torch.no_grad():
        m(sample)
        images, image_list = head.sample_latents(head.last_cond, sample["noise"], sample["step_noise"], eta, T,
                                                 latent_steps=True)
    ref = torch.from_numpy(g["z"]["image_list"])
    sl = int(g["z"]["image_list_stride"])
    assert image_list.shape == (T, B, 16, (H + 1) // 2, (W + 1) // 2) and torch.equal(images, image_list[-1])
    got = image_list.cpu()[..., ::sl, ::sl]
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() < 5e-4 * max(1.0, ref.abs().max().item())
    with torch.no_grad():
        r = head.pipeline(B, DEV, torch.float32, ref.shape[-3:], (head.last_cond, None, None, None), eta=eta,
                          num_inference_steps=T)
        r0 = head.pipeline(B, DEV, torch.float32, ref.shape[-3:], (head.last_cond, None, None, None), eta=0.0,
                           num_inference_steps=T, return_dict=False)
    assert sorted(r) == ["image_list", "images"] and len(r["image_list"]) == T
    assert len(r0) == 2 and len(r0[1]) == T and torch.equal(r0[0], r0[1][-1])


def test_cuda_draw_order_and_forward_without_injected_noise():
    T, shape = 4, (1, 16, 20, 28)
    torch.cuda.manual_seed(5)
    want = [torch.randn(shape, device=DEV) for _ in range(T + 1)]
    torch.cuda.manual_seed(5)
    x_T, steps = draw_pipeline_noise(T, shape, DEV)
    assert torch.equal(x_T, want[0]) and all(torch.equal(steps[i], want[i + 1]) for i in range(T))
    head = _head("DDIMDepthEstimate_Res", T)
    head.ddim_eta = 1.0
    g = torch.Generator().manual_seed(2)
    fp = [torch.randn(1, c, 20 // s, 28 // s, generator=g).to(DEV) for c, s in zip((64, 128, 256, 512), (1, 2, 4, 8))]
    gt = (torch.rand(1, 1, 40, 56, generator=g) * 80).to(DEV)
    torch.cuda.manual_seed(5)
    a = head(fp, gt, gt > 0, gt_depth_map=gt)["pred"]
    b = head(fp, gt, gt > 0, gt_depth_map=gt, noise=want[0], step_noise=torch.stack(want[1:]))["pred"]
    assert torch.equal(a, b)
    c = head(fp, gt, gt > 0, gt_depth_map=gt, noise=want[0], step_noise=torch.stack(want[1:]) * 0.5)["pred"]
    assert not torch.equal(a, c)


def test_graph_staging_takes_each_calls_noise():
    T, B, (h, w) = 3, 1, (16, 24)
    head = _head("DDIMDepthEstimate_Swin_ADDHAHI", T)
    g = torch.Generator().manual_seed(8)
    cond = torch.randn(B, 256, h // 2, w // 2, generator=g).abs().to(DEV)
    noise = torch.randn(B, 16, h, w, generator=g).to(DEV)
    zs = [torch.randn(T, B, 16, h, w, generator=g).to(DEV) for _ in range(2)]
    res = {}
    for graph in (True, False):
        head.invalidate_engines()
        head.use_cuda_graph = graph
        res[graph] = [head.sample_latents(cond, noise, z, 1.0, T)[0].clone() for z in zs]
    assert not torch.equal(res[True][0], res[True][1])
    for i in range(2):
        assert torch.equal(res[True][i], res[False][i])


def test_batch_of_two_equals_two_batch_one_runs():
    case = "g_swinl_small_eta"
    family, T, B, H, W, eta = eta_oracle.GOLDEN_ETA[case]
    m = helpers.build_mirror(family, T).to(DEV)
    head = m.depth_head
    head.capture_logits = True
    head.ddim_eta = eta

    def run(n, first):
        s = restate.synthetic_sample(n, H, W, configs.SEED_INPUTS, first=first)
        s["noise"] = restate.synthetic_noise(n, H, W, configs.SEED_NOISE, first=first)
        s["step_noise"] = eta_oracle.synthetic_step_noise(T, n, H, W, first=first)
        with torch.no_grad():
            m({k: v.to(DEV) for k, v in s.items()})
        return head.last_logits.cpu()

    try:
        both = run(2, 0)
        ones = torch.cat([run(1, 0), run(1, 1)])
    finally:
        head.ddim_eta = 0.0
    assert (both - ones).abs().max().item() < 1e-5


def test_generator_handling():
    T, shape = 3, (16, 16, 24)
    head = _head("DDIMDepthEstimate_Swin_ADDHAHI", T)
    cond = torch.randn(1, 256, 8, 12, device=DEV).abs()
    outs = []
    for _ in range(2):
        gen = torch.Generator(device=DEV).manual_seed(99)
        outs.append(head.pipeline(1, DEV, torch.float32, shape, (cond, None, None, None), generator=gen, eta=1.0,
                                  num_inference_steps=T)["images"])
    assert torch.equal(outs[0], outs[1])
    with pytest.raises(ValueError):
        head.pipeline(1, DEV, torch.float32, shape, (cond, None, None, None), generator=torch.Generator(), eta=1.0,
                      num_inference_steps=T)
