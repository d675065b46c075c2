"""TEST INFRASTRUCTURE ONLY — stochastic DDIM (eta > 0) on top of the CPU restatement (oracle/restate.py), the golden
cases that pin it, and (run as a script, where the reference sources are importable) their generator:

    python tests/eta_oracle.py [case ...]     # writes tests/golden/<case>.npz, ref_scheduler_eta.npz,
                                              # ref_pipeline_signature.json

The step is the reference's three-expression form (scheduling_ddim.py:285-350, use_clipped_model_output=True) with
sigma_t = eta sqrt((1 - a_p) / (1 - a_t) (1 - a_t / a_p)) and the step's noise z_t added last."""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import configs, restate  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
SEED_STEP_NOISE = 4321
INTER_STRIDE, LIST_STRIDE = 2, 4  # spatial sub-sampling of the Vis goldens' per-step maps / latents

# name -> (family, T, batch, H, W, eta)
GOLDEN_ETA = {
    "g_res18_eta": ("res18", 5, 1, 228, 304, 1.0),           # BASELINE config 1, full sampler noise
    "g_swinl_small_eta": ("swinl", 5, 1, 96, 160, 0.5),      # Swin head on a small grid
    "g_swinl_vis_eta": ("swinl_vis", 5, 1, 96, 160, 1.0),    # Vis head: pred_inter + the latent after every step
    "g_swinl_c3_eta": ("swinl", 20, 1, 352, 1216, 1.0),      # image 0 of BASELINE config 3
}


def synthetic_step_noise(steps, batch, height, width, seed=SEED_STEP_NOISE, first=0):
    """Per-step noise [T,B,16,ceil(H/2),ceil(W/2)] ~ N(0,1); image i of the global batch has its own generator
    (seed, first + i), so any shard of a batch sees exactly the noise the full batch would."""
    out = []
    for i in range(first, first + batch):
        g = torch.Generator().manual_seed(seed * 1000003 + i)
        out.append(torch.randn(steps, 16, (height + 1) // 2, (width + 1) // 2, generator=g))
    return torch.stack(out, 1)


def ddim_step(eps, t: int, x, alphas_cumprod, num_inference_steps, eta=0.0, z=None, num_train_timesteps=1000):
    """scheduling_ddim.py:285-350, epsilon prediction, no clipping, use_clipped_model_output=True."""
    prev_t = t - num_train_timesteps // num_inference_steps
    a_t = alphas_cumprod[t].to(x.dtype)
    a_prev = alphas_cumprod[prev_t].to(x.dtype) if prev_t >= 0 else torch.tensor(1.0, dtype=x.dtype)
    b_t = 1 - a_t
    x0 = (x - b_t ** 0.5 * eps) / a_t ** 0.5
    variance = (1 - a_prev) / (1 - a_t) * (1 - a_t / a_prev)
    sigma = eta * variance ** 0.5
    eps2 = (x - a_t ** 0.5 * x0) / b_t ** 0.5
    prev = a_prev ** 0.5 * x0 + (1 - a_prev - sigma ** 2) ** 0.5 * eps2
    if eta > 0:
        prev = prev + variance ** 0.5 * eta * z
    return prev


def ddim_loop(sd, cond, noise, num_inference_steps, variant, eta=0.0, step_noise=None, collect=False):
    """CNNDDIMPipiline.__call__ (head :254-303) with x_T and the per-step noise injected."""
    acp = restate.ddim_tables()
    x, trace = noise, []
    for i, t in enumerate(restate.ddim_timesteps(num_inference_steps)):
        eps = restate.denoiser(sd, x, t, cond, variant)
        x = ddim_step(eps, t, x, acp, num_inference_steps, eta, step_noise[i].to(x.dtype) if eta > 0 else None)
        if collect:
            trace.append(x)
    return (x, trace) if collect else x


def forward(sd, sample, backbone, num_inference_steps, noise, eta=0.0, step_noise=None, dtype=torch.float32):
    """restate.forward with stochastic DDIM.  Returns dict(pred, logits, latent, cond, trace)."""
    variant = "swin" if "depth_head.model.upsample_fuse.convA.conv.weight" in sd else "res"
    with torch.no_grad():
        cond = restate.condition_features(sd, sample["rgb"].to(dtype), backbone)
        latent, trace = ddim_loop(sd, cond, noise.to(dtype), num_inference_steps, variant, eta, step_noise, collect=True)
        z = restate.decode_logits(sd, latent)
        pred = 1.0 / torch.sigmoid(z).clamp(1e-6) - 1
    return dict(pred=pred, logits=z, latent=latent, cond=cond, trace=trace)


# -------------------------------------------------------------------------------------------------- golden generation
def _inject_randn(queue):
    """Hand the reference's `torch.randn` draws of x_T's shape our tensors, in order (x_T, then one per step); every
    other draw (ddim_loss, after the loop) is left alone."""
    real = torch.randn
    state = {"used": 0}

    def fake(*size, **kw):
        shape = tuple(size[0]) if len(size) == 1 and not isinstance(size[0], int) else tuple(size)
        if state["used"] < len(queue) and shape == tuple(queue[0].shape):
            t = queue[state["used"]]
            state["used"] += 1
            return t.clone().to(kw.get("device") or "cpu", kw.get("dtype") or t.dtype)
        return real(*size, **kw)

    return real, fake, state


def run_reference(net, sample, noise, eta, step_noise):
    """The reference model's own forward with `head.pipeline(..., eta=eta)` and the T + 1 draws injected.
    -> dict(pred, logits, latent, pred_inter?, image_list?)."""
    head = net.depth_head
    cap, lat_steps = {}, []
    orig = head.pipeline

    def pipeline(*a, **k):  # the reference head calls its pipeline without `eta`
        out = orig(*a, eta=eta, **k)
        if isinstance(out, tuple) and len(out) == 2:
            lat_steps.extend(x.detach().clone() for x in out[1])
        return out

    hooks = [head.depth_transform.conv_inv_transform.register_forward_pre_hook(
                 lambda m, a: cap.__setitem__("latent", a[0].detach().clone())),
             head.depth_transform.conv_inv_transform[3].register_forward_hook(
                 lambda m, a, o: cap.__setitem__("logits", o.detach().clone()))]
    real, fake, state = _inject_randn([noise] + list(step_noise.unbind(0)))
    head.pipeline = pipeline
    torch.randn = fake
    try:
        with torch.no_grad():
            out = net(sample)
    finally:
        torch.randn = real
        head.pipeline = orig
        for h in hooks:
            h.remove()
    assert state["used"] == 1 + step_noise.shape[0], state
    r = dict(pred=out["pred"], logits=cap["logits"], latent=cap["latent"])
    if out.get("pred_inter") is not None:
        r["pred_inter"] = torch.stack([p.detach() for p in out["pred_inter"]])
        r["image_list"] = torch.stack(lat_steps)
    return r


def generate(case):
    from oracle import make_golden, ref_import
    family, T, B, H, W, eta = GOLDEN_ETA[case]
    t0 = time.time()
    mirror = make_golden.build_mirror(family, T)
    sd = {k: v.detach().clone() for k, v in mirror.state_dict().items()}
    fam = configs.FAMILIES[family]
    ref = ref_import.build_reference_model(ref_import.make_args(fam["backbone_module"], fam["backbone_name"],
                                                                fam["head_specify"], T))
    ref.load_state_dict(sd, strict=True)
    sample = restate.synthetic_sample(B, H, W, configs.SEED_INPUTS)
    noise = restate.synthetic_noise(B, H, W, configs.SEED_NOISE)
    z_steps = synthetic_step_noise(T, B, H, W)
    torch.manual_seed(0)
    r = run_reference(ref, sample, noise, eta, z_steps)
    o = forward(sd, sample, fam["backbone_name"], T, noise, eta, z_steps)
    pm = restate.parity_metrics(o["logits"], r["logits"], o["pred"], r["pred"])
    print(f"[{case}] reference {time.time() - t0:.1f}s; oracle-vs-reference max|dz|={pm['max_dz']:.2e}", flush=True)
    arrays = {}
    for name in ("logits", "pred", "latent"):
        arr, stride = make_golden.subsample(name, r[name], H, W)
        arrays[name], arrays[name + "_stride"] = arr.numpy(), np.int32(stride)
    if "pred_inter" in r:
        # every step's map and latent, sub-sampled (the final ones are stored above at full density)
        arrays["pred_inter"] = r["pred_inter"][..., ::INTER_STRIDE, ::INTER_STRIDE].float().contiguous().numpy()
        arrays["image_list"] = r["image_list"][..., ::LIST_STRIDE, ::LIST_STRIDE].float().contiguous().numpy()
        arrays["pred_inter_stride"], arrays["image_list_stride"] = np.int32(INTER_STRIDE), np.int32(LIST_STRIDE)
    arrays.update(meta=np.array([T, B, H, W], dtype=np.int32), family=np.array(family), eta=np.float64(eta),
                  weight_checksum=np.float64(make_golden.weight_checksum(sd)),
                  latent_absmax=np.float64(r["latent"].abs().max()), oracle_max_dz=np.float64(pm["max_dz"]))
    np.savez_compressed(os.path.join(GOLDEN_DIR, case + ".npz"), **arrays)


def fixture_scheduler_eta():
    """The reference DDIMScheduler.step with `variance_noise`: one seeded chain per (eta, T), every step stored."""
    from oracle import ref_import
    ref = ref_import.reference_modules().scheduling_ddim.DDIMScheduler(num_train_timesteps=1000, clip_sample=False)
    out = {}
    g = torch.Generator().manual_seed(17)
    for eta in (0.3, 1.0):
        for T in (5, 20, 50):
            ref.set_timesteps(T)
            x = torch.randn(1, 16, 2, 3, generator=g)
            xs, eps_l, zs, prev = [], [], [], []
            for t in ref.timesteps:
                eps, z = torch.rand(x.shape, generator=g), torch.randn(x.shape, generator=g)
                nxt = ref.step(eps, t, x, eta=eta, use_clipped_model_output=True, variance_noise=z)["prev_sample"]
                xs.append(x), eps_l.append(eps), zs.append(z), prev.append(nxt)
                x = nxt
            k = f"eta{eta}_T{T}_"
            for name, v in (("x", xs), ("eps", eps_l), ("z", zs), ("prev", prev)):
                out[k + name] = torch.stack(v).numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "ref_scheduler_eta.npz"), **out)


def fixture_pipeline_signature():
    """inspect.signature of the reference's plain and Vis CNNDDIMPipiline.__call__."""
    import importlib
    import inspect
    from oracle import ref_import
    mods = ref_import.reference_modules()
    vis = importlib.import_module("model.head.ddim_depth_estimate_res_swin_addHAHI_vis")
    sig = {"plain": str(inspect.signature(mods.head_swin.CNNDDIMPipiline.__call__)),
           "vis": str(inspect.signature(vis.CNNDDIMPipiline.__call__))}
    with open(os.path.join(GOLDEN_DIR, "ref_pipeline_signature.json"), "w") as f:
        json.dump(sig, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    cases = sys.argv[1:] or ["fixtures"] + list(GOLDEN_ETA)
    for c in cases:
        if c == "fixtures":
            fixture_scheduler_eta()
            fixture_pipeline_signature()
        else:
            generate(c)
