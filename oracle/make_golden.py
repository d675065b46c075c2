"""TEST INFRASTRUCTURE ONLY — generate tests/golden/*.npz from the REAL reference (/root/reference, imported
unmodified under oracle/refstub).  Run in the build container:  python -m oracle.make_golden [case ...]

Weights: the product mirror's default construction under torch.manual_seed(7240) (same init distributions as
the reference's modules; its state_dict matches the reference key-for-key), loaded into the reference with
load_state_dict(strict=True).  Inputs/noise: oracle.restate.synthetic_sample / synthetic_noise.
Stored per case: decoder logits z, depth, final latent, condition map (sub-sampled where large), summary
statistics and a weight checksum so a consumer can tell whether it regenerated the same weights."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import configs, ref_import, reference_runner, restate  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def build_mirror(family, steps, trained=False):
    from diffusiondepth_b200.model import get
    args = configs.make_args(family, steps)
    torch.manual_seed(configs.SEED_WEIGHTS)
    m = get(args)(args).eval()
    return configs.trainedify(m) if trained else m


def weight_checksum(sd):
    """sum |w| in fp64 over the hot-path parameters + a few producer tensors."""
    keys = sorted(k for k in sd if k.startswith("depth_head.model.") or "conv_inv_transform" in k
                  or k.startswith("depth_head.conv_lateral") or k.endswith("relative_position_bias_table"))
    return float(sum(sd[k].double().abs().sum() for k in keys if sd[k].is_floating_point()))


def subsample(name, t, H, W):
    t = t.detach().float()
    if name in ("logits", "pred"):
        s = 1 if H * W <= 80000 else 4
        return t[..., ::s, ::s].contiguous(), s
    if name == "latent":
        s = 1 if H * W <= 20000 else (2 if H * W <= 80000 else 4)
        return t[..., ::s, ::s].contiguous(), s
    if name == "cond":
        return t[:, ::32, ::4, ::4].contiguous(), 4
    raise KeyError(name)


def generate(case):
    trained = case in configs.GOLDEN_TRAINED
    family, T, B, H, W = (configs.GOLDEN_TRAINED if trained else configs.GOLDEN)[case]
    t0 = time.time()
    mirror = build_mirror(family, T, trained)
    sd = {k: v.detach().clone() for k, v in mirror.state_dict().items()}
    ref = ref_import.build_reference_model(ref_import.make_args(
        configs.FAMILIES[family]["backbone_module"], configs.FAMILIES[family]["backbone_name"],
        configs.FAMILIES[family]["head_specify"], T))
    ref.load_state_dict(sd, strict=True)
    sample = restate.synthetic_sample(B, H, W, configs.SEED_INPUTS)
    noise = restate.synthetic_noise(B, H, W, configs.SEED_NOISE)
    torch.manual_seed(0)
    r = reference_runner.run_reference(ref, sample, noise)
    t_ref = time.time() - t0
    # pin the restatement against the reference on this very case
    o = restate.forward(sd, sample, configs.FAMILIES[family]["backbone_name"], T, noise)
    pm = restate.parity_metrics(o["logits"], r["logits"], o["pred"], r["pred"])
    lat_err = (o["latent"] - r["latent"]).abs().max().item() / max(r["latent"].abs().max().item(), 1e-30)
    cond_err = (o["cond"] - r["cond"]).abs().max().item() / max(r["cond"].abs().max().item(), 1e-30)
    print(f"[{case}] reference {t_ref:.1f}s; oracle-vs-reference: max|dz|={pm['max_dz']:.2e} rms={pm['rms_dz']:.2e} "
          f"latent rel {lat_err:.2e} cond rel {cond_err:.2e}", flush=True)
    arrays = {}
    for name in ("logits", "pred", "latent", "cond"):
        arr, stride = subsample(name, r[name], H, W)
        arrays[name] = arr.numpy()
        arrays[name + "_stride"] = np.int32(stride)
    if "pred_inter" in r:
        arrays["pred_inter"] = r["pred_inter"].float().numpy()
    z = r["logits"].double()
    arrays.update(
        meta=np.array([T, B, H, W], dtype=np.int32), family=np.array(family),
        weight_checksum=np.float64(weight_checksum(sd)),
        logits_mean=np.float64(z.mean()), logits_std=np.float64(z.std()), logits_absmax=np.float64(z.abs().max()),
        latent_std=np.float64(r["latent"].double().std()), latent_absmax=np.float64(r["latent"].abs().max()),
        cond_absmax=np.float64(r["cond"].abs().max()),
        frac_clamped=np.float64((r["pred"] >= 999998.0).double().mean()),
        oracle_max_dz=np.float64(pm["max_dz"]), output_keys=np.array(r["keys"]))
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, case + ".npz"), **arrays)
    print(f"[{case}] wrote {case}.npz ({os.path.getsize(os.path.join(OUT, case + '.npz')) / 1e3:.0f} kB)", flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# Module-level fixtures: what the reference's own sub-modules return on the seeded inputs of the tests that compare
# against them (tests/test_scheduler.py, test_io_contract.py, test_plugin_surface.py, test_oracle_golden.py,
# test_dropin.py), so those comparisons run wherever the suite runs.

def digest(t):
    """sha256 of a tensor's bytes: a bitwise-equality check that does not need the tensor stored."""
    import hashlib
    return hashlib.sha256(t.detach().contiguous().numpy().tobytes()).hexdigest()


def sample_rows(n, k, seed):
    """A fixed, seeded, sorted sample of k of n row indices (all of them when n <= k)."""
    if n <= k:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:k].sort().values


def official_swin_like(C=8):
    """A tiny state_dict in the official Swin checkpoint layout (the input of swin_convert)."""
    g = torch.Generator().manual_seed(0)
    r = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    return {"patch_embed.proj.weight": r(C, 3, 4, 4), "patch_embed.norm.weight": r(C),
            "layers.0.blocks.0.attn.qkv.weight": r(3 * C, C), "layers.0.blocks.0.attn.relative_position_bias_table": r(169, 2),
            "layers.0.blocks.0.mlp.fc1.weight": r(4 * C, C), "layers.0.blocks.0.mlp.fc2.bias": r(C),
            "layers.0.blocks.0.norm1.weight": r(C), "layers.0.downsample.reduction.weight": r(2 * C, 4 * C),
            "layers.0.downsample.norm.weight": r(4 * C), "layers.0.downsample.norm.bias": r(4 * C),
            "norm.weight": r(8 * C), "head.weight": r(10, 8 * C)}


SWIN_HEAD_CFG = dict(type="DDIMDepthEstimate_Swin_ADDHAHI", in_channels=[64, 128, 256, 512], inference_steps=3,
                     num_train_timesteps=1000, depth_feature_dim=16, loss_cfgs=[], init_cfg=None)
SWIN_HEAD_SEED = 11
WINDOW_MSA_CASES = (((24, 40), 0), ((24, 40), 3), ((13, 9), 3))
WINDOW_MSA_ROWS = 32  # stored output tokens per image and case
# the flags of src/main.py's test mode in tests/test_dropin.py
MAIN_FLAGS = ["--test_only", "--model_name", "Diffusion_DCbase_", "--backbone_module", "mmbev_resnet", "--backbone_name",
              "mmbev_res18", "--head_specify", "DDIMDepthEstimate_Res", "--inference_steps", "5", "--gpus", "0"]


def swin_head_inputs():
    """Synthetic Swin-L-shaped feature maps, depth and initial latent of the Swin head fixture."""
    gen = torch.Generator().manual_seed(2)
    H, W = 40, 56
    fp = [torch.randn(1, c, -(-H // s), -(-W // s), generator=gen) for c, s in ((192, 4), (384, 8), (768, 16), (1536, 32))]
    gt = torch.rand(1, 1, H, W, generator=gen) * 80
    noise = torch.randn(1, 16, H // 2, W // 2, generator=gen)
    return fp, gt, noise


def swin_head_mirror():
    """The mirror's Swin head under SWIN_HEAD_SEED with a zero HAHI level embedding (the fixture's weights)."""
    from diffusiondepth_b200.model.registry import HEADS
    torch.manual_seed(SWIN_HEAD_SEED)
    head = HEADS.build(dict(SWIN_HEAD_CFG)).eval()
    with torch.no_grad():
        head.hahineck.level_embed.zero_()
    return head


def window_msa_inputs(hw, heads, C):
    """Relative-position table and tokens of one window-attention case (one CPU generator, table drawn first)."""
    gen = torch.Generator().manual_seed(6)
    table = torch.randn(169, heads, generator=gen) * 0.7
    return table, torch.randn(2, hw[0] * hw[1], C, generator=gen)


def fixture_scheduler():
    """The reference DDIMScheduler: alphas_cumprod, timesteps, and every step of one seeded chain per T."""
    ref = ref_import.reference_modules().scheduling_ddim.DDIMScheduler(num_train_timesteps=1000, clip_sample=False)
    out = {"alphas_cumprod": ref.alphas_cumprod.numpy()}
    g = torch.Generator().manual_seed(3)
    for T in (5, 20, 50):
        ref.set_timesteps(T)
        out[f"T{T}_timesteps"] = ref.timesteps.numpy()
        x = torch.randn(1, 16, 6, 10, generator=g)
        prev, orig = [], []
        for t in ref.timesteps:
            eps = torch.rand(x.shape, generator=g)
            a = ref.step(eps, t, x, eta=0.0, use_clipped_model_output=True)
            prev.append(digest(a["prev_sample"]))
            orig.append(digest(a["pred_original_sample"]))
            x = a["prev_sample"]
        out[f"T{T}_prev_sample_sha256"], out[f"T{T}_pred_original_sha256"] = np.array(prev), np.array(orig)
        out[f"T{T}_last_prev_sample"], out[f"T{T}_last_pred_original"] = x.numpy(), a["pred_original_sample"].numpy()
    t = torch.tensor([7, 300])
    x0, n = torch.randn(2, 16, 3, 3, generator=g), torch.randn(2, 16, 3, 3, generator=g)
    out["add_noise"] = ref.add_noise(x0, n, t).numpy()
    return out


def fixture_swin_convert():
    """The reference's swin_convert of official_swin_like(): keys in order, values."""
    conv = ref_import.reference_modules().swin.swin_convert(official_swin_like())
    return {"keys": np.array(list(conv)), **{f"v{i}": v.numpy() for i, v in enumerate(conv.values())}}


def fixture_state_dict_layout():
    """Key, shape and dtype of every state_dict entry of the reference model per family (+ one Swin index buffer)."""
    out = {}
    for family in ("res18", "swinl", "swinl_add", "mpvit_s"):
        f = configs.FAMILIES[family]
        sd = ref_import.build_reference_model(ref_import.make_args(f["backbone_module"], f["backbone_name"],
                                                                   f["head_specify"], 5)).state_dict()
        out[family + "_keys"] = np.array(list(sd))
        out[family + "_shapes"] = np.array(["x".join(str(s) for s in v.shape) for v in sd.values()])
        out[family + "_dtypes"] = np.array([str(v.dtype) for v in sd.values()])
        if family == "swinl":
            out["swinl_relative_position_index"] = sd[
                "depth_backbone.stages.2.blocks.1.attn.w_msa.relative_position_index"].numpy()
    return out


def fixture_swin_head():
    """The reference's Swin head (HAHI neck + FPN + upsample_fuse loop + decoder) under the mirror's seeded weights."""
    mods = ref_import.reference_modules()
    mine = swin_head_mirror()
    sd = mine.state_dict()
    cfg = {k: v for k, v in SWIN_HEAD_CFG.items() if k != "type"}
    head = mods.head_swin.DDIMDepthEstimate_Swin_ADDHAHI(**cfg).eval()
    head.load_state_dict(sd, strict=True)
    fp, gt, noise = swin_head_inputs()
    cap = {}
    hk = head.depth_transform.conv_inv_transform[3].register_forward_hook(lambda m, a, o: cap.__setitem__("z", o))
    with torch.no_grad(), reference_runner._inject_first_randn(noise):
        out = head(fp, gt, gt > 0, gt_depth_map=gt)
    hk.remove()
    ck = float(sum(v.double().abs().sum() for v in sd.values() if v.is_floating_point()))
    return {"logits": cap["z"].numpy(), "pred": out["pred"].numpy(), "weight_checksum": np.float64(ck)}


def fixture_window_msa():
    """The reference's ShiftWindowMSA (non-zero relative-position table; padded and shifted windows) on seeded tokens:
    a seeded sample of WINDOW_MSA_ROWS output tokens per image, and the absolute maximum of the whole output."""
    mods = ref_import.reference_modules()
    C, heads = 96, 3
    out = {}
    for i, (hw, shift) in enumerate(WINDOW_MSA_CASES):
        torch.manual_seed(5)
        ref = mods.swin.ShiftWindowMSA(embed_dims=C, num_heads=heads, window_size=7, shift_size=shift).eval()
        table, x = window_msa_inputs(hw, heads, C)
        with torch.no_grad():
            ref.w_msa.relative_position_bias_table.copy_(table)
            want = ref(x, hw)
        rows = sample_rows(hw[0] * hw[1], WINDOW_MSA_ROWS, seed=i)
        sd = ref.state_dict()
        out[f"c{i}_weight_checksum"] = np.float64(sum(v.double().abs().sum() for v in sd.values() if v.is_floating_point()))
        out[f"c{i}_rows"], out[f"c{i}_out"] = rows.numpy(), want[:, rows].numpy()
        out[f"c{i}_out_absmax"] = np.float64(want.abs().max())
    return out


def fixture_main_args():
    """The Namespace the reference's src/main.py hands to test() for the flags of tests/test_dropin.py (its config.py
    parse + check_args), as JSON; `pretrain` and `save_dir` are per-run paths and are left out."""
    import json
    import subprocess
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        ckpt = os.path.join(tmp, "model_00001.pt")
        torch.save({"net": {}}, ckpt)
        code = ("import json, main; a = vars(main.check_args(main.args_config)); "
                "print(json.dumps({k: v for k, v in a.items() if k not in ('pretrain', 'save_dir')}, sort_keys=True))")
        r = subprocess.run([sys.executable, "-c", code, *MAIN_FLAGS, "--pretrain", ckpt], cwd=tmp, capture_output=True,
                           text=True, check=True, env=dict(os.environ, PYTHONPATH=os.pathsep.join(
                               [os.path.join(ROOT, "oracle", "refstub"), ref_import.REF_SRC])))
    return json.loads(r.stdout.strip().splitlines()[-1])


FIXTURES = {"ref_scheduler": fixture_scheduler, "ref_swin_convert": fixture_swin_convert,
            "ref_state_dict_layout": fixture_state_dict_layout, "ref_swin_head": fixture_swin_head,
            "ref_window_msa": fixture_window_msa, "ref_main_args": fixture_main_args}


def generate_fixture(name):
    data = FIXTURES[name]()
    if name == "ref_main_args":
        import json
        path = os.path.join(OUT, name + ".json")
        with open(path, "w") as f:
            json.dump(data, f, indent=0, sort_keys=True)
            f.write("\n")
    else:
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **data)
    print(f"[{name}] wrote {os.path.basename(path)} ({os.path.getsize(path) / 1e3:.0f} kB)", flush=True)


if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count() or 8)
    for c in (sys.argv[1:] or list(configs.GOLDEN) + list(configs.GOLDEN_TRAINED) + list(FIXTURES)):
        generate_fixture(c) if c in FIXTURES else generate(c)
