"""The drop-in boundary, exercised the way a maintainer of the reference would (INTEGRATION.md §1):
`diffusiondepth_b200/model` symlinked into a source tree as the top-level package `model`, then the call sequence of the
reference's `src/main.py::test()` (:404-470): get_model(args)(args) -> .cuda() -> torch.load + load_state_dict(
ckpt['net'], strict=False) -> nn.DataParallel -> .eval() -> DataLoader(batch_size=1) -> sample.cuda() -> net(sample).

CPU part: the symlinked import works; main.py's test() sequence, with the arguments the reference's own config.py
parses, runs on the mirror up to the first CUDA call.  GPU part: the same sequence end to end against the golden
vectors the real reference produced."""
import copy
import os
import subprocess
import sys
import textwrap

import pytest
import torch

from oracle import configs, restate
import dd_helpers as helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODEL_DIR = os.path.join(ROOT, "diffusiondepth_b200", "model")


def _src_tree(tmp_path):
    """A stand-in for DiffusionDepth/src with `model` -> the mirror (what INTEGRATION.md tells a maintainer to do)."""
    src = tmp_path / "src"
    src.mkdir()
    os.symlink(MODEL_DIR, src / "model")
    return str(src)


def _run(code, paths, argv=(), **extra_env):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(paths), **extra_env)
    return subprocess.run([sys.executable, "-c", textwrap.dedent(code), *argv], env=env, capture_output=True, text=True,
                          timeout=600)


def test_mirror_imports_as_toplevel_model(tmp_path):
    """`import model` through the symlink: no relative import may climb above the package (round-1 ADVICE)."""
    r = _run("""
        import sys
        from argparse import Namespace
        import model
        assert model.__name__ == "model" and "diffusiondepth_b200.model" not in sys.modules
        args = Namespace(model_name="Diffusion_DCbase_", backbone_module="mmbev_resnet", backbone_name="mmbev_res18",
                         head_specify="DDIMDepthEstimate_Res", inference_steps=5, num_train_timesteps=1000)
        net = model.get(args)(args)
        from model.backbone import get as get_bb
        from model.diffusers.schedulers.scheduling_ddim import DDIMScheduler
        from model.ops.depth_transform import DEPTH_TRANSFORM
        from model.head import DDIMDepthEstimate_Swin_ADDHAHI, DDIMDepthEstimate_Swin_ADDHAHIVis
        assert type(net).__module__ == "model.diffusion_dcbase_model" and len(net.state_dict()) == 190
        print("OK", type(net).__name__)
        """, [_src_tree(tmp_path), ROOT])
    assert r.returncode == 0 and "OK Diffusion_DCbase_Model" in r.stdout, r.stderr[-2000:]


def test_main_py_test_runs_up_to_the_first_cuda_call(tmp_path):
    """The reference's src/main.py::test() (:404-470) on the mirror, with the Namespace the reference's config.py +
    check_args produce for the usual flags (tests/golden/ref_main_args.json, oracle.make_golden.fixture_main_args):
    `model` imported through the symlink, get_model(args)(args), a checkpoint through load_state_dict(strict=False),
    nn.DataParallel, a DataLoader(batch_size=1) of the reference's sample dicts, net(sample).  With no GPU visible,
    `.cuda()` is a no-op and the forward must then fail LOUDLY in the plugin (EngineError: no CPU path) — i.e. the
    sequence got all the way there."""
    ckpt = tmp_path / "model_00001.pt"
    m = helpers.build_mirror("res18", 5)
    torch.save({"net": m.state_dict(), "args": None}, ckpt)
    r = _run("""
        import json, os, sys, torch
        from argparse import Namespace
        from torch import nn
        from torch.utils.data import DataLoader, Dataset
        torch.nn.Module.cuda = lambda self, *a, **k: self          # no GPU visible
        torch.Tensor.cuda = lambda self, *a, **k: self
        import model
        assert model.__file__.startswith(os.environ["DD_TMP_SRC"]), model.__file__   # ... running on the mirror
        from model import get as get_model
        with open(sys.argv[1]) as f:
            args = Namespace(**json.load(f), pretrain=sys.argv[2], save_dir=os.environ["DD_TMP_EXP"])
        args.num_threads = 0
        class TwoSamples(Dataset):                                   # emits the reference's sample dict (kittidc.py:273)
            def __init__(self, args, mode): pass
            def __len__(self): return 2
            def __getitem__(self, i):
                g = torch.Generator().manual_seed(i)
                dep = torch.rand(1, 36, 52, generator=g) * 80
                return dict(rgb=torch.randn(3, 36, 52, generator=g), dep=dep, gt=dep, K=torch.zeros(4),
                            depth_mask=dep > 0, depth_map=dep)
        try:
            loader_test = DataLoader(dataset=TwoSamples(args, 'test'), batch_size=1, shuffle=False,
                                     num_workers=args.num_threads)
            net = get_model(args)(args)
            net.cuda()
            checkpoint = torch.load(args.pretrain)
            key_m, key_u = net.load_state_dict(checkpoint['net'], strict=False)
            if key_m:
                raise KeyError(key_m)
            net = nn.DataParallel(net)
            net.eval()
            for batch, sample in enumerate(loader_test):
                sample = {key: val.cuda() for key, val in sample.items() if val is not None}
                with torch.no_grad():
                    output = net(sample)
        except Exception as e:
            print("RAISED", type(e).__name__, str(e)[:120])
        """, [_src_tree(tmp_path), ROOT], [os.path.join(helpers.GOLDEN_DIR, "ref_main_args.json"), str(ckpt)],
             DD_TMP_SRC=str(tmp_path), DD_TMP_EXP=str(tmp_path / "exp"), CUDA_VISIBLE_DEVICES="")
    assert "RAISED EngineError" in r.stdout and "no CPU path" in r.stdout, (r.stdout[-1500:], r.stderr[-1500:])


def test_deepcopy_and_replica_do_not_share_engines_or_bridges():
    """round-1 ADVICE: weakrefs / engine caches copied verbatim made a copied model run with the ORIGINAL's weights."""
    from diffusiondepth_b200.model.head._ddim_head import collect_tensors
    m = helpers.build_mirror("res18", 5)
    c = copy.deepcopy(m)
    assert c.depth_head.model._bridge() is c.depth_head and m.depth_head.model._bridge() is m.depth_head
    assert c.depth_head._engines is not m.depth_head._engines and len(c.depth_head._engines) == 0
    assert c.depth_head._backbone_ref is None
    with torch.no_grad():
        c.depth_head.model.pred[0].weight.add_(1.0)
    assert not torch.equal(c.depth_head.model.pred[0].weight, m.depth_head.model.pred[0].weight)
    # what the engine packs == the state_dict, also for an nn.DataParallel replica (parameters are plain attributes there)
    want = {k: v for k, v in m.depth_backbone.state_dict(keep_vars=True).items()}
    got = collect_tensors(m.depth_backbone)
    assert list(got) == list(want) and all(got[k] is want[k] for k in want)
    from torch.nn.parallel.replicate import replicate
    if torch.cuda.is_available():
        rep = replicate(m.cuda(), [0])[0]
        got = collect_tensors(rep.depth_backbone)
        assert sorted(got) == sorted(want)


# ------------------------------------------------------------------------------------------------ GPU: the sequence itself
def _main_py_test_sequence(src, family, case, tmp_path, device_ids=None):
    """reference src/main.py:404-470, line for line, with `model` imported as the top-level package from `src`."""
    g = helpers.load_golden(case)
    code = """
        import sys, json, torch
        from argparse import Namespace
        from torch import nn
        from torch.utils.data import DataLoader, Dataset
        sys.path.insert(0, sys.argv[2]); sys.path.insert(0, sys.argv[3])
        from oracle import configs, restate
        from model import get as get_model                                     # main.py:18
        family, T, B, H, W, ckpt, out_path, ids = json.loads(sys.argv[1])
        args = configs.make_args(family, T)

        class Synthetic(Dataset):                                              # main.py:406-411 (synthetic stand-in)
            def __len__(self): return B
            def __getitem__(self, i):
                s = restate.synthetic_sample(1, H, W, configs.SEED_INPUTS, first=i)
                s = {k: v[0] for k, v in s.items()}
                s["noise"] = restate.synthetic_noise(1, H, W, configs.SEED_NOISE, first=i)[0]  # reproducible x_T
                return s
        loader_test = DataLoader(dataset=Synthetic(), batch_size=1, shuffle=False, num_workers=0)
        model = get_model(args)                                                # :414
        net = model(args)                                                      # :415
        net.cuda()                                                             # :416
        checkpoint = torch.load(ckpt)                                          # :422
        key_m, key_u = net.load_state_dict(checkpoint['net'], strict=False)    # :423
        assert not key_m and not key_u, (key_m, key_u)                         # :425-432 (missing keys raise there)
        net = nn.DataParallel(net, device_ids=ids)                             # :434
        net.eval()                                                             # :448
        preds, keys = [], None
        for batch, sample in enumerate(loader_test):                           # :456
            sample = {key: val.cuda() for key, val in sample.items() if val is not None}   # :457-458
            with torch.no_grad():                                              # :462-464 (opt_level O0)
                output = net(sample)
            preds.append(output['pred'].cpu()); keys = sorted(output.keys())
        torch.save({"pred": torch.cat(preds), "keys": keys}, out_path)
        print("SEQUENCE_OK")
        """
    import json
    m = helpers.build_mirror(family, g["T"])
    ckpt = tmp_path / "model_00001.pt"
    torch.save({"net": {k: v.cpu() for k, v in m.state_dict().items()}, "args": None}, ckpt)
    out = tmp_path / "out.pt"
    r = _run(code, [src, ROOT], [json.dumps([family, g["T"], g["B"], g["H"], g["W"], str(ckpt), str(out), device_ids]),
                                 ROOT, os.path.join(ROOT, "tests")])
    assert r.returncode == 0 and "SEQUENCE_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])
    return g, torch.load(out)


@pytest.mark.gpu
@pytest.mark.parametrize("family,case,device_ids", [("res18", "g_res18_ragged", None), ("res18", "g_res18_ragged", [0, 0]),
                                                    ("swinl", "g_swinl_small", None)])
def test_main_py_test_sequence_on_the_mirror(tmp_path, family, case, device_ids):
    """device_ids=[0, 0] forces nn.DataParallel through scatter / replicate / parallel_apply / gather on one GPU (what
    main.py does on a multi-GPU box at batch 1)."""
    g, res = _main_py_test_sequence(_src_tree(tmp_path), family, case, tmp_path, device_ids)
    assert res["keys"] == sorted(str(k) for k in g["z"]["output_keys"])
    pred = helpers.golden_view(g, "pred", res["pred"])
    ref, z_ref = torch.from_numpy(g["z"]["pred"]), torch.from_numpy(g["z"]["logits"])
    rel = (pred - ref).abs() / ref.abs().clamp_min(1e-6)
    well = (z_ref < 6) & (z_ref > -13)
    assert rel[well].max().item() < 1e-3
    assert ((pred >= 999998.0) == (ref >= 999998.0))[z_ref < -14.5].all()
