"""Drop-in boundary (SURVEY.md §8b): same registries / class names / ctor arguments / state_dict keys /
output-dict keys as the reference's src/model, and no silent CPU path."""
import os
from argparse import Namespace

import numpy as np
import pytest
import torch

import diffusiondepth_b200 as dd
from diffusiondepth_b200 import model as plugin
from diffusiondepth_b200.model.registry import DEPTH_TRANSFORM, HEADS
from oracle import configs
import dd_helpers as helpers

OUTPUT_KEYS = ['aff', 'blur_depth_t', 'confidence', 'ddim_loss', 'gamma', 'gt_map_t', 'guidance', 'offset', 'pred',
               'pred_init', 'pred_inter', 'pred_uncertainty', 'weight_map']


def test_registries_expose_reference_names():
    # every head reference src/model/head/__init__.py registers
    for name in ("DDIMDepthEstimate_Res", "DDIMDepthEstimate_Swin_ADDHAHI", "DDIMDepthEstimate_ResVis",
                 "DDIMDepthEstimate_Swin_ADDHAHIVis", "DDIMDepthEstimate_Swin_ADD", "DDIMDepthEstimate_MPVIT_ADDHAHI"):
        assert name in HEADS
    assert "DeepDepthTransformWithUpsampling" in DEPTH_TRANSFORM
    codec = DEPTH_TRANSFORM.build(dict(type='DeepDepthTransformWithUpsampling', hidden=16, eps=1e-6))
    d = torch.rand(1, 1, 10, 14) * 80
    lat = codec.t(d)
    assert lat.shape == (1, 16, 5, 7) and codec.inv_t(lat).shape == (1, 1, 10, 14)
    with pytest.raises(KeyError):
        HEADS.build(dict(type="NoSuchHead"))


def test_model_get_and_backbone_factories():
    args = configs.make_args("res18", 5)
    cls = plugin.get(args)
    assert cls.__name__ == "Diffusion_DCbase_Model"
    with pytest.raises(ModuleNotFoundError):
        plugin.get(Namespace(model_name="NLSPN"))
    from diffusiondepth_b200.model.backbone import get as get_bb
    assert get_bb(args).__name__ == "mmbev_res18"
    feats = get_bb(args)()(torch.randn(1, 3, 228, 304))
    # the only shape fixture in the reference: src/model/backbone/mmbev_resnet.py:214-222
    assert [tuple(f.shape[1:]) for f in feats] == [(64, 114, 152), (128, 57, 76), (256, 29, 38), (512, 15, 19)]


def test_state_dict_layout_res18():
    m = helpers.build_mirror("res18", 5)
    sd = m.state_dict()
    assert len(sd) == 190 and sum(p.numel() for p in m.parameters()) == 16422529  # SURVEY.md Appendix A
    for k in ("depth_head.model.noise_embedding.0.weight", "depth_head.model.time_embedding.weight",
              "depth_head.depth_transform.conv_inv_transform.3.0.bias", "depth_head.convup_fp.0.weight",
              "depth_head.conv_lateral.3.1.running_var", "depth_backbone.layers.0.0.downsample.bias"):
        assert k in sd
    assert sd["depth_head.model.time_embedding.weight"].shape == (1280, 256)
    assert sd["depth_head.depth_transform.conv_inv_transform.0.weight"].shape == (16, 16, 4, 4)


def test_heads_have_no_cpu_fallback():
    m = helpers.build_mirror("res18", 5)
    from oracle import restate
    sample = restate.synthetic_sample(1, 36, 52)
    with pytest.raises(dd.EngineError):
        m(sample)  # CPU tensors: the engine must refuse, not fall back to torch
    with pytest.raises(dd.EngineError):
        m.depth_head.model(torch.zeros(1, 16, 18, 26), torch.tensor(5), torch.zeros(1, 256, 18, 26), None, None, None)


@pytest.mark.parametrize("family", ["res18", "swinl", "swinl_add", "mpvit_s"])
def test_state_dict_matches_reference_key_for_key(family):
    """Against the reference model's state_dict layout (tests/golden/ref_state_dict_layout.npz: key, shape and dtype of
    every entry), and a state_dict of exactly that layout loads into the mirror strictly."""
    ref = np.load(os.path.join(helpers.GOLDEN_DIR, "ref_state_dict_layout.npz"), allow_pickle=False)
    dtypes = {str(d): d for d in (torch.float32, torch.int64)}
    a = {k: torch.zeros([int(s) for s in shape.split("x") if s], dtype=dtypes[dt])
         for k, shape, dt in zip(ref[family + "_keys"].tolist(), ref[family + "_shapes"].tolist(),
                                 ref[family + "_dtypes"].tolist())}
    mine = helpers.build_mirror(family, 5)
    b = mine.state_dict()
    assert sorted(a) == sorted(b)
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, k
    saved = {k: v.clone() for k, v in b.items()}
    mine.load_state_dict(a, strict=True)
    mine.load_state_dict(saved, strict=True)  # build_mirror caches the model for other tests
    if family == "swinl":
        k = "depth_backbone.stages.2.blocks.1.attn.w_msa.relative_position_index"
        assert torch.equal(torch.from_numpy(ref["swinl_relative_position_index"]), b[k])
        assert len(a) == 532


def test_mpvit_spec_of_every_factory():
    """What the head hands to dd_enable_backbone(kind = MPViT) is read off the torch module: layers, widths, paths, mlp
    ratio of the four reference factories (backbone/mpvit.py:743-870); anything the engine does not instantiate -> None."""
    from diffusiondepth_b200.model.backbone import mpvit
    from diffusiondepth_b200.model.head._ddim_head import DDIMHeadBase
    want = {"mpvit_tiny": ([1, 2, 4, 1], [64, 96, 176, 216], [2, 3, 3, 3], 2),
            "mpvit_xsmall": ([1, 2, 4, 1], [64, 128, 192, 256], [2, 3, 3, 3], 4),
            "mpvit_small": ([1, 3, 6, 3], [64, 128, 216, 288], [2, 3, 3, 3], 4),
            "mpvit_base": ([1, 3, 8, 3], [128, 224, 368, 480], [2, 3, 3, 3], 4)}
    for name, spec in want.items():
        bb = getattr(mpvit, name)()
        assert tuple(DDIMHeadBase.mpvit_spec(bb)) == spec, name
    wide = mpvit.MPViT(num_stages=4, num_path=(2, 3, 3, 3), num_layers=(1, 1, 1, 1), embed_dims=(64, 128, 256, 640),
                       mlp_ratios=(4,) * 4, num_heads=(8,) * 4)
    assert DDIMHeadBase.mpvit_spec(wide) is None            # 640 / 8 = 80 channels per head > 64
    assert DDIMHeadBase.mpvit_spec(torch.nn.Identity()) is None
