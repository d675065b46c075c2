"""On-disk contract around the path: official-Swin key/row conversion, checkpoint ingestion, KITTI PNG values."""
import os

import numpy as np
import pytest
import torch

from diffusiondepth_b200 import io as ddio
from diffusiondepth_b200.model.backbone.convert_ckpt import swin_convert
from oracle import make_golden
import dd_helpers as helpers


def test_swin_convert_names_and_merge_order():
    src = make_golden.official_swin_like()
    out = swin_convert(src)
    assert "head.weight" not in out
    for k in ("patch_embed.projection.weight", "stages.0.blocks.0.attn.w_msa.qkv.weight",
              "stages.0.blocks.0.attn.w_msa.relative_position_bias_table", "stages.0.blocks.0.ffn.layers.0.0.weight",
              "stages.0.blocks.0.ffn.layers.1.bias", "stages.0.blocks.0.norm1.weight",
              "stages.0.downsample.reduction.weight", "stages.0.downsample.norm.bias", "norm.weight"):
        assert k in out, k
    # semantic check of the permutation: official concat [x0,x1,x2,x3] (positions (0,0),(1,0),(0,1),(1,1)) vs unfold
    C = 8
    x = torch.randn(1, C, 4, 6)
    x0, x1, x2, x3 = x[:, :, 0::2, 0::2], x[:, :, 1::2, 0::2], x[:, :, 0::2, 1::2], x[:, :, 1::2, 1::2]
    official = torch.cat([x0, x1, x2, x3], 1).flatten(2).transpose(1, 2)          # [1, L, 4C]
    unfold = torch.nn.functional.unfold(x, 2, stride=2).transpose(1, 2)          # [1, L, 4C] channel-major
    w = src["layers.0.downsample.reduction.weight"]
    assert torch.allclose(official @ w.t(), unfold @ out["stages.0.downsample.reduction.weight"].t(), atol=1e-5)
    g = src["layers.0.downsample.norm.weight"]
    assert torch.allclose((official * g).sum(-1), (unfold * out["stages.0.downsample.norm.weight"]).sum(-1), atol=1e-5)


def test_swin_convert_matches_reference():
    """Against the reference's swin_convert of the same checkpoint (tests/golden/ref_swin_convert.npz)."""
    ref = np.load(os.path.join(helpers.GOLDEN_DIR, "ref_swin_convert.npz"), allow_pickle=False)
    b = swin_convert(make_golden.official_swin_like())
    assert list(b) == ref["keys"].tolist()
    for i, k in enumerate(b):
        assert torch.equal(b[k], torch.from_numpy(ref[f"v{i}"])), k


def test_checkpoint_ingestion_and_png(tmp_path):
    import dd_helpers
    m = dd_helpers.build_mirror("res18", 5)
    path = tmp_path / "model_00001.pt"
    torch.save({"net": {"module." + k: v for k, v in m.state_dict().items()}, "args": {"inference_steps": 5}}, path)
    args = ddio.load_reference_checkpoint(m, str(path))
    assert args == {"inference_steps": 5}
    sd = m.state_dict()
    sd.pop("depth_head.model.pred.0.weight")
    torch.save({"net": sd}, path)
    with pytest.raises(KeyError, match="Missing keys"):
        ddio.load_reference_checkpoint(m, str(path))
    pred = torch.tensor([[[[0.5, -1.0], [80.0, 255.99]]]])
    png = ddio.depth_to_kitti_png(pred)
    assert png.dtype == np.uint16 and png.tolist() == [[128, 0], [20480, 65533]]
    ddio.save_kitti_png(pred, str(tmp_path / "x.png"))
    from PIL import Image
    assert np.array(Image.open(tmp_path / "x.png")).tolist() == png.tolist()
