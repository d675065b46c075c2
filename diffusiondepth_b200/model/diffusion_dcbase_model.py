"""`Diffusion_DCbase_Model` — the plugin class `src/main.py` instantiates and calls
(reference src/model/diffusion_dcbase_model.py:24-224).  sample dict in, 13-key dict out."""
import torch
import torch.nn as nn

from ._blocks import exact_fp32
from .backbone import get as get_backbone
from .registry import HEADS
from . import head as _heads  # noqa: F401  (registers the head classes)


class Diffusion_DCbase_Model(nn.Module):
    def __init__(self, args, depth_backbone=None, depth_head=None, ip_basic=False, depth_keys='all', **unused):
        super().__init__()
        self.args = args
        if ip_basic:
            raise NotImplementedError("ip_basic pre-filling is a CPU/cv2 data-prep path; out of scope")
        self.depth_backbone = depth_backbone if depth_backbone is not None else get_backbone(args)()
        if depth_head is None:
            steps = getattr(args, 'inference_steps', 20)
            train_steps = getattr(args, 'num_train_timesteps', 1000)
            if getattr(args, 'head_specify', None) is None:
                raise ValueError("args.head_specify must name a DDIM head (e.g. DDIMDepthEstimate_Swin_ADDHAHI)")
            depth_head = HEADS.build(dict(
                type=args.head_specify, in_channels=[64, 128, 256, 512], inference_steps=steps,
                num_train_timesteps=train_steps, depth_feature_dim=16,
                loss_cfgs=[dict(loss_func='l1_depth_loss', name='depth_loss', weight=0.2, pred_indices=0, gt_indices=0),
                           dict(loss_func='l1_depth_loss', name='blur_depth_loss', weight=0.1, pred_indices=1,
                                gt_indices=0)],
                init_cfg=args))
        self.depth_head = depth_head
        self.depth_keys = depth_keys
        if hasattr(self.depth_head, "attach_backbone"):
            self.depth_head.attach_backbone(self.depth_backbone)

    def extract_depth(self, img, depth_map, depth_mask, gt_depth_map, return_loss=False, img_metas=None,
                      weight_map=None, instance_masks=None, **kwargs):
        B, C, H, W = img.shape
        depth_map = depth_map.view(B, 1, *depth_map.shape[-2:])
        if gt_depth_map is not None:
            gt_depth_map = gt_depth_map.view(B, 1, *depth_map.shape[-2:])
        depth_mask = depth_mask.view(*depth_map.shape)
        head = self.depth_head
        if hasattr(head, "can_run_backbone") and head.can_run_backbone(self.depth_backbone, img):
            fp = None  # the engine runs the Swin backbone itself (DenoiseEngine.run_backbone)
        else:
            with torch.no_grad(), exact_fp32():
                fp = self.depth_backbone(img)
        # the backbone travels with the call: an nn.DataParallel replica / deep copy of this model then packs ITS weights
        extra = {'backbone': self.depth_backbone} if hasattr(head, "can_run_backbone") else {}
        return self.depth_head(fp, depth_map, depth_mask, gt_depth_map=gt_depth_map, return_loss=return_loss,
                               weight_map=weight_map, instance_masks=instance_masks, image=img, **extra, **kwargs)

    def forward(self, sample):
        extra = {k: sample[k] for k in ('noise', 'step_noise') if k in sample}  # seeded / sharded runs inject the draws
        return self.extract_depth(sample['rgb'], sample['depth_map'], sample['depth_mask'], sample['gt'],
                                  return_loss=True, sparse_depth=sample['dep'], **extra)
