"""Shared machinery of the DDIM depth heads: parameter containers with the reference's key layout and the
bridge to the CUDA engine.

Reference call chain being replaced (src/model/head/ddim_depth_estimate_res_swin_addHAHI.py):
  forward :87-185  ->  encoder t() :102, hahineck :110, FPN :112-122, pipeline(...) :130-144 =
  CNNDDIMPipiline.__call__ :254-303 (T x {denoiser :361-382, DDIMScheduler.step})  ->  depth_transform.inv_t :146.
Here all of it — and the backbone in front of it — runs inside the CUDA engine (C ABI, include/dd_engine.h) whenever the
engine instantiates the architecture; the torch modules below only hold the parameters under the reference's keys.
The torch-op producer path (TF32 off) remains for architectures the engine does not instantiate.

The engine bits are imported absolutely (`diffusiondepth_b200.*`), everything else relatively, so that this package
works both as `diffusiondepth_b200.model` and as the reference's top-level `model` (INTEGRATION.md: symlink into
`src/`, tested by tests/test_dropin.py)."""
import collections
import copy
import threading
import weakref
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from diffusiondepth_b200._cabi import EngineError
from diffusiondepth_b200.engine import (DECODER_KEYS, DENOISER_KEYS, ENCODER_KEYS, FUSE_KEYS, DenoiseEngine,
                                        WorkspacePool)
from .._blocks import ConvModule, exact_fp32
from ..diffusers.schedulers.scheduling_ddim import DDIMScheduler
from ..ops import depth_transform as _codec  # noqa: F401  (registers the codec classes)
from ..registry import DEPTH_TRANSFORM
from ._pipeline import CNNDDIMPipiline, draw_step_noise

FPN_DIM = 256
MAX_ENGINES = 4  # per head: least-recently-used engines beyond this are closed (packed weights + CUDA graphs freed)


def collect_tensors(module: nn.Module, prefix: str = "") -> Dict[str, torch.Tensor]:
    """`module.state_dict(keep_vars=True)` that also works on `nn.DataParallel` replicas, whose parameters are plain
    tensor attributes listed in `_former_parameters` (torch/nn/parallel/replicate.py) and absent from `state_dict()`."""
    out: Dict[str, torch.Tensor] = {}

    def walk(m, pre):
        for k, v in m._parameters.items():
            if v is not None:
                out[pre + k] = v
        for k, v in getattr(m, "_former_parameters", {}).items():
            if v is not None:
                out.setdefault(pre + k, v)
        for k, v in m._buffers.items():
            if v is not None and k not in m._non_persistent_buffers_set:
                out[pre + k] = v
        for k, c in m._modules.items():
            if c is not None:
                walk(c, pre + k + ".")

    walk(module, prefix)
    return out


def _gn_conv_stack(cin, mid, cout):
    """conv3x3 -> GN(4) -> ReLU -> conv3x3 -> GN(4) -> ReLU; indices 0,1,3,4 carry parameters."""
    return nn.Sequential(nn.Conv2d(cin, mid, 3, 1, 1), nn.GroupNorm(4, mid), nn.ReLU(True),
                         nn.Conv2d(mid, cout, 3, 1, 1), nn.GroupNorm(4, cout), nn.ReLU(True))


class UpSample_add(nn.Module):
    """Parameters of the Swin heads' fusion block: convA / convB = bare 3x3 conv + bias (head :321-333)."""

    def __init__(self, cin, cout):
        super().__init__()
        self.convA = ConvModule(cin, cout, 3, padding=1, norm=False, act=False)
        self.convB = ConvModule(cout, cout, 3, padding=1, norm=False, act=False)


class ScheduledCNNRefine(nn.Module):
    """The denoiser's parameters (head :336-359 / res.py:301-322).  It has no torch forward: the operator
    `model(noisy, t, cond, None, None, None) -> eps` is served by the engine (`DenoiseEngine.denoiser_forward`)."""

    def __init__(self, channels_in, channels_noise, with_fuse):
        super().__init__()
        self.noise_embedding = _gn_conv_stack(channels_noise, 64, channels_in)
        if with_fuse:
            self.upsample_fuse = UpSample_add(channels_in, channels_in)
        self.time_embedding = nn.Embedding(1280, channels_in)
        self.pred = _gn_conv_stack(channels_in, 64, channels_noise)
        self.__dict__['_bridge'] = None  # weakref to the owning head, set by it

    def forward(self, noisy_image, t, feat, *unused):
        head = self._bridge() if self._bridge is not None else None
        if head is None:
            raise EngineError("ScheduledCNNRefine is not attached to a DDIM head / CUDA engine")
        return head.denoiser(noisy_image, t, feat)


def _fpn_lateral(cin):
    return nn.Sequential(nn.Conv2d(cin, FPN_DIM, 3, 1, 1, bias=False), nn.BatchNorm2d(FPN_DIM), nn.ReLU(True))


def _fpn_up():
    return nn.Sequential(nn.ConvTranspose2d(FPN_DIM, FPN_DIM, 2, 2, bias=False), nn.BatchNorm2d(FPN_DIM), nn.ReLU(True))


class DDIMHeadBase(nn.Module):
    """Common ctor surface: HEADS.build(dict(type=..., in_channels, inference_steps, num_train_timesteps,
    depth_feature_dim=16, loss_cfgs, init_cfg=args)) as in reference diffusion_dcbase_model.py:77-91."""

    variant = "res"          # engine variant
    fpn_in_channels = (64, 128, 256, 512)
    has_neck = False         # HAHI neck in front of the FPN (the *HAHI heads)
    return_intermediates = False  # *Vis heads: also decode every intermediate latent -> 'pred_inter'

    def __init__(self, in_channels=None, up_scale_factor=1, inference_steps=20, num_train_timesteps=1000,
                 return_indices=None, depth_transform_cfg=None, detach_fp=False, depth_embed_dim=16,
                 depth_feature_dim=16, loss_cfgs=(), init_cfg=None, **unused):
        super().__init__()
        self.init_cfg, self.detach_fp, self.loss_cfgs = init_cfg, detach_fp, list(loss_cfgs)
        self.return_indices = return_indices
        self.depth_embed_dim = depth_embed_dim
        cfg = depth_transform_cfg or dict(type="DeepDepthTransformWithUpsampling", hidden=16, eps=1e-6)
        self.depth_transform = DEPTH_TRANSFORM.build(cfg)
        self.model = ScheduledCNNRefine(FPN_DIM, depth_feature_dim, with_fuse=self.variant == "swin")
        self.model.__dict__['_bridge'] = weakref.ref(self)  # plain attribute: must not register as a submodule
        self.diffusion_inference_steps = inference_steps
        self.scheduler = DDIMScheduler(num_train_timesteps=num_train_timesteps, clip_sample=False)
        self.conv_lateral = nn.ModuleList(_fpn_lateral(c) for c in self.fpn_in_channels)
        self.conv_up = nn.ModuleList(_fpn_up() for _ in self.fpn_in_channels[1:])
        # engine state (not parameters)
        self.eval_ddim_loss = False       # reference computes it in eval too; it is RNG noise there
        self.use_cuda_graph = True
        self.check_range = True
        self.capture_logits = False      # tests: also keep the decoder's pre-sigmoid z of the last forward
        self.native_producers = True     # neck + FPN on the engine's tensor-core conv path when the pyramid allows
        self.native_backbone = True      # Swin-L backbone on the engine's GEMM/attention path (needs native_producers)
        self.fp8_corrections = True      # Swin heads: correction products of convA / convB as e4m3 MMAs (DD_FLAG_FP8_CORR;
        #                                  ~1.5x on the dominant kernel, max |dz| 3.4e-4 of the 1e-3 budget on config 3).
        #                                  False = the exact 3-pass fp16 split everywhere.
        self.__dict__['_backbone_ref'] = None  # weakref to the model's depth_backbone (Diffusion_DCbase_Model passes the
        #                                        backbone with every call; this is the fallback for direct head calls)
        self.capture_cond = False        # tests: keep the NCHW condition map of the last forward
        self.noise_generator: Optional[torch.Generator] = None
        self.ddim_eta = 0.0  # eta of the DDIM sampler forward() runs (reference pipeline `eta=`); > 0: stochastic DDIM
        self._reset_engine_state()

    def _reset_engine_state(self):
        self.__dict__['_engines'] = collections.OrderedDict()  # key -> DenoiseEngine, least recently used first
        self.__dict__['_packed'] = {}                          # key -> (tensor list, signature) of the packed weights
        self.__dict__['_pools'] = {}                           # device -> WorkspacePool
        self.__dict__['_lock'] = threading.RLock()             # nn.DataParallel replicas (threads) share the three dicts

    def invalidate_engines(self):
        """Close every engine (call after replacing Parameter OBJECTS; in-place updates, load_state_dict and .to() are
        picked up automatically through data_ptr / _version)."""
        for e in self._engines.values():
            e.close()
        self._reset_engine_state()

    def __deepcopy__(self, memo):
        """copy.deepcopy(model) (EMA / eval copies): the copy gets its own engines, packed from ITS parameters, and its
        denoiser operator bridges to the copy — never to the original's ctypes handles or weights."""
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k in ("_engines", "_packed", "_pools", "_backbone_ref", "_lock"):
                continue
            new.__dict__[k] = copy.deepcopy(v, memo)
        new.__dict__['_backbone_ref'] = None
        new._reset_engine_state()
        new.model.__dict__['_bridge'] = weakref.ref(new)
        return new

    def _replicate_for_data_parallel(self):
        """nn.DataParallel replicas (reference src/main.py:434): same idea — the replica bridges to itself and reads the
        replica's (broadcast) tensors; engines are cached per device in the dict shared with the original."""
        replica = super()._replicate_for_data_parallel()
        replica.__dict__['_backbone_ref'] = None
        return replica

    @property
    def pipeline(self) -> CNNDDIMPipiline:
        """`self.pipeline(batch_size, device, dtype, shape, input_args, generator, eta, num_inference_steps, return_dict)`
        of the reference heads (head :49, :254-303), served by this head's engines (_pipeline.py)."""
        return CNNDDIMPipiline(self.model, self.scheduler, with_image_list=bool(self.return_intermediates))

    # ------------------------------------------------------------------------------------------ engine bridge
    def _engine_tensors(self):
        sd = {}
        for k in DENOISER_KEYS + DECODER_KEYS + ENCODER_KEYS + (FUSE_KEYS if self.variant == "swin" else ()):
            mod, _, leaf = k.rpartition(".")
            obj = self.get_submodule(mod)
            sd[k] = getattr(obj, leaf)
        return sd

    def _producer_tensors(self):
        sd = {}
        for name in ("hahineck", "conv_lateral", "conv_up"):
            if name in self._modules:
                sd.update(collect_tensors(self._modules[name], name + "."))
        return sd

    @staticmethod
    def _sizes_ok(sizes):
        """Native FPN: each level at most 2x its coarser neighbour (== 2x: adaptive_avg_pool2d is the identity;
        smaller, e.g. 57 vs 2*29: the engine's pooling kernel resamples)."""
        return all(b[0] <= a[0] <= 2 * b[0] and b[1] <= a[1] <= 2 * b[1] for a, b in zip(sizes[:-1], sizes[1:]))

    @classmethod
    def _pyramid_ok(cls, feats):
        return cls._sizes_ok([tuple(f.shape[-2:]) for f in feats]) and all(f.shape[1] % 8 == 0 for f in feats)  # 16-byte NHWC rows (TMA)

    def attach_backbone(self, backbone):
        self.__dict__['_backbone_ref'] = weakref.ref(backbone)

    def _backbone(self, given=None):
        if given is not None:
            return given
        bb = self._backbone_ref() if self._backbone_ref is not None else None
        if bb is None:
            raise EngineError("native backbone requested but no backbone module is attached to this head "
                              "(Diffusion_DCbase_Model passes it; direct callers use head.attach_backbone)")
        return bb

    @staticmethod
    def swin_pyramid(image_hw):
        """Stage output sizes of a patch-4 Swin for an (H, W) image, finest first."""
        h, w = (image_hw[0] + 3) // 4, (image_hw[1] + 3) // 4
        sizes = []
        for _ in range(4):
            sizes.append((h, w))
            h, w = (h + 1) // 2, (w + 1) // 2
        return sizes

    @staticmethod
    def resnet_pyramid(image_hw):
        """Stage output sizes of the stem-less stride-2-per-stage ResNet (3x3, pad 1), finest first."""
        h, w = image_hw
        sizes = []
        for _ in range(4):
            h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
            sizes.append((h, w))
        return sizes

    def backbone_pyramid(self, image_hw, backbone=None):
        """Stage output sizes of this head's backbone family (MPViT halves per stage like the stem-less ResNet)."""
        if self.variant == "swin" and type(backbone).__name__ != "MPViT":
            return self.swin_pyramid(image_hw)
        return self.resnet_pyramid(image_hw)

    @staticmethod
    def mpvit_spec(backbone):
        """(layers per stage, stage widths, paths per stage, mlp ratio) of an MPViT module, or None when it is not one of
        the shapes the engine instantiates (8 heads, crpe windows {3: 2, 5: 3, 7: 3}, <= 3 paths, widths <= 512)."""
        try:
            stages = backbone.mhca_stages
            dims = [st.InvRes.conv1.conv.in_channels for st in stages]
            paths = [len(st.mhca_blks) for st in stages]
            layers = [len(st.mhca_blks[0].MHCA_layers) for st in stages]
            blk = stages[0].mhca_blks[0].MHCA_layers[0]
            ratio = blk.mlp.fc1.out_features // dims[0]
            ok = (len(stages) == 4 and max(paths) <= 3 and max(dims) <= 512 and all(d % 8 == 0 for d in dims)
                  and dims[0] % 16 == 0 and blk.factoratt_crpe.num_heads == 8
                  and [c.kernel_size[0] for c in stages[0].mhca_blks[0].crpe.conv_list] == [3, 5, 7]
                  and all(st.mhca_blks[0].MHCA_layers[0].mlp.fc1.out_features == ratio * d for st, d in zip(stages, dims))
                  and list(backbone.out_channels) == dims[1:] + dims[-1:])
            return (layers, dims, paths, ratio) if ok else None
        except (AttributeError, IndexError):
            return None

    def can_run_backbone(self, backbone, img) -> bool:
        """Native backbone path: CUDA input and an architecture the engine instantiates — Swin-L for the Swin heads,
        BasicBlock ResNetForMMBEV (64/128/256/512, stride 2 per stage) for the Res heads, MPViT for the MPViT head."""
        if not (self.native_producers and self.native_backbone and img.is_cuda):
            return False
        name = type(backbone).__name__
        if name == "MPViT":
            spec = self.mpvit_spec(backbone)
            if spec is None or self.variant != "swin" or list(self.fpn_in_channels) != list(backbone.out_channels):
                return False
        elif self.variant == "swin":
            if name != "SwinTransformer" or getattr(backbone, "num_features", None) != [192, 384, 768, 1536]:
                return False
            if [len(s.blocks) for s in backbone.stages] != [2, 2, 18, 2]:
                return False
        else:
            if name != "ResNetForMMBEV" or list(backbone.backbone_output_ids) != [0, 1, 2, 3]:
                return False
            if [st[0].conv2.out_channels for st in backbone.layers] != [64, 128, 256, 512]:
                return False
        return self._sizes_ok(self.backbone_pyramid(img.shape[-2:], backbone))

    def _gather(self, native, image_hw, backbone):
        tensors = self._engine_tensors()
        if native:
            tensors.update(self._producer_tensors())
        if image_hw is not None:
            for k, v in collect_tensors(self._backbone(backbone), "backbone.").items():
                if v.is_floating_point():
                    tensors[k] = v
        return tensors

    def _engine(self, batch, latent_hw, cond_hw, device, feats=None, image_hw=None, backbone=None, steps=None,
                eta=0.0, latent_steps=False) -> DenoiseEngine:
        """feats: backbone feature maps, or a (channels, sizes) pyramid spec -> native neck/FPN;
        image_hw: additionally run the backbone natively (`backbone`: the module holding its parameters);
        steps: T (default diffusion_inference_steps); eta > 0 or latent_steps (the latent after every step): a
        stochastic engine (dd_denoise_decode_stochastic) with that eta's schedule."""
        with self._lock:
            return self._engine_locked(batch, latent_hw, cond_hw, device, feats, image_hw, backbone,
                                       self.diffusion_inference_steps if steps is None else int(steps), float(eta),
                                       bool(latent_steps))

    def _engine_locked(self, batch, latent_hw, cond_hw, device, feats, image_hw, backbone, steps=None, eta=0.0,
                       latent_steps=False) -> DenoiseEngine:
        native = feats is not None
        if native and not isinstance(feats, tuple):
            feats = ([f.shape[1] for f in feats], [tuple(f.shape[-2:]) for f in feats])
        device = torch.device(device)
        steps = self.diffusion_inference_steps if steps is None else steps
        stochastic = eta > 0 or latent_steps
        key = (batch, tuple(latent_hw), tuple(cond_hw), str(device), steps,
               self.use_cuda_graph, native, tuple(image_hw) if image_hw is not None else None,
               bool(self.return_intermediates), bool(self.fp8_corrections), float(eta), bool(latent_steps))
        eng = self._engines.get(key)
        if eng is None:
            pool = self._pools.setdefault(str(device), WorkspacePool(device))
            eng = DenoiseEngine(self.variant, batch, latent_hw, cond_hw, steps, device,
                                cuda_graph=self.use_cuda_graph, check_range=False,
                                step_decode=bool(self.return_intermediates), workspace_pool=pool,
                                fp8_corr=bool(self.fp8_corrections), stochastic=stochastic)
            if native:
                eng.enable_producers(feats[0], feats[1], has_neck=self.has_neck)
            if image_hw is not None:
                if type(self._backbone(backbone)).__name__ == "MPViT":
                    layers, dims, paths, ratio = self.mpvit_spec(self._backbone(backbone))
                    eng.enable_backbone(image_hw, depths=layers, kind="mpvit", mp_dims=dims, mp_paths=paths, mlp_ratio=ratio)
                elif self.variant == "swin":
                    eng.enable_backbone(image_hw)
                else:
                    eng.enable_backbone(image_hw, depths=[len(st) for st in self._backbone(backbone).layers], kind="resnet")
            if stochastic:
                eng.set_schedule(*self.scheduler.stochastic_coefficients(steps, eta))
            else:
                ts, cx, ce = self.scheduler.fused_coefficients(steps)
                eng.set_schedule(ts, cx, ce)
            self._engines[key] = eng
            self._packed.pop(key, None)
            while len(self._engines) > MAX_ENGINES:  # a ragged last batch / a new image size must not pile up engines
                old_key, old = self._engines.popitem(last=False)
                old.close()
                self._packed.pop(old_key, None)
        else:
            self._engines.move_to_end(key)
        # Re-pack when a parameter changed.  The ~500 tensors are walked once per pack; per forward only their
        # (data_ptr, _version) pairs are compared (0.3 ms instead of 2.6 ms for a Swin-L model).
        packed = self._packed.get(key)
        if packed is not None and packed[2] is not (backbone if image_hw is not None else None):
            packed = None  # a different backbone module (DataParallel replica): look its tensors up again
        if packed is None:
            tensors = self._gather(native, image_hw, backbone)
            sig = None
        else:
            tensors = packed[0]
            sig = tuple((t.data_ptr(), t._version) for t in tensors.values())
        if packed is None or sig != packed[1]:
            if packed is not None:  # something changed: the owning modules may hold new tensors
                tensors = self._gather(native, image_hw, backbone)
            eng.load_weights(tensors)
            self._packed[key] = (tensors, tuple((t.data_ptr(), t._version) for t in tensors.values()),
                                 backbone if image_hw is not None else None)
        return eng

    def _any_engine(self, batch, latent_hw, cond_hw, device):
        """An engine of this geometry for the bare operators (denoiser / decode): reuse the forward's engine (same
        packed denoiser + codec weights) instead of packing a second one."""
        want = (batch, tuple(latent_hw), tuple(cond_hw), str(torch.device(device)))
        for key in reversed(self._engines):
            if key[:4] == want and key[4] == self.diffusion_inference_steps and self._packed.get(key) is not None:
                tensors, sig, _ = self._packed[key]
                if tuple((t.data_ptr(), t._version) for t in tensors.values()) == sig:
                    self._engines.move_to_end(key)
                    return self._engines[key]
                break
        return self._engine(batch, latent_hw, cond_hw, device)

    def denoiser(self, noisy, t, cond):
        """`self.model(noisy, t, cond, None, None, None)` of the reference, on the engine."""
        B = noisy.shape[0]
        eng = self._any_engine(B, noisy.shape[-2:], cond.shape[-2:], noisy.device)
        tl = t.reshape(-1).tolist() if torch.is_tensor(t) else t
        return eng.denoiser_forward(cond.contiguous().float(), noisy.contiguous().float(), tl)

    def sample_latents(self, cond, x_T, step_noise, eta, steps, latent_steps=False):
        """The DDIM loop alone on the engine (the pipeline's work): cond [B,256,hc,wc], x_T [B,16,h,w], step_noise
        [T,B,16,h,w] (None: eta = 0) -> (final latent, latent after every step [T,B,16,h,w] or None)."""
        B = x_T.shape[0]
        eng = self._engine(B, x_T.shape[-2:], cond.shape[-2:], x_T.device, steps=steps, eta=eta,
                           latent_steps=latent_steps)
        if eng.stochastic:
            if step_noise is None:  # eta = 0 with per-step latents: sigma = 0, the noise is never weighted in
                step_noise = torch.zeros((steps, *x_T.shape), device=x_T.device, dtype=torch.float32)
            _, latent, lsteps, _, _ = eng.denoise_decode_stochastic(cond, x_T, step_noise.contiguous().float(),
                                                                    want_latent=True, want_latent_steps=latent_steps)
        else:
            _, latent, _ = eng.denoise_decode(cond, x_T, want_latent=True)
            lsteps = None
        if self.check_range:
            eng.poll_status()
        return latent, lsteps

    # ------------------------------------------------------------------------------------------ condition path
    def _condition(self, fp):
        """Top-down FPN that builds the 256-channel condition map x (head :112-122 / res.py:108-118)."""
        x = None
        for i in reversed(range(len(fp))):
            lat = self.conv_lateral[i](fp[i])
            if x is not None:
                lat = lat + F.adaptive_avg_pool2d(self.conv_up[i](x), lat.shape[-2:])
            x = lat
        return x

    def _neck(self, fp):
        return fp

    def _draw_noise(self, shape, device, dtype, override):
        if override is not None:
            return override.to(device=device, dtype=dtype).contiguous()
        g = self.noise_generator
        if g is not None and g.device.type != torch.device(device).type:
            return torch.randn(shape, generator=g, dtype=dtype).to(device)
        return torch.randn(shape, generator=g, device=device, dtype=dtype)

    def _draw_step_noise(self, steps, shape, device, dtype, override):
        """The stochastic loop's per-step noise [T, *shape]: `override`, or T draws in the reference's order (after x_T)."""
        if override is not None:
            return override.to(device=device, dtype=torch.float32).contiguous()
        g = self.noise_generator
        z = draw_step_noise(steps, shape, g.device if g is not None else device, dtype, g)
        return z.to(device=device, dtype=torch.float32).contiguous()

    # ------------------------------------------------------------------------------------------ forward
    def forward(self, fp, depth_map, depth_mask, gt_depth_map=None, return_loss=False, noise=None, image=None,
                backbone=None, step_noise=None, **kwargs):
        """fp: backbone feature maps — or None, meaning "run the backbone natively from `image`" (the model
        wrapper does that when `can_run_backbone` holds, and passes `backbone` = the module holding its weights).
        With `self.ddim_eta` > 0 the loop is stochastic DDIM; `step_noise` [T,B,16,h,w] then replaces its T draws."""
        with_backbone = fp is None
        if with_backbone:
            B, dev, dtype = image.shape[0], image.device, torch.float32
            sizes = self.backbone_pyramid(image.shape[-2:], self._backbone(backbone))
            native = True
        else:
            if self.detach_fp is not False and self.detach_fp is not None:
                idx = self.detach_fp if isinstance(self.detach_fp, (list, tuple, range)) else range(len(fp))
                fp = [f.detach() if i in idx else f for i, f in enumerate(fp)]
            fp = [f.contiguous().float() for f in fp]
            B, dev, dtype = fp[0].shape[0], fp[0].device, fp[0].dtype
            native = self.native_producers and fp[0].is_cuda and self._pyramid_ok(fp)
        Hd, Wd = gt_depth_map.shape[-2:]
        latent_hw = ((Hd + 1) // 2, (Wd + 1) // 2)  # shape of depth_transform.t(gt): conv3x3 stride 2 pad 1
        gt_map_t = None
        if not native:
            with torch.no_grad(), exact_fp32():
                gt_map_t = self.depth_transform.t(gt_depth_map)
                cond = self._condition(self._neck(fp)).contiguous()
        else:
            cond = None
        x_T = self._draw_noise((B, 16, *latent_hw), dev, dtype, noise)
        eta = float(self.ddim_eta)
        z = self._draw_step_noise(self.diffusion_inference_steps, (B, 16, *latent_hw), dev, dtype, step_noise) \
            if eta > 0 else None
        if native:  # (backbone +) neck + FPN + loop + decoder inside the engine; the condition map never leaves NHWC
            want_cond = self.capture_cond or self.training or self.eval_ddim_loss
            if with_backbone:
                eng = self._engine(B, latent_hw, sizes[0], dev, feats=(list(self.fpn_in_channels), sizes),
                                   image_hw=tuple(image.shape[-2:]), backbone=backbone, eta=eta)
                eng.run_backbone(image.contiguous().float())
                cond = eng.build_condition(None, want_cond=want_cond)
            else:
                eng = self._engine(B, latent_hw, tuple(fp[0].shape[-2:]), dev, feats=fp, eta=eta)
                cond = eng.build_condition(fp, want_cond=want_cond)
            gt_map_t = eng.encode(gt_depth_map.contiguous().float())  # returned as pred_init / gt_map_t only
            loop_cond = None
        else:
            eng = self._engine(B, latent_hw, tuple(cond.shape[-2:]), dev, eta=eta)
            loop_cond = cond
        inter = None
        if z is not None:  # stochastic DDIM: x <- c_x x + c_eps eps + sigma_t z_t (dd_denoise_decode_stochastic)
            refined_depth, refined_depth_t, _, logits, steps = eng.denoise_decode_stochastic(
                loop_cond, x_T.float().contiguous(), z, want_latent=True, want_logits=self.capture_logits,
                want_depth_steps=self.return_intermediates)
            if self.return_intermediates:
                inter = list(steps.unbind(0))
                refined_depth = inter[-1]
        elif self.return_intermediates:  # *Vis heads: inv_t of every intermediate latent, decoded inside the graph
            steps, refined_depth_t, logits = eng.denoise_decode_steps(loop_cond, x_T, want_latent=True,
                                                                      want_logits=self.capture_logits)
            inter = list(steps.unbind(0))
            refined_depth = inter[-1]
        else:
            refined_depth, refined_depth_t, logits = eng.denoise_decode(loop_cond, x_T, want_latent=True,
                                                                        want_logits=self.capture_logits)
        self.last_latent, self.last_logits, self.last_cond = refined_depth_t, logits, cond
        if self.check_range:
            eng.poll_status()  # syncs; raises if an activation left the fp16 split range (DESIGN.md "Numerics")
        ddim_loss = self._ddim_loss(cond, refined_depth_t) if (self.eval_ddim_loss or self.training) \
            else refined_depth.new_zeros(())
        return {'pred': refined_depth, 'pred_init': gt_map_t, 'blur_depth_t': gt_map_t, 'ddim_loss': ddim_loss,
                'gt_map_t': gt_map_t, 'pred_uncertainty': None, 'pred_inter': inter, 'weight_map': None,
                'guidance': None, 'offset': None, 'aff': None, 'gamma': None, 'confidence': None}

    def _ddim_loss(self, cond, latent):
        """Reference head :207-223 — one extra denoiser call on a re-noised latent; RNG-dependent."""
        noise = torch.randn(latent.shape).to(latent.device)
        t = torch.randint(0, self.scheduler.num_train_timesteps, (latent.shape[0],), device=latent.device).long()
        noisy = self.scheduler.add_noise(latent, noise, t)
        return F.mse_loss(self.denoiser(noisy, t, cond), noise)  # == self.model(noisy, t, cond, None, None, None)

    ddim_loss = _ddim_loss
