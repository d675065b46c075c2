"""Python handle over the C ABI: packs a head's parameters into the engine and runs the hot path.

PyTorch is used only for device memory (tensors, caching allocator) and the current stream."""
import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _cabi
from ._cabi import EngineError  # noqa: F401

# reference state_dict keys (relative to `depth_head.`) the engine consumes — SURVEY.md Appendix A
DENOISER_KEYS = (
    "model.noise_embedding.0.weight", "model.noise_embedding.0.bias", "model.noise_embedding.1.weight",
    "model.noise_embedding.1.bias", "model.noise_embedding.3.weight", "model.noise_embedding.3.bias",
    "model.noise_embedding.4.weight", "model.noise_embedding.4.bias", "model.time_embedding.weight",
    "model.pred.0.weight", "model.pred.0.bias", "model.pred.1.weight", "model.pred.1.bias",
    "model.pred.3.weight", "model.pred.3.bias", "model.pred.4.weight", "model.pred.4.bias")
FUSE_KEYS = ("model.upsample_fuse.convA.conv.weight", "model.upsample_fuse.convA.conv.bias",
             "model.upsample_fuse.convB.conv.weight", "model.upsample_fuse.convB.conv.bias")
ENCODER_KEYS = (
    "depth_transform.conv_transform.0.0.weight", "depth_transform.conv_transform.0.1.weight",
    "depth_transform.conv_transform.0.1.bias", "depth_transform.conv_transform.0.1.running_mean",
    "depth_transform.conv_transform.0.1.running_var", "depth_transform.conv_transform.1.0.weight",
    "depth_transform.conv_transform.1.1.weight", "depth_transform.conv_transform.1.1.bias",
    "depth_transform.conv_transform.1.1.running_mean", "depth_transform.conv_transform.1.1.running_var")
DECODER_KEYS = (
    "depth_transform.conv_inv_transform.0.weight", "depth_transform.conv_inv_transform.0.bias",
    "depth_transform.conv_inv_transform.1.weight", "depth_transform.conv_inv_transform.1.bias",
    "depth_transform.conv_inv_transform.1.running_mean", "depth_transform.conv_inv_transform.1.running_var",
    "depth_transform.conv_inv_transform.3.0.weight", "depth_transform.conv_inv_transform.3.0.bias")


def ddim_coefficients(alphas_cumprod: torch.Tensor, num_inference_steps: int, num_train_timesteps: int,
                      final_alpha_cumprod: float = 1.0) -> Tuple[list, list, list]:
    """Timesteps of `DDIMScheduler.set_timesteps` (reference scheduling_ddim.py:215-229) and the two scalars
    that `DDIMScheduler.step` (:285-326, eta=0, epsilon prediction, no clipping) reduces to:
        x_{t-1} = c_x * x_t + c_eps * eps,
        c_x = sqrt(a_prev / a_t),  c_eps = sqrt(1 - a_prev) - sqrt(a_prev * (1 - a_t) / a_t)
    evaluated in fp64 from the scheduler's fp32 `alphas_cumprod` table (SURVEY.md §3.3)."""
    ratio = num_train_timesteps // num_inference_steps
    ts = [int(round(i * ratio)) for i in range(num_inference_steps)][::-1]
    acp = alphas_cumprod.detach().to("cpu", torch.float64)
    cx, ce = [], []
    for t in ts:
        prev = t - ratio
        a_t = float(acp[t])
        a_p = float(acp[prev]) if prev >= 0 else float(final_alpha_cumprod)
        cx.append((a_p / a_t) ** 0.5)
        ce.append((1.0 - a_p) ** 0.5 - (a_p * (1.0 - a_t) / a_t) ** 0.5)
    return ts, cx, ce


class WorkspacePool:
    """One growing device buffer shared by several engines that never run concurrently (the engines of one head):
    a ragged last batch or a second image size then costs packed weights only, not another workspace (1.3 GB at C3)."""

    def __init__(self, device):
        self.device, self.buf = torch.device(device), None

    def get(self, nbytes: int) -> torch.Tensor:
        if self.buf is None or self.buf.numel() < nbytes:
            self.buf = None  # release before growing
            self.buf = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return self.buf


class DenoiseEngine:
    """One engine per (device, geometry).  `variant`: 'swin' (cond at half the latent resolution, bilinear
    upsample + convA/convB) or 'res' (cond at latent resolution)."""

    def __init__(self, variant: str, batch: int, latent_hw: Sequence[int], cond_hw: Sequence[int],
                 num_inference_steps: int, device: torch.device, cuda_graph: bool = True,
                 simt_conv: bool = False, check_range: bool = False, halo_conv: bool = True,
                 swap_narrow: bool = True, pair_wide: bool = True, step_decode: bool = False, workspace_pool=None,
                 fp8_corr: bool = True, stochastic: bool = False):
        self.lib = _cabi.load_library()
        device = torch.device(device)
        if device.type != "cuda":
            raise EngineError("DenoiseEngine runs on CUDA (sm_100a) only; there is no CPU path")
        self.device = device
        self.variant = variant
        self.batch, self.latent_hw, self.cond_hw = int(batch), tuple(latent_hw), tuple(cond_hw)
        self.steps = int(num_inference_steps)
        flags = (_cabi.FLAG_CUDA_GRAPH if cuda_graph else 0) | (_cabi.FLAG_SIMT_CONV if simt_conv else 0) | \
                (_cabi.FLAG_CHECK_RANGE if check_range else 0) | (_cabi.FLAG_HALO_CONV if halo_conv else 0) | \
                (_cabi.FLAG_SWAP_NARROW if swap_narrow else 0) | (_cabi.FLAG_PAIR_WIDE if pair_wide else 0) | \
                (_cabi.FLAG_STEP_DECODE if step_decode else 0) | (_cabi.FLAG_FP8_CORR if fp8_corr else 0) | \
                (_cabi.FLAG_STOCHASTIC if stochastic else 0)
        self.fp8_corr = bool(fp8_corr)
        self.stochastic = bool(stochastic)
        self.step_decode = bool(step_decode)
        cfg = _cabi.DDConfig(_cabi.ABI_VERSION, {"res": _cabi.VARIANT_RES, "swin": _cabi.VARIANT_SWIN}[variant],
                             self.batch, self.latent_hw[0], self.latent_hw[1], self.cond_hw[0], self.cond_hw[1],
                             self.steps, device.index if device.index is not None else torch.cuda.current_device(),
                             flags)
        h = C.c_void_p()
        _cabi.check(self.lib.dd_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self._ws: Optional[torch.Tensor] = None
        self._pool = workspace_pool  # optional WorkspacePool shared by the engines of one head (one buffer per device)
        self._keep = []  # fp32 contiguous copies handed to dd_set_weight must outlive finalize
        self.producers = None
        self.backbone = None

    # ---------------------------------------------------------------- setup
    def load_weights(self, tensors: Dict[str, torch.Tensor]):
        keys = DENOISER_KEYS + DECODER_KEYS + (FUSE_KEYS if self.variant == "swin" else ())
        if all(k in tensors for k in ENCODER_KEYS):
            keys = keys + ENCODER_KEYS
        if self.backbone is not None:
            keys = keys + tuple(k for k in tensors if k.startswith("backbone.") and tensors[k].is_floating_point())
        if self.producers is not None:
            keys = keys + tuple(k for k in tensors if k.startswith(("hahineck.", "conv_lateral.", "conv_up."))
                                and not k.endswith("num_batches_tracked") and tensors[k].dim() <= 4
                                and not k.startswith(("hahineck.multi_att", "hahineck.self_attn",
                                                      "hahineck.reference_points", "hahineck.level_embed")))
        self._keep = []
        for k in keys:
            if k not in tensors:
                raise EngineError(f"missing parameter {k}")
            t = tensors[k].detach().to(self.device, torch.float32).contiguous()
            self._keep.append(t)
            shape = (C.c_int64 * t.dim())(*t.shape)
            _cabi.check(self.lib.dd_set_weight(self._h, k.encode(), C.c_void_p(t.data_ptr()), shape, t.dim()))
        _cabi.check(self.lib.dd_finalize_weights(self._h, C.c_void_p(self._stream())))
        self._keep = []

    def enable_producers(self, channels, sizes, has_neck: bool):
        """Run the HAHI neck (if any) + FPN natively too; call before load_weights.  `sizes`: [(h, w)] per level."""
        pc = _cabi.DDProducerConfig()
        pc.num_levels = len(channels)
        for i, (c, (hh, ww)) in enumerate(zip(channels, sizes)):
            pc.channels[i], pc.heights[i], pc.widths[i] = int(c), int(hh), int(ww)
        pc.has_neck = 1 if has_neck else 0
        _cabi.check(self.lib.dd_enable_producers(self._h, C.byref(pc)))
        self.producers = (tuple(channels), tuple(tuple(s_) for s_ in sizes), bool(has_neck))
        self._ws = None

    def enable_backbone(self, image_hw, embed_dims=192, depths=(2, 2, 18, 2), num_heads=(6, 12, 24, 48), window=7,
                        kind="swin", mp_dims=(64, 128, 216, 288), mp_paths=(2, 3, 3, 3), mlp_ratio=4):
        """Run the backbone natively as well (after enable_producers, before load_weights).  kind: 'swin' (Swin-L),
        'resnet' (ResNetForMMBEV BasicBlock stages; only `depths` is used) or 'mpvit' (`depths` = encoder layers per
        stage, `mp_dims` / `mp_paths` / `mlp_ratio`)."""
        bc = _cabi.DDBackboneConfig()
        bc.kind, bc.embed_dims, bc.window = {"swin": 1, "resnet": 2, "mpvit": 3}[kind], int(embed_dims), int(window)
        bc.height, bc.width = int(image_hw[0]), int(image_hw[1])
        bc.mlp_ratio = int(mlp_ratio)
        for i in range(4):
            bc.depths[i], bc.num_heads[i] = int(depths[i]), int(num_heads[i])
            bc.mp_dims[i], bc.mp_paths[i] = int(mp_dims[i]), int(mp_paths[i])
        _cabi.check(self.lib.dd_enable_backbone(self._h, C.byref(bc)))
        self.backbone = (tuple(image_hw), int(embed_dims))
        self._ws = None

    def set_schedule(self, timesteps, c_x, c_eps, sigma=None):
        """`sigma`: per-step noise scale of stochastic DDIM (`DDIMScheduler.stochastic_coefficients`); None = 0."""
        n = len(timesteps)
        args = (self._h, (C.c_int64 * n)(*[int(t) for t in timesteps]), (C.c_double * n)(*c_x), (C.c_double * n)(*c_eps))
        if sigma is None:
            _cabi.check(self.lib.dd_set_schedule(*args, n))
        else:
            _cabi.check(self.lib.dd_set_schedule_eta(*args, (C.c_double * n)(*[float(v) for v in sigma]), n))

    # ---------------------------------------------------------------- calls
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _workspace(self) -> torch.Tensor:
        need = int(self.lib.dd_workspace_bytes(self._h))
        if self._pool is not None:
            return self._pool.get(need + 1024)
        if self._ws is None or self._ws.numel() < need + 1024:
            self._ws = torch.empty(need + 1024, dtype=torch.uint8, device=self.device)
        return self._ws

    @staticmethod
    def _aligned(ws: torch.Tensor) -> int:
        return (ws.data_ptr() + 1023) // 1024 * 1024

    def _check_in(self, t: torch.Tensor, shape):
        if t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
            raise EngineError(f"expected contiguous fp32 {tuple(shape)} on {self.device}, got {tuple(t.shape)} "
                              f"{t.dtype} {t.device}")

    def run_backbone(self, rgb: torch.Tensor, want_feats=False):
        """rgb [B,3,H,W] -> the four Swin stage outputs, left inside the workspace for `build_condition(None)`;
        `want_feats` also returns them as fp32 NCHW tensors."""
        if self.backbone is None:
            raise EngineError("enable_backbone() was not called")
        self._check_in(rgb, (self.batch, 3, *self.backbone[0]))
        chans, sizes, _ = self.producers
        feats = [torch.empty(self.batch, c, *hw, device=self.device) for c, hw in zip(chans, sizes)] if want_feats else None
        ptrs = (C.c_void_p * 4)(*[f.data_ptr() for f in feats]) if want_feats else None
        ws = self._workspace()
        _cabi.check(self.lib.dd_run_backbone(self._h, C.c_void_p(rgb.data_ptr()), ptrs, C.c_void_p(self._aligned(ws)),
                                             ws.numel() - 1024, C.c_void_p(self._stream())))
        return feats

    def build_condition(self, feats, want_cond=False):
        """Backbone feature maps (fp32 NCHW, finest first) -> condition map, natively (neck + FPN).  The result
        stays inside the workspace for the next `denoise_decode(None, noise)`; `want_cond` also returns it."""
        if self.producers is None:
            raise EngineError("enable_producers() was not called")
        chans, sizes, _ = self.producers
        ptrs = None
        if feats is not None:
            for f, c, hw in zip(feats, chans, sizes):
                self._check_in(f, (self.batch, c, *hw))
            ptrs = (C.c_void_p * 4)(*([f.data_ptr() for f in feats] + [0] * (4 - len(feats))))
        cond = torch.empty(self.batch, 256, *self.cond_hw, device=self.device) if want_cond else None
        ws = self._workspace()
        _cabi.check(self.lib.dd_build_condition(self._h, ptrs, C.c_void_p(cond.data_ptr() if want_cond else 0),
                                                C.c_void_p(self._aligned(ws)), ws.numel() - 1024,
                                                C.c_void_p(self._stream())))
        return cond

    def denoise_decode(self, cond: Optional[torch.Tensor], noise: torch.Tensor, want_latent=False, want_logits=False):
        """cond [B,256,hc,wc] (or None right after build_condition), noise [B,16,h,w] -> depth [B,1,2h,2w]
        (+ latent [B,16,h,w], logits)."""
        B, (h, w) = self.batch, self.latent_hw
        if cond is not None:
            self._check_in(cond, (B, 256, *self.cond_hw))
        self._check_in(noise, (B, 16, h, w))
        depth = torch.empty(B, 1, 2 * h, 2 * w, device=self.device, dtype=torch.float32)
        latent = torch.empty(B, 16, h, w, device=self.device, dtype=torch.float32) if want_latent else None
        logits = torch.empty_like(depth) if want_logits else None
        ws = self._workspace()
        _cabi.check(self.lib.dd_denoise_decode(
            self._h, C.c_void_p(cond.data_ptr() if cond is not None else 0), C.c_void_p(noise.data_ptr()),
            C.c_void_p(latent.data_ptr() if want_latent else 0), C.c_void_p(logits.data_ptr() if want_logits else 0),
            C.c_void_p(depth.data_ptr()), C.c_void_p(self._aligned(ws)), ws.numel() - 1024, C.c_void_p(self._stream())))
        return depth, latent, logits

    def denoise_decode_steps(self, cond: Optional[torch.Tensor], noise: torch.Tensor, want_latent=False,
                             want_logits=False):
        """As `denoise_decode`, additionally decoding the latent after every step inside the captured graph (the *Vis
        heads' `pred_inter`): returns (depth_steps [T,B,1,2h,2w], latent, logits of the final step)."""
        if not self.step_decode:
            raise EngineError("engine was created without step_decode=True")
        B, (h, w) = self.batch, self.latent_hw
        if cond is not None:
            self._check_in(cond, (B, 256, *self.cond_hw))
        self._check_in(noise, (B, 16, h, w))
        steps = torch.empty(self.steps, B, 1, 2 * h, 2 * w, device=self.device, dtype=torch.float32)
        latent = torch.empty(B, 16, h, w, device=self.device, dtype=torch.float32) if want_latent else None
        logits = torch.empty(B, 1, 2 * h, 2 * w, device=self.device, dtype=torch.float32) if want_logits else None
        ws = self._workspace()
        _cabi.check(self.lib.dd_denoise_decode_steps(
            self._h, C.c_void_p(cond.data_ptr() if cond is not None else 0), C.c_void_p(noise.data_ptr()),
            C.c_void_p(latent.data_ptr() if want_latent else 0), C.c_void_p(logits.data_ptr() if want_logits else 0),
            C.c_void_p(steps.data_ptr()), C.c_void_p(self._aligned(ws)), ws.numel() - 1024, C.c_void_p(self._stream())))
        return steps, latent, logits

    def denoise_decode_stochastic(self, cond: Optional[torch.Tensor], noise: torch.Tensor, step_noise: torch.Tensor,
                                  want_latent=False, want_latent_steps=False, want_logits=False, want_depth_steps=False):
        """Stochastic DDIM (engine created with stochastic=True): as `denoise_decode`, each step adding sigma_t * z_t with
        z_t = step_noise[t] ([T,B,16,h,w]).  Returns (depth [B,1,2h,2w], latent, latent_steps [T,B,16,h,w], logits,
        depth_steps [T,B,1,2h,2w]); the optional ones are None unless asked for (depth_steps needs step_decode=True)."""
        if not self.stochastic:
            raise EngineError("engine was created without stochastic=True")
        if want_depth_steps and not self.step_decode:
            raise EngineError("engine was created without step_decode=True")
        B, (h, w), T = self.batch, self.latent_hw, self.steps
        if cond is not None:
            self._check_in(cond, (B, 256, *self.cond_hw))
        self._check_in(noise, (B, 16, h, w))
        self._check_in(step_noise, (T, B, 16, h, w))
        f32 = dict(device=self.device, dtype=torch.float32)
        depth = torch.empty(B, 1, 2 * h, 2 * w, **f32)
        latent = torch.empty(B, 16, h, w, **f32) if want_latent else None
        lsteps = torch.empty(T, B, 16, h, w, **f32) if want_latent_steps else None
        logits = torch.empty_like(depth) if want_logits else None
        dsteps = torch.empty(T, B, 1, 2 * h, 2 * w, **f32) if want_depth_steps else None
        ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)  # noqa: E731
        ws = self._workspace()
        _cabi.check(self.lib.dd_denoise_decode_stochastic(
            self._h, ptr(cond), ptr(noise), ptr(step_noise), ptr(latent), ptr(lsteps), ptr(logits), ptr(depth),
            ptr(dsteps), C.c_void_p(self._aligned(ws)), ws.numel() - 1024, C.c_void_p(self._stream())))
        return depth, latent, lsteps, logits, dsteps

    def denoiser_forward(self, cond: torch.Tensor, noisy: torch.Tensor, t) -> torch.Tensor:
        """eps = ScheduledCNNRefine(noisy, t, cond); t: int or per-image sequence."""
        B, (h, w) = self.batch, self.latent_hw
        self._check_in(cond, (B, 256, *self.cond_hw))
        self._check_in(noisy, (B, 16, h, w))
        ts = [int(t)] * B if not hasattr(t, "__len__") else [int(v) for v in t]
        if len(ts) == 1:
            ts = ts * B
        eps = torch.empty_like(noisy)
        ws = self._workspace()
        _cabi.check(self.lib.dd_denoiser_forward(
            self._h, C.c_void_p(cond.data_ptr()), C.c_void_p(noisy.data_ptr()), (C.c_int64 * B)(*ts),
            C.c_void_p(eps.data_ptr()), C.c_void_p(self._aligned(ws)), ws.numel() - 1024, C.c_void_p(self._stream())))
        return eps

    def encode(self, depth: torch.Tensor) -> torch.Tensor:
        """latent = depth_transform.t(depth): [B,1,H,W] -> [B,16,ceil(H/2),ceil(W/2)]."""
        B, (h, w) = self.batch, self.latent_hw
        H, W = depth.shape[-2:]
        self._check_in(depth, (B, 1, H, W))
        out = torch.empty(B, 16, h, w, device=self.device, dtype=torch.float32)
        _cabi.check(self.lib.dd_encode(self._h, C.c_void_p(depth.data_ptr()), H, W, C.c_void_p(out.data_ptr()),
                                       C.c_void_p(self._stream())))
        return out

    def decode(self, latent: torch.Tensor, want_logits=False):
        B, (h, w) = self.batch, self.latent_hw
        self._check_in(latent, (B, 16, h, w))
        depth = torch.empty(B, 1, 2 * h, 2 * w, device=self.device, dtype=torch.float32)
        logits = torch.empty_like(depth) if want_logits else None
        ws = self._workspace()
        _cabi.check(self.lib.dd_decode(self._h, C.c_void_p(latent.data_ptr()),
                                       C.c_void_p(logits.data_ptr() if want_logits else 0), C.c_void_p(depth.data_ptr()),
                                       C.c_void_p(self._aligned(ws)), ws.numel() - 1024, C.c_void_p(self._stream())))
        return depth, logits

    def conv3x3(self, x: torch.Tensor, w: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
        """Single 3x3/s1/p1 conv + bias on the engine's convolution path (parity tests, roofline)."""
        B, cin, H, W = x.shape
        cout = w.shape[0]
        x, w, b = (t.detach().to(self.device, torch.float32).contiguous() for t in (x, w, b))
        y = torch.empty(B, cout, H, W, device=self.device, dtype=torch.float32)
        need = int(self.lib.dd_conv3x3_workspace_bytes(B, cin, cout, H, W))
        ws = torch.empty(need + 1024, dtype=torch.uint8, device=self.device)
        _cabi.check(self.lib.dd_conv3x3(self._h, C.c_void_p(x.data_ptr()), C.c_void_p(w.data_ptr()),
                                        C.c_void_p(b.data_ptr()), C.c_void_p(y.data_ptr()), B, cin, cout, H, W,
                                        C.c_void_p(self._aligned(ws)), need, C.c_void_p(self._stream())))
        return y

    def bench_conv(self, cin: int, cout: int, iters: int = 20) -> float:
        """Average milliseconds per launch of the (cin -> cout) conv on this engine's latent grid."""
        ms = C.c_float()
        ws = self._workspace()
        _cabi.check(self.lib.dd_bench_conv(self._h, cin, cout, iters, C.byref(ms), C.c_void_p(self._aligned(ws)),
                                           ws.numel() - 1024, C.c_void_p(self._stream())))
        return float(ms.value)

    def bench_gemm(self, M: int, K: int, N: int, mode: int = 0, iters: int = 20) -> float:
        ms = C.c_float()
        _cabi.check(self.lib.dd_bench_gemm(self._h, M, K, N, mode, iters, C.byref(ms)))
        return float(ms.value)

    def poll_status(self) -> None:
        """Synchronise the current stream; raises EngineError(DD_ERR_RANGE) if the fp16 split overflowed."""
        _cabi.check(self.lib.dd_poll_status(self._h, C.c_void_p(self._stream())))

    @property
    def last_launch_count(self) -> int:
        return int(self.lib.dd_last_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.dd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # pragma: no cover
            pass
