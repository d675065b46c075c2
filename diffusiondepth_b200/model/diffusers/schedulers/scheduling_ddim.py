"""DDIM sampler with the public surface of the reference's scheduler
(reference src/model/diffusers/schedulers/scheduling_ddim.py:100-376): ctor tables, `set_timesteps`,
`step`, `add_noise`, `.config`.  Added for the engine: `fused_coefficients()` — the per-step scalars the
CUDA loop consumes (x_{t-1} = c_x x_t + c_eps eps; SURVEY.md §3.3)."""
import math
from types import SimpleNamespace

import numpy as np
import torch


class DDIMScheduler:
    order = 1
    config_name = "scheduler_config.json"

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 trained_betas=None, clip_sample=False, set_alpha_to_one=True, steps_offset=0,
                 prediction_type="epsilon", **kwargs):
        self._cfg = dict(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                         beta_schedule=beta_schedule, trained_betas=trained_betas, clip_sample=clip_sample,
                         set_alpha_to_one=set_alpha_to_one, steps_offset=steps_offset,
                         prediction_type=prediction_type)
        for k, v in self._cfg.items():  # the reference exposes every ctor argument as an attribute too
            setattr(self, k, v)
        if trained_betas is not None:
            betas = torch.tensor(trained_betas, dtype=torch.float32)
        elif beta_schedule == "linear":
            betas = torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
        elif beta_schedule == "scaled_linear":
            betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
        elif beta_schedule == "squaredcos_cap_v2":
            bar = lambda s: math.cos((s + 0.008) / 1.008 * math.pi / 2) ** 2  # noqa: E731
            n = num_train_timesteps
            betas = torch.tensor([min(1 - bar((i + 1) / n) / bar(i / n), 0.999) for i in range(n)],
                                 dtype=torch.float32)
        else:
            raise NotImplementedError(f"{beta_schedule} is not implemented for {type(self).__name__}")
        self.betas = betas
        self.alphas = 1.0 - betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(np.arange(num_train_timesteps)[::-1].copy().astype(np.int64))

    @property
    def config(self):
        return SimpleNamespace(**self._cfg)

    def scale_model_input(self, sample, timestep=None):
        return sample

    # -- schedule -----------------------------------------------------------------------------------------
    def set_timesteps(self, num_inference_steps, device=None):
        self.num_inference_steps = int(num_inference_steps)
        stride = self._cfg["num_train_timesteps"] // self.num_inference_steps
        ts = (np.arange(self.num_inference_steps) * stride).round()[::-1].copy().astype(np.int64)
        self.timesteps = torch.from_numpy(ts).to(device) + self._cfg["steps_offset"]

    def _alpha_pair(self, timestep, prev_timestep):
        a_t = self.alphas_cumprod[timestep]
        a_prev = self.alphas_cumprod[prev_timestep] if prev_timestep >= 0 else self.final_alpha_cumprod
        return a_t, a_prev

    def _get_variance(self, timestep, prev_timestep):
        a_t, a_prev = self._alpha_pair(timestep, prev_timestep)
        return ((1 - a_prev) / (1 - a_t)) * (1 - a_t / a_prev)

    def fused_coefficients(self, num_inference_steps=None):
        """(timesteps, c_x, c_eps) for eta = 0 / epsilon prediction / no clipping, fp64 from the fp32 table."""
        if num_inference_steps is not None:
            self.set_timesteps(num_inference_steps)
        if self._cfg["prediction_type"] != "epsilon" or self._cfg["clip_sample"]:
            raise NotImplementedError("the fused CUDA loop covers the reference configuration only "
                                      "(prediction_type='epsilon', clip_sample=False)")
        stride = self._cfg["num_train_timesteps"] // self.num_inference_steps
        acp = self.alphas_cumprod.to("cpu", torch.float64)
        ts, cx, ce = [int(t) for t in self.timesteps.tolist()], [], []
        for t in ts:
            a_t = float(acp[t])
            a_p = float(acp[t - stride]) if t - stride >= 0 else float(self.final_alpha_cumprod)
            cx.append(math.sqrt(a_p / a_t))
            ce.append(math.sqrt(1.0 - a_p) - math.sqrt(a_p * (1.0 - a_t) / a_t))
        return ts, cx, ce

    def stochastic_coefficients(self, num_inference_steps=None, eta=0.0):
        """(timesteps, c_x, c_eps, sigma) of the step with `eta` >= 0 (reference scheduling_ddim.py:313-350,
        formula (16) of the DDIM paper), fp64 from the fp32 table:
            x_{t-1} = c_x x_t + c_eps eps + sigma z,   sigma = eta sqrt((1 - a_p) / (1 - a_t) (1 - a_t / a_p)),
            c_x = sqrt(a_p / a_t),   c_eps = sqrt(1 - a_p - sigma^2) - sqrt(a_p (1 - a_t) / a_t).
        eta = 0 returns exactly `fused_coefficients` and sigma = 0.  Unlike the reference, which yields NaN there, an
        eta with 1 - a_p - sigma^2 < 0 on some step (possible only for eta > 1) raises ValueError, as does eta < 0."""
        eta = float(eta)
        if not eta >= 0.0:
            raise ValueError(f"eta must be >= 0, got {eta}")
        ts, cx, ce = self.fused_coefficients(num_inference_steps)
        if eta == 0.0:
            return ts, cx, ce, [0.0] * len(ts)
        stride = self._cfg["num_train_timesteps"] // self.num_inference_steps
        acp = self.alphas_cumprod.to("cpu", torch.float64)
        ce, sg = [], []
        for t in ts:
            a_t = float(acp[t])
            a_p = float(acp[t - stride]) if t - stride >= 0 else float(self.final_alpha_cumprod)
            s = eta * math.sqrt((1.0 - a_p) / (1.0 - a_t) * (1.0 - a_t / a_p))
            dir2 = 1.0 - a_p - s * s
            if dir2 < 0.0:
                raise ValueError(f"eta = {eta} makes 1 - alpha_prev - sigma^2 negative at timestep {t}")
            ce.append(math.sqrt(dir2) - math.sqrt(a_p * (1.0 - a_t) / a_t))
            sg.append(s)
        return ts, cx, ce, sg

    # -- one reverse step (torch; API parity with the reference, not on the CUDA hot path) -----------------
    def step(self, model_output, timestep, sample, eta=0.0, use_clipped_model_output=False, generator=None,
             variance_noise=None, return_dict=True):
        if self.num_inference_steps is None:
            raise ValueError("Number of inference steps is 'None', you need to run 'set_timesteps' first")
        prev_timestep = timestep - self._cfg["num_train_timesteps"] // self.num_inference_steps
        a_t, a_prev = self._alpha_pair(timestep, prev_timestep)
        b_t = 1 - a_t
        kind = self._cfg["prediction_type"]
        if kind == "epsilon":
            x0 = (sample - b_t ** 0.5 * model_output) / a_t ** 0.5
        elif kind == "sample":
            x0 = model_output
        elif kind == "v_prediction":
            x0 = a_t ** 0.5 * sample - b_t ** 0.5 * model_output
            model_output = a_t ** 0.5 * model_output + b_t ** 0.5 * sample
        else:
            raise ValueError(f"prediction_type {kind!r} must be one of epsilon, sample, v_prediction")
        if self._cfg["clip_sample"]:
            x0 = x0.clamp(-1, 1)
        sigma = eta * self._get_variance(timestep, prev_timestep) ** 0.5
        if use_clipped_model_output:
            model_output = (sample - a_t ** 0.5 * x0) / b_t ** 0.5
        prev_sample = a_prev ** 0.5 * x0 + (1 - a_prev - sigma ** 2) ** 0.5 * model_output
        if eta > 0:
            if variance_noise is not None and generator is not None:
                raise ValueError("Cannot pass both generator and variance_noise")
            if variance_noise is None:
                variance_noise = torch.randn(model_output.shape, generator=generator, device=model_output.device,
                                             dtype=model_output.dtype)
            prev_sample = prev_sample + sigma * variance_noise
        if not return_dict:
            return (prev_sample,)
        return dict(prev_sample=prev_sample, pred_original_sample=x0)

    def add_noise(self, original_samples, noise, timesteps):
        acp = self.alphas_cumprod.to(device=original_samples.device, dtype=original_samples.dtype)
        self.alphas_cumprod = acp
        a = acp[timesteps.to(original_samples.device)].flatten()
        shape = (-1,) + (1,) * (original_samples.dim() - 1)
        return (a ** 0.5).view(shape) * original_samples + ((1 - a) ** 0.5).view(shape) * noise

    def __len__(self):
        return self._cfg["num_train_timesteps"]
