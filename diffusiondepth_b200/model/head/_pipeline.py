"""`CNNDDIMPipiline` — the heads' DDIM sampler entry point, `head.pipeline(...)` (reference
src/model/head/ddim_depth_estimate_res_swin_addHAHI.py:243-303; the *Vis variant, ..._swin_addHAHI_vis.py:255-303, also
returns `image_list`, the latent after every step).  Same signature and return shapes as the reference; the loop runs on
the head's CUDA engine: eta = 0 on the deterministic loop, eta > 0 on the stochastic one (dd_denoise_decode_stochastic),
with the noise drawn in the reference's order (x_T, then one draw per step) on the caller's generator.

Deliberate difference: the reference reads `self.device`, which its pipeline does not have, so any `generator` raises
AttributeError there.  Here a generator whose device type matches `device` drives every draw, and one on another device
type raises ValueError."""
from typing import Dict, Optional, Tuple, Union

import torch

from diffusiondepth_b200._cabi import EngineError


def draw_pipeline_noise(num_steps: int, shape, device, dtype=torch.float32, generator=None, stochastic=True):
    """x_T and the per-step noise in the reference pipeline's draw order: one `torch.randn(shape)` for x_T, then (eta > 0)
    one inside every `DDIMScheduler.step`, the last step included.  The T step draws go into the slices of one
    [T, *shape] buffer, each its own `randn` call (one draw of the whole buffer would be a different stream)."""
    x_T = torch.randn(shape, generator=generator, device=device, dtype=dtype)
    return x_T, (draw_step_noise(num_steps, shape, device, dtype, generator) if stochastic else None)


def draw_step_noise(num_steps: int, shape, device, dtype=torch.float32, generator=None):
    """[T, *shape]: T separate `torch.randn(shape)` draws, written into the slices of one buffer."""
    steps = torch.empty((num_steps, *shape), device=device, dtype=dtype)
    for i in range(num_steps):
        torch.randn(shape, generator=generator, dtype=dtype, out=steps[i])
    return steps


class CNNDDIMPipiline:
    """Bound to a head's denoiser (`model`) and scheduler like the reference's; `model` bridges to the head's engines."""

    def __init__(self, model, scheduler, with_image_list=False):
        self.model = model
        self.scheduler = scheduler
        self.with_image_list = with_image_list

    def __call__(
            self,
            batch_size,
            device,
            dtype,
            shape,
            input_args,
            generator: Optional[torch.Generator] = None,
            eta: float = 0.0,
            num_inference_steps: int = 50,
            return_dict: bool = True,
            **kwargs,
    ) -> Union[Dict, Tuple]:
        device = torch.device(device)
        if generator is not None and generator.device.type != device.type:
            raise ValueError(f"the generator is on {generator.device} but the pipeline samples on {device}: "
                             f"use torch.Generator(device='{device.type}')")
        head = self.model._bridge() if self.model._bridge is not None else None
        if head is None:
            raise EngineError("CNNDDIMPipiline is not attached to a DDIM head / CUDA engine")
        eta = float(eta)
        T = int(num_inference_steps)
        self.scheduler.stochastic_coefficients(T, eta)  # validates eta (ValueError), sets the scheduler's timesteps
        cond = input_args[0]
        if device.type != "cuda" or not torch.is_tensor(cond) or not cond.is_cuda:
            raise EngineError("the DDIM pipeline runs on the CUDA engine (sm_100a) only; there is no CPU path")
        image_shape = (int(batch_size), *[int(s) for s in shape])
        x_T, step_noise = draw_pipeline_noise(T, image_shape, device, dtype, generator, stochastic=eta > 0)
        image, image_list = head.sample_latents(cond.contiguous().float(), x_T.float(), step_noise, eta, T,
                                                self.with_image_list)
        image = image.to(dtype)
        if self.with_image_list:
            image_list = [im.to(dtype) for im in image_list.unbind(0)]
            return (image, image_list) if not return_dict else {'images': image, 'image_list': image_list}
        return (image,) if not return_dict else {'images': image}
