"""ORACLE (test infrastructure only).  The img2img additions of [3P] diffusers==0.30.0 `StableDiffusionXLImg2ImgPipeline`
on top of the text-to-image restatement in oracle/scheduler_ref.py: `get_timesteps(strength)`, the initial latents
(`prepare_latents`: posterior sample, `scaling_factor`, batch expansion, `EulerDiscreteScheduler.add_noise` at the
scheduler's begin index) and the denoise loop over the truncated timestep list."""
from __future__ import annotations

from typing import Callable, List, Optional, Tuple, Union

import torch

from .scheduler_ref import euler_tables, rescale_noise_cfg
from .vae_encoder_ref import posterior_sample_ref


def get_timesteps(num_inference_steps: int, strength: float) -> Tuple[int, int]:
    """-> (t_start, executed steps): init_timestep = min(int(T * strength), T), t_start = max(T - init_timestep, 0)."""
    init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
    t_start = max(num_inference_steps - init_timestep, 0)
    return t_start, num_inference_steps - t_start


def add_noise_ref(latents16: torch.Tensor, noise16: torch.Tensor, sigma: float) -> torch.Tensor:
    """EulerDiscreteScheduler.add_noise on fp16 tensors: sigma cast to fp16, noise * sigma and the sum rounded in fp16."""
    s = torch.tensor([sigma], dtype=torch.float32).to(device=latents16.device, dtype=torch.float16).reshape(1, 1, 1, 1)
    return latents16 + noise16 * s


def init_latents_ref(moments: torch.Tensor, batch: int, generator: Union[torch.Generator, List[torch.Generator], None],
                     scaling_factor: float, sigma: float) -> torch.Tensor:
    """img2img initial latents from the moments of the source image(s) [Bi, 2 L, h, w].  Draw order: the posterior eps
    (fp32, shape of the mean: one draw for all images from a single generator, one [1, L, h, w] draw per batch slot from a
    list, the images replicated to the batch), then the noise (fp16, likewise)."""
    Bi, L2, h, w = moments.shape
    L = L2 // 2

    def randn(shape, g, dtype):
        dev = g.device if g is not None else "cpu"
        return torch.randn(shape, generator=g, device=dev, dtype=dtype).to(moments.device)

    if isinstance(generator, list):
        if len(generator) != batch or batch % Bi:
            raise ValueError("a generator list needs one generator per image of a batch that is a multiple of the images")
        m = torch.cat([moments] * (batch // Bi), dim=0)
        sample = torch.cat([posterior_sample_ref(m[i:i + 1], randn((1, L, h, w), g, torch.float32))
                            for i, g in enumerate(generator)], dim=0)
    else:
        sample = posterior_sample_ref(moments, randn((Bi, L, h, w), generator, torch.float32))
    z = scaling_factor * sample.to(torch.float16)
    if batch > z.shape[0]:
        if batch % z.shape[0]:
            raise ValueError("batch is not a multiple of the number of images")
        z = torch.cat([z] * (batch // z.shape[0]), dim=0)
    if isinstance(generator, list):
        noise = torch.cat([randn((1, L, h, w), g, torch.float16) for g in generator], dim=0)
    else:
        noise = randn((batch, L, h, w), generator, torch.float16)
    return add_noise_ref(z, noise, sigma)


@torch.no_grad()
def img2img_denoise_loop(unet_fn: Callable, latents: torch.Tensor, prompt_embeds: torch.Tensor,
                         neg_prompt_embeds: torch.Tensor, pooled: torch.Tensor, neg_pooled: torch.Tensor,
                         time_ids: torch.Tensor, num_inference_steps: int, strength: float, guidance_scale: float = 5.0,
                         set_scale: Optional[Callable[[float], None]] = None, conditioning_scale: float = 1.0,
                         control_guidance_start: float = 0.0, control_guidance_end: float = 1.0,
                         guidance_rescale: float = 0.0, denoising_end: Optional[float] = None,
                         callback: Optional[Callable] = None, callback_steps: int = 1) -> torch.Tensor:
    """scheduler_ref.denoise_loop over timesteps[t_start:] (cut by `denoising_end`), sigma index t_start + i.  The
    gating fractions and the callback index count the executed steps from 0 (`enumerate(timesteps)`)."""
    timesteps, sigmas, _ = euler_tables(num_inference_steps)
    t_start, _ = get_timesteps(num_inference_steps, strength)
    ks = list(range(t_start, num_inference_steps))
    if denoising_end is not None and isinstance(denoising_end, float) and 0 < denoising_end < 1:
        cutoff = int(round(1000 - denoising_end * 1000))
        ks = [k for k in ks if timesteps[k] >= cutoff]
    cfg = guidance_scale > 1.0
    if cfg:
        ehs = torch.cat([neg_prompt_embeds, prompt_embeds], dim=0)
        text_embeds = torch.cat([neg_pooled, pooled], dim=0)
        tids = torch.cat([time_ids, time_ids], dim=0)
    else:
        ehs, text_embeds, tids = prompt_embeds, pooled, time_ids
    n = len(ks)
    for i, k in enumerate(ks):
        if set_scale is not None:
            off = (i / n < control_guidance_start) or ((i + 1) / n > control_guidance_end)
            set_scale(0.0 if off else conditioning_scale)
        sigma, sigma_next = float(sigmas[k]), float(sigmas[k + 1])
        x2 = torch.cat([latents] * 2) if cfg else latents
        x2 = (x2 / ((sigma ** 2 + 1) ** 0.5)).to(latents.dtype)
        noise = unet_fn(x2, float(timesteps[k]), ehs, text_embeds, tids)
        if cfg:
            u, c = noise.chunk(2)
            eps = u + guidance_scale * (c - u)
            if guidance_rescale > 0.0:
                eps = rescale_noise_cfg(eps, c, guidance_rescale)
        else:
            eps = noise
        x = latents.float()
        x0 = x - (sigma * eps.float()).to(eps.dtype).float()
        deriv = (x - x0) / sigma
        latents = (x + deriv * (sigma_next - sigma)).to(eps.dtype)
        if callback is not None and i % callback_steps == 0:
            callback(i, float(timesteps[k]), latents)
    return latents
