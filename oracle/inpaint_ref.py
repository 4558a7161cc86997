"""ORACLE (test infrastructure only).  The inpainting additions of [3P] diffusers==0.30.0
`StableDiffusionXLInpaintPipeline` with a 4-channel (SDXL-base) UNet, on top of the img2img restatement in
oracle/img2img_ref.py.  diffusers is not installed here; these are the rules it follows:

- Size: `height` / `width` default to unet.config.sample_size * 8 (1024 for SDXL), not to the image size, and must be
  multiples of 8.  A PIL source image is converted to RGB and Lanczos-resized to (width, height) when its size differs.
- Mask: a PIL mask (or a list of them) is converted to "L", Lanczos-resized to (width, height), divided by 255 in fp32
  and binarized at 0.5 (v >= 128 for uint8 pixels).  A float tensor mask [H, W], [B, H, W] or [B, 1, H, W] in [0, 1]
  must already be (height, width) and is binarized at 0.5.  The latent mask is F.interpolate(mask, size=(h, w)) in its
  default nearest mode: latent (y, x) takes pixel (8y, 8x).  It is binary and fp16.  Batch slot b uses mask b % Bm.
- Schedule: img2img's get_timesteps(T, strength); `strength` defaults to 0.9999.
- Start latents: z0 = fp16(scaling_factor * fp16(posterior sample)) per source image, repeated to the batch.  A single
  generator draws eps (fp32, [n_img, 4, h, w]) and then the noise (fp16, [batch, 4, h, w]).  A generator list (one per
  batch slot) draws the eps of source image i from generator[i] for i < n_img only -- the images are not replicated
  before encoding, unlike img2img -- and then one noise per batch slot from generator[b].
  strength < 1: latents = add_noise(z0, noise, sigma[t_start]).  strength == 1: latents = fp16(noise * init_noise_sigma)
  (pure noise; z0 is still encoded for the blend).
- Per-step blend, after the Euler update of the executed step with absolute schedule index k:
  proper = fp16(z0 + fp16(noise * fp16(sigma[k + 1]))) except on the last executed step (also the last one under
  `denoising_end`, where sigma[k + 1] != 0), where proper = z0 without noise;
  latents = (1 - m) * proper + m * latents in the latents' dtype (fp16: rounded after each op).
  The next model input and the callback see the blended latents.
- Everything else is img2img: CFG on / off, guidance_rescale, denoising_end, gating and callback indices counted over the
  executed steps from 0, time ids defaulting to (height, width).  No pixel-space overlay after decode (diffusers applies
  one only with `padding_mask_crop`)."""
from __future__ import annotations

from typing import Callable, List, Optional, Tuple, Union

import numpy as np
import torch
import torch.nn.functional as F

from .img2img_ref import add_noise_ref, get_timesteps, img2img_denoise_loop
from .scheduler_ref import denoising_end_steps, euler_tables
from .vae_encoder_ref import posterior_sample_ref


def mask_ref(mask_image, height: int, width: int) -> torch.Tensor:
    """PIL mask(s) or a float tensor -> binarized fp32 pixel mask [Bm, 1, height, width]."""
    from PIL import Image
    if isinstance(mask_image, torch.Tensor):
        m = mask_image.float()
        m = m.reshape(1, 1, *m.shape) if m.dim() == 2 else (m.unsqueeze(1) if m.dim() == 3 else m)
        if tuple(m.shape[2:]) != (height, width):
            raise ValueError("tensor mask must be (height, width)")
    else:
        ims = [mask_image] if isinstance(mask_image, Image.Image) else list(mask_image)
        arrs = []
        for im in ims:
            im = im.convert("L")
            if im.size != (width, height):
                im = im.resize((width, height), resample=Image.LANCZOS)
            arrs.append(np.asarray(im, dtype=np.float32) / np.float32(255.0))
        m = torch.from_numpy(np.stack(arrs))[:, None]
    return (m >= 0.5).float()


def latent_mask_ref(mask: torch.Tensor, h: int, w: int) -> torch.Tensor:
    """prepare_mask_latents: nearest interpolation of the binarized pixel mask to the latent size, fp16."""
    return F.interpolate(mask, size=(h, w)).to(torch.float16)


def init_latents_ref(moments: torch.Tensor, batch: int, generator: Union[torch.Generator, List[torch.Generator], None],
                     scaling_factor: float, sigma: float, is_strength_max: bool = False,
                     init_noise_sigma: float = 1.0) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """-> (start latents, z0, noise), all fp16 [batch, L, h, w], from the moments of the source images
    [n_img, 2 L, h, w], in the draw order of the module docstring."""
    n_img, L2, h, w = moments.shape
    L = L2 // 2

    def randn(shape, g, dtype):
        dev = g.device if g is not None else "cpu"
        return torch.randn(shape, generator=g, device=dev, dtype=dtype).to(moments.device)

    if batch % n_img:
        raise ValueError("batch is not a multiple of the number of images")
    if isinstance(generator, list):
        if len(generator) != batch:
            raise ValueError("a generator list needs one generator per batch slot")
        sample = torch.cat([posterior_sample_ref(moments[i:i + 1], randn((1, L, h, w), generator[i], torch.float32))
                            for i in range(n_img)], dim=0)
    else:
        sample = posterior_sample_ref(moments, randn((n_img, L, h, w), generator, torch.float32))
    z0 = (scaling_factor * sample.to(torch.float16)).repeat(batch // n_img, 1, 1, 1)
    if isinstance(generator, list):
        noise = torch.cat([randn((1, L, h, w), g, torch.float16) for g in generator], dim=0)
    else:
        noise = randn((batch, L, h, w), generator, torch.float16)
    if is_strength_max:
        latents = (noise.float() * torch.tensor(init_noise_sigma, dtype=torch.float32)).to(torch.float16)
    else:
        latents = add_noise_ref(z0, noise, sigma)
    return latents, z0, noise


def blend_ref(latents: torch.Tensor, mask: torch.Tensor, z0: torch.Tensor, noise: torch.Tensor, sigma_next: float,
              last: bool) -> torch.Tensor:
    """(1 - m) * proper + m * latents in the latents' dtype; mask [Bm, 1, h, w], batch slot b uses mask b % Bm."""
    dt = latents.dtype
    m = mask.to(device=latents.device, dtype=dt).repeat(latents.shape[0] // mask.shape[0], 1, 1, 1)
    z = z0.to(device=latents.device, dtype=dt)
    proper = z if last else add_noise_ref(z, noise.to(device=latents.device, dtype=dt), sigma_next)
    return (1 - m) * proper + m * latents


@torch.no_grad()
def inpaint_denoise_loop(unet_fn: Callable, latents: torch.Tensor, prompt_embeds: torch.Tensor,
                         neg_prompt_embeds: torch.Tensor, pooled: torch.Tensor, neg_pooled: torch.Tensor,
                         time_ids: torch.Tensor, num_inference_steps: int, strength: float, mask: torch.Tensor,
                         z0: torch.Tensor, noise: torch.Tensor, denoising_end: Optional[float] = None,
                         callback: Optional[Callable] = None, callback_steps: int = 1, **img2img_opts) -> torch.Tensor:
    """img2img_denoise_loop plus the blend.  img2img_denoise_loop hands its callback the latents it continues from,
    so the blend is applied there, in place, after every step; `callback` then sees the blended latents.
    `mask` is the fp16 latent mask [Bm, 1, h, w]; `img2img_opts` are img2img_denoise_loop's loop options."""
    _, sigmas, _ = euler_tables(num_inference_steps)
    t_start, _ = get_timesteps(num_inference_steps, strength)
    n_exec = denoising_end_steps(num_inference_steps, denoising_end) - t_start

    def blend(i, t, x):
        x.copy_(blend_ref(x, mask, z0, noise, float(sigmas[t_start + i + 1]), last=i == n_exec - 1))
        if callback is not None and i % callback_steps == 0:
            callback(i, t, x)
    return img2img_denoise_loop(unet_fn, latents, prompt_embeds, neg_prompt_embeds, pooled, neg_pooled, time_ids,
                                num_inference_steps, strength, denoising_end=denoising_end, callback=blend,
                                callback_steps=1, **img2img_opts)
