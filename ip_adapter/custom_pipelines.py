"""StableDiffusionXLCustomPipeline with the reference's call surface (ip_adapter/custom_pipelines.py:16-394) on the
native UNet / DenoiseEngine.  The reference class derives from diffusers' StableDiffusionXLPipeline; diffusers is not
a dependency here, so the pieces the reference touches are provided directly:

    .unet (.config.{cross_attention_dim, block_out_channels, in_channels}, .attn_processors, .set_attn_processor)
    .scheduler, .set_scale(scale), .to(device), .enable_vae_tiling(), .encode_prompt(...), .__call__(...)

Denoise loop semantics follow custom_pipelines.py:188-363 (CFG batch [negative, positive], per-step IP-scale gating
by control_guidance_start/end, Euler update); the loop itself runs as replayed CUDA graphs (imagharmony_b200/denoise.py).
VAE decode / PIL post-processing (:365-386, scope row f1) runs on the native decoder `imagharmony_b200.vae` when the
pipeline owns one (`from_random`, or `from_pretrained` with a `vae/` folder); a `vae_decode` callable overrides it and
`output_type="latent"` skips it.
"""
from __future__ import annotations

import hashlib
import os
from dataclasses import dataclass
from typing import Any, Callable, Dict, List, Optional, Tuple, Union

import torch

from imagharmony_b200._lib import IHError
from imagharmony_b200.config import SDXL_BASE, UNetConfig
from imagharmony_b200.denoise import DenoiseEngine
from imagharmony_b200.scheduler import EulerDiscreteScheduler
from imagharmony_b200.unet import UNet2DConditionModel

from .utils import is_torch2_available

if is_torch2_available():
    from .attention_processor import IPAttnProcessor2_0 as IPAttnProcessor
else:  # pragma: no cover
    from .attention_processor import IPAttnProcessor


@dataclass
class StableDiffusionXLPipelineOutput:
    images: Any


class SyntheticPromptEncoder:
    """Stand-in for the two CLIP text encoders when no weights are on disk (this environment has no network):
    deterministic N(0,1) embeddings seeded by a hash of the prompt string.  Shapes/dtypes match encode_prompt [3P]."""

    def __init__(self, cfg: UNetConfig):
        self.cfg = cfg

    def __call__(self, prompts: List[str]) -> Tuple[torch.Tensor, torch.Tensor]:
        hs, pooled = [], []
        for p in prompts:
            seed = int.from_bytes(hashlib.sha256(p.encode()).digest()[:8], "little") & 0x7FFFFFFFFFFFFFFF
            g = torch.Generator("cpu").manual_seed(seed)
            hs.append(torch.randn(77, self.cfg.cross_attention_dim, generator=g))
            pooled.append(torch.randn(self.cfg.pooled_embed_dim, generator=g))
        return torch.stack(hs).half(), torch.stack(pooled).half()


class StableDiffusionXLCustomPipeline:
    vae_scale_factor = 8
    force_zeros_for_empty_prompt = True     # [3P] SDXL-base pipeline config

    def __init__(self, unet: UNet2DConditionModel, prompt_encoder: Optional[Callable] = None,
                 vae_decode: Optional[Callable] = None, scheduler: Optional[EulerDiscreteScheduler] = None,
                 vae=None):
        self.unet = unet
        self.vae = vae                      # imagharmony_b200.vae.AutoencoderKLDecoder or None
        self.scheduler = scheduler or EulerDiscreteScheduler()
        self.prompt_encoder = prompt_encoder or SyntheticPromptEncoder(unet.config)
        self.vae_decode = vae_decode
        self.default_sample_size = unet.config.sample_size
        self._engine: Optional[DenoiseEngine] = None
        self.device = unet.conv_in.weight.device

    # ---- construction ------------------------------------------------------------------------------------------
    @classmethod
    def from_random(cls, cfg: UNetConfig = SDXL_BASE, seed: int = 0, device="cuda", vae_cfg=None):
        """Random-init weights of the given architecture (the benchmark / test configuration)."""
        from imagharmony_b200.weights import random_state_dict, shapes_of
        with torch.device("meta"):
            shapes = shapes_of(UNet2DConditionModel(cfg))
        gen_dev = device if str(device).startswith("cuda") else "cpu"
        unet = UNet2DConditionModel.from_state_dict(cfg, random_state_dict(shapes, seed, device=gen_dev), device=device)
        vae = None
        if vae_cfg is not None:
            from imagharmony_b200.vae import AutoencoderKLDecoder
            with torch.device("meta"):
                vshapes = shapes_of(AutoencoderKLDecoder(vae_cfg))
            vae = AutoencoderKLDecoder.from_state_dict(vae_cfg, random_state_dict(vshapes, seed + 17, device=gen_dev),
                                                       device=device)
        return cls(unet, vae=vae)

    @classmethod
    def from_pretrained(cls, path: str, torch_dtype=torch.float16, add_watermarker: bool = False, device="cuda",
                        cfg: UNetConfig = SDXL_BASE, vae_cfg=None, **kwargs):
        """test.py:68-72.  Loads `<path>/unet/diffusion_pytorch_model.safetensors` (diffusers key names are the native
        UNet's key names, so no key map is needed)."""
        from safetensors.torch import load_file
        f = os.path.join(path, "unet", "diffusion_pytorch_model.safetensors")
        if not os.path.exists(f):
            f = os.path.join(path, "unet", "diffusion_pytorch_model.fp16.safetensors")
        if not os.path.exists(f):
            raise FileNotFoundError(f"no SDXL UNet weights under {path}/unet (safetensors)")
        unet = UNet2DConditionModel.from_state_dict(cfg, load_file(f), device=device)
        vae = None
        for name in ("diffusion_pytorch_model.fp16.safetensors", "diffusion_pytorch_model.safetensors"):
            vf = os.path.join(path, "vae", name)
            if os.path.exists(vf):
                import dataclasses
                import json
                from imagharmony_b200.config import SDXL_VAE
                from imagharmony_b200.vae import AutoencoderKLDecoder
                vcfg = vae_cfg or SDXL_VAE
                cj = os.path.join(path, "vae", "config.json")
                if vae_cfg is None and os.path.exists(cj):
                    # `force_upcast` decides between the scaled residual stream (the reference's fp32 upcast,
                    # custom_pipelines.py:366-371) and plain fp16 (fp16-fix checkpoints set it to false)
                    meta = json.load(open(cj))
                    vcfg = dataclasses.replace(vcfg, force_upcast=bool(meta.get("force_upcast", True)),
                                               scaling_factor=float(meta.get("scaling_factor", vcfg.scaling_factor)))
                vae = AutoencoderKLDecoder.from_state_dict(vcfg, load_file(vf), device=device)  # decoder keys only
                break
        enc = None
        from .encoders import ClipPromptEncoder
        if ClipPromptEncoder.available(path):
            enc = ClipPromptEncoder.from_pretrained(path, device=device, dtype=torch_dtype)
        return cls(unet, prompt_encoder=enc, vae=vae)

    def to(self, device=None, *args, **kwargs):
        """Weights live on the device the UNet was built on (from_random / from_pretrained take `device=`); moving 5 GB
        of kernel-layout weights behind the caller's back is not offered, a mismatching request raises."""
        if device is not None and not isinstance(device, torch.dtype):
            want = torch.device(device)
            have = torch.device(self.device)
            if want.type != have.type or (want.index is not None and have.index is not None and want.index != have.index):
                raise IHError(f"pipeline was built on {have}; build it with device={want!s} instead of .to({want!s})")
        return self

    def enable_vae_tiling(self):  # test.py:73
        if self.vae is not None:
            self.vae.use_tiling = True

    # ---- reference surface -------------------------------------------------------------------------------------
    def set_scale(self, scale):
        for attn_processor in self.unet.attn_processors.values():           # custom_pipelines.py:17-20
            if isinstance(attn_processor, IPAttnProcessor):
                attn_processor.scale = scale

    @property
    def engine(self) -> DenoiseEngine:
        if self._engine is None or self._engine.scheduler is not self.scheduler:
            # the loop integrates the SAME scheduler object whose init_noise_sigma scaled the initial latents
            self._engine = DenoiseEngine(self.unet, scheduler=self.scheduler)
        return self._engine

    @torch.no_grad()
    def encode_prompt(self, prompt, prompt_2=None, device=None, num_images_per_prompt: int = 1,
                      do_classifier_free_guidance: bool = True, negative_prompt=None, negative_prompt_2=None,
                      prompt_embeds=None, negative_prompt_embeds=None, pooled_prompt_embeds=None,
                      negative_pooled_prompt_embeds=None, lora_scale=None, **kwargs):
        """-> (prompt_embeds [n,77,2048], negative_prompt_embeds, pooled [n,1280], negative_pooled)  ([3P] A.4)."""
        if prompt_embeds is None:
            prompts = [prompt] if isinstance(prompt, str) else list(prompt)
            prompt_embeds, pooled_prompt_embeds = self.prompt_encoder(prompts)
            prompt_embeds = prompt_embeds.repeat_interleave(num_images_per_prompt, dim=0)
            pooled_prompt_embeds = pooled_prompt_embeds.repeat_interleave(num_images_per_prompt, dim=0)
        if do_classifier_free_guidance and negative_prompt_embeds is None and negative_prompt is None \
                and self.force_zeros_for_empty_prompt:
            # [3P] SDXL-base model_index.json: force_zeros_for_empty_prompt = true -> no negative prompt means ZERO embeds
            negative_prompt_embeds = torch.zeros_like(prompt_embeds)
            negative_pooled_prompt_embeds = torch.zeros_like(pooled_prompt_embeds)
        elif do_classifier_free_guidance and negative_prompt_embeds is None:
            negs = negative_prompt if negative_prompt is not None else ""
            negs = [negs] * (prompt_embeds.shape[0] // num_images_per_prompt) if isinstance(negs, str) else list(negs)
            negative_prompt_embeds, negative_pooled_prompt_embeds = self.prompt_encoder(negs)
            negative_prompt_embeds = negative_prompt_embeds.repeat_interleave(num_images_per_prompt, dim=0)
            negative_pooled_prompt_embeds = negative_pooled_prompt_embeds.repeat_interleave(num_images_per_prompt, dim=0)
        return prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds

    def prepare_latents(self, batch_size, num_channels_latents, height, width, dtype, device, generator, latents=None):
        """[3P] diffusers prepare_latents: randn * init_noise_sigma; a list of generators draws one sample each."""
        shape = (batch_size, num_channels_latents, height // self.vae_scale_factor, width // self.vae_scale_factor)
        if latents is None:
            if isinstance(generator, list):
                if len(generator) != batch_size:
                    raise ValueError(f"got {len(generator)} generators for a batch of {batch_size}")
                parts = [torch.randn((1,) + shape[1:], generator=g, device=g.device, dtype=torch.float32) for g in generator]
                latents = torch.cat([p.to("cpu") for p in parts], dim=0)
            else:
                gdev = generator.device if generator is not None else "cpu"
                latents = torch.randn(shape, generator=generator, device=gdev, dtype=torch.float32).to("cpu")
        latents = latents.to(torch.float32) * self.scheduler.init_noise_sigma
        return latents.to(dtype)

    @torch.no_grad()
    def __call__(self, prompt: Optional[Union[str, List[str]]] = None, prompt_2=None, height: Optional[int] = None,
                 width: Optional[int] = None, num_inference_steps: int = 50, denoising_end: Optional[float] = None,
                 guidance_scale: float = 5.0, negative_prompt=None, negative_prompt_2=None,
                 num_images_per_prompt: Optional[int] = 1, eta: float = 0.0, generator=None,
                 latents: Optional[torch.Tensor] = None, prompt_embeds: Optional[torch.Tensor] = None,
                 negative_prompt_embeds: Optional[torch.Tensor] = None,
                 pooled_prompt_embeds: Optional[torch.Tensor] = None,
                 negative_pooled_prompt_embeds: Optional[torch.Tensor] = None, output_type: Optional[str] = "pil",
                 return_dict: bool = True, callback=None, callback_steps: int = 1,
                 cross_attention_kwargs: Optional[Dict[str, Any]] = None, guidance_rescale: float = 0.0,
                 original_size: Optional[Tuple[int, int]] = None, crops_coords_top_left: Tuple[int, int] = (0, 0),
                 target_size: Optional[Tuple[int, int]] = None, negative_original_size=None,
                 negative_crops_coords_top_left=(0, 0), negative_target_size=None,
                 control_guidance_start: float = 0.0, control_guidance_end: float = 1.0, **ignored):
        """Parameter list of custom_pipelines.py:23-56.  Unknown keyword arguments are accepted and ignored, because
        IPAdapterXL.generate forwards a stray `number_class_crossattention=` into this call (test.py:38, demo.py:124)."""
        height = height or self.default_sample_size * self.vae_scale_factor           # :189-190
        width = width or self.default_sample_size * self.vae_scale_factor
        original_size = original_size or (height, width)                              # :192-193
        target_size = target_size or (height, width)
        if callback is not None and (not isinstance(callback_steps, int) or callback_steps <= 0):
            raise ValueError(f"`callback_steps` has to be a positive integer but is {callback_steps}")   # [3P] check_inputs
        do_classifier_free_guidance = guidance_scale > 1.0                            # :223
        (prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds) = \
            self.encode_prompt(prompt, prompt_2, None, num_images_per_prompt, do_classifier_free_guidance,
                               negative_prompt, negative_prompt_2, prompt_embeds, negative_prompt_embeds,
                               pooled_prompt_embeds, negative_pooled_prompt_embeds)  # :229-247
        batch = prompt_embeds.shape[0]
        self.scheduler.set_timesteps(num_inference_steps)                             # :250
        lat = self.prepare_latents(batch, self.unet.config.in_channels, height, width, torch.float16, self.device,
                                   generator, latents)                               # :255-265

        def time_ids(size, crop, target):                                             # :277-284 _get_add_time_ids [3P]
            return torch.tensor([list(size) + list(crop) + list(target)], dtype=torch.float32).repeat(batch, 1)
        add_time_ids = time_ids(original_size, crops_coords_top_left, target_size)
        negative_add_time_ids = None
        if negative_original_size is not None and negative_target_size is not None:   # :285-294
            negative_add_time_ids = time_ids(negative_original_size, negative_crops_coords_top_left, negative_target_size)
        loop_steps = num_inference_steps
        if denoising_end is not None and isinstance(denoising_end, float) and 0 < denoising_end < 1:   # :307-316
            n_train = self.scheduler.num_train_timesteps
            cutoff = int(round(n_train - denoising_end * n_train))
            loop_steps = int(sum(1 for t in self.scheduler.timesteps if t >= cutoff))
        conditioning_scale = 1.0
        for attn_processor in self.unet.attn_processors.values():                     # :319-322
            if isinstance(attn_processor, IPAttnProcessor):
                conditioning_scale = attn_processor.scale
                break
        if loop_steps > 0:
            out = self.engine.run(lat, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds,
                                  negative_pooled_prompt_embeds, add_time_ids, num_inference_steps,
                                  guidance_scale=guidance_scale, ip_scale=conditioning_scale,
                                  control_guidance_start=control_guidance_start,
                                  control_guidance_end=control_guidance_end, guidance_rescale=guidance_rescale,
                                  num_loop_steps=loop_steps, callback=callback, callback_steps=callback_steps,
                                  negative_time_ids=negative_add_time_ids)
        else:
            out = lat.to(self.device)
        self.set_scale(conditioning_scale)
        if output_type == "latent":
            image = out
        else:
            if self.vae_decode is not None:
                image = self.vae_decode(out / 0.13025, output_type)                   # :373 (scaling_factor [3P])
            elif self.vae is not None:
                from imagharmony_b200.vae import postprocess
                image = postprocess(self.vae.decode(out), output_type)                # :373 + :383 (/ scaling_factor folded)
            else:
                raise IHError("this pipeline has no VAE decoder: call with output_type='latent', build it with a `vae` "
                              "(from_random(vae_cfg=...), from_pretrained with a vae/ folder) or pass a vae_decode callable")
        if not return_dict:
            return (image,)
        return StableDiffusionXLPipelineOutput(images=image)


class StableDiffusionXLImg2ImgCustomPipeline(StableDiffusionXLCustomPipeline):
    """Image-to-image editing on the same call surface: `image=` (the source) and `strength=` on top of the
    text-to-image parameters, following [3P] diffusers==0.30.0 `StableDiffusionXLImg2ImgPipeline`.

    The source image is encoded by the native VAE encoder (`imagharmony_b200.vae.AutoencoderKLEncoder`), its posterior
    sample is scaled and noised to sigma[t_start] in one kernel, and the denoise loop runs only the last
    T - t_start = min(int(T * strength), T) steps of the T-step schedule.  IPAdapterXL.generate(image=..., strength=...)
    reaches this call through its **kwargs."""

    def __init__(self, unet: UNet2DConditionModel, prompt_encoder: Optional[Callable] = None,
                 vae_decode: Optional[Callable] = None, scheduler: Optional[EulerDiscreteScheduler] = None,
                 vae=None, vae_encoder=None):
        super().__init__(unet, prompt_encoder=prompt_encoder, vae_decode=vae_decode, scheduler=scheduler, vae=vae)
        self.vae_encoder = vae_encoder      # imagharmony_b200.vae.AutoencoderKLEncoder or None

    # ---- construction ------------------------------------------------------------------------------------------
    @classmethod
    def from_random(cls, cfg: UNetConfig = SDXL_BASE, seed: int = 0, device="cuda", vae_cfg=None):
        """As the text-to-image pipeline, plus a random-init VAE encoder when `vae_cfg` is given."""
        pipe = super().from_random(cfg, seed=seed, device=device, vae_cfg=vae_cfg)
        if vae_cfg is not None:
            from imagharmony_b200.vae import AutoencoderKLEncoder
            from imagharmony_b200.weights import random_state_dict, shapes_of
            with torch.device("meta"):
                eshapes = shapes_of(AutoencoderKLEncoder(vae_cfg))
            gen_dev = device if str(device).startswith("cuda") else "cpu"
            pipe.vae_encoder = AutoencoderKLEncoder.from_state_dict(
                vae_cfg, random_state_dict(eshapes, seed + 18, device=gen_dev), device=device)
        return pipe

    @classmethod
    def from_pretrained(cls, path: str, torch_dtype=torch.float16, add_watermarker: bool = False, device="cuda",
                        cfg: UNetConfig = SDXL_BASE, vae_cfg=None, **kwargs):
        """As the text-to-image pipeline; the encoder half is loaded from the same `vae/` safetensors, with the same
        `force_upcast` / `scaling_factor` from its config.json."""
        pipe = super().from_pretrained(path, torch_dtype=torch_dtype, add_watermarker=add_watermarker, device=device,
                                       cfg=cfg, vae_cfg=vae_cfg, **kwargs)
        if pipe.vae is not None:
            from safetensors.torch import load_file
            from imagharmony_b200.vae import AutoencoderKLEncoder
            for name in ("diffusion_pytorch_model.fp16.safetensors", "diffusion_pytorch_model.safetensors"):
                vf = os.path.join(path, "vae", name)
                if os.path.exists(vf):
                    pipe.vae_encoder = AutoencoderKLEncoder.from_state_dict(pipe.vae.config, load_file(vf), device=device)
                    break
        return pipe

    def enable_vae_tiling(self):  # test.py:73; tiles both halves
        super().enable_vae_tiling()
        if self.vae_encoder is not None:
            self.vae_encoder.use_tiling = True

    # ---- img2img -----------------------------------------------------------------------------------------------
    @staticmethod
    def get_timesteps(num_inference_steps: int, strength: float) -> Tuple[int, int]:
        """[3P] get_timesteps: -> (t_start, executed steps), init_timestep = min(int(T * strength), T)."""
        init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
        t_start = max(num_inference_steps - init_timestep, 0)
        return t_start, num_inference_steps - t_start

    def preprocess_image(self, image):
        """-> ("pixels", uint8 NHWC [B, H, W, 3]) for PIL input (size rounded down to a multiple of 8 with a Lanczos resize,
        [3P] VaeImageProcessor), ("image", float32 NCHW in [-1, 1]) for a 3-channel tensor (normalised 2 x - 1 unless its
        minimum is < 0), ("latents", fp16 NCHW) for a tensor with latent_channels channels (used as it is)."""
        import numpy as np
        from PIL import Image
        if isinstance(image, Image.Image) or (isinstance(image, (list, tuple)) and image
                                              and isinstance(image[0], Image.Image)):
            images = [image] if isinstance(image, Image.Image) else list(image)
            arrs = []
            for im in images:
                im = im.convert("RGB")
                w, h = (im.width // self.vae_scale_factor) * self.vae_scale_factor, \
                       (im.height // self.vae_scale_factor) * self.vae_scale_factor
                if (w, h) != im.size:
                    im = im.resize((w, h), resample=Image.LANCZOS)
                arrs.append(np.asarray(im, dtype=np.uint8))
            if len({a.shape for a in arrs}) != 1:
                raise ValueError("all source images must have the same size")
            return "pixels", torch.from_numpy(np.stack(arrs)).to(self.device)
        if isinstance(image, torch.Tensor):
            x = image if image.dim() == 4 else image.unsqueeze(0)
            if x.shape[1] == self.unet.config.in_channels:
                return "latents", x.to(self.device, torch.float16).contiguous()
            x = x.to(torch.float32)
            if x.min() >= 0:
                x = 2.0 * x - 1.0
            return "image", x.to(self.device).contiguous()
        raise TypeError(f"image must be a PIL image, a list of PIL images or a torch tensor, got {type(image)}")

    def prepare_img2img_latents(self, image, batch: int, generator, sigma: float) -> Tuple[torch.Tensor, Tuple[int, int]]:
        """Initial latents [batch, 4, h, w] fp16 on the device, and the source image size (H, W).

        Draw order ([3P] prepare_latents + retrieve_latents + randn_tensor): the posterior eps (fp32, the mean's shape)
        first, then the noise (fp16).  With a generator list, one [1, 4, h, w] eps per batch slot (the images replicated
        to the batch) and then one noise per slot, so a candidate does not depend on its batch slot."""
        kind, x = self.preprocess_image(image)
        n_img = x.shape[0]
        if batch % n_img:
            raise ValueError(f"cannot duplicate {n_img} source images to a batch of {batch}")
        if isinstance(generator, list) and len(generator) != batch:
            raise ValueError(f"got {len(generator)} generators for a batch of {batch}")
        L = self.unet.config.in_channels

        def randn(shape, g, dtype):
            return torch.randn(shape, generator=g, device=g.device if g is not None else "cpu", dtype=dtype)
        if kind == "latents":
            moments, eps = x.permute(0, 2, 3, 1).contiguous(), None
            h, w = x.shape[2], x.shape[3]
            size = (h * self.vae_scale_factor, w * self.vae_scale_factor)
        else:
            if self.vae_encoder is None:
                raise IHError("this pipeline has no VAE encoder: build it with from_random(vae_cfg=...) or from_pretrained "
                              "with a vae/ folder, or pass latents as a 4-channel image tensor")
            size = (x.shape[1], x.shape[2]) if kind == "pixels" else (x.shape[2], x.shape[3])
            moments = self.vae_encoder.encode(x)                  # once per source image: the moments are deterministic
            h, w = moments.shape[1], moments.shape[2]
            if isinstance(generator, list):
                eps = torch.cat([randn((1, L, h, w), g, torch.float32).to(self.device) for g in generator], dim=0)
            else:
                eps = randn((n_img, L, h, w), generator, torch.float32).to(self.device)
        if isinstance(generator, list):
            noise = torch.cat([randn((1, L, h, w), g, torch.float16).to(self.device) for g in generator], dim=0)
        else:
            noise = randn((batch, L, h, w), generator, torch.float16).to(self.device)
        from imagharmony_b200 import ops
        sf = 1.0 if eps is None else self.vae_encoder.config.scaling_factor
        return ops.vae_sample_add_noise(moments, eps, noise, L, sf, sigma), size

    @torch.no_grad()
    def __call__(self, prompt: Optional[Union[str, List[str]]] = None, prompt_2=None, image=None, strength: float = 0.3,
                 height: Optional[int] = None, width: Optional[int] = None, num_inference_steps: int = 50,
                 denoising_end: Optional[float] = None, guidance_scale: float = 5.0, negative_prompt=None,
                 negative_prompt_2=None, num_images_per_prompt: Optional[int] = 1, eta: float = 0.0, generator=None,
                 latents: Optional[torch.Tensor] = None, prompt_embeds: Optional[torch.Tensor] = None,
                 negative_prompt_embeds: Optional[torch.Tensor] = None,
                 pooled_prompt_embeds: Optional[torch.Tensor] = None,
                 negative_pooled_prompt_embeds: Optional[torch.Tensor] = None, output_type: Optional[str] = "pil",
                 return_dict: bool = True, callback=None, callback_steps: int = 1,
                 cross_attention_kwargs: Optional[Dict[str, Any]] = None, guidance_rescale: float = 0.0,
                 original_size: Optional[Tuple[int, int]] = None, crops_coords_top_left: Tuple[int, int] = (0, 0),
                 target_size: Optional[Tuple[int, int]] = None, negative_original_size=None,
                 negative_crops_coords_top_left=(0, 0), negative_target_size=None,
                 control_guidance_start: float = 0.0, control_guidance_end: float = 1.0, aesthetic_score: float = 6.0,
                 negative_aesthetic_score: float = 2.5, **ignored):
        """The text-to-image parameters plus `image` and `strength`.  The latent size comes from the image (`height` /
        `width` and `latents` are not used); `aesthetic_score*` are accepted and ignored (SDXL-base has
        requires_aesthetics_score = false, so its time ids equal the text-to-image ones)."""
        if image is None:
            raise ValueError("img2img needs a source `image`")
        t_start = self._check_edit_args(strength, num_inference_steps, callback, callback_steps)
        do_classifier_free_guidance = guidance_scale > 1.0
        (prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds) = \
            self.encode_prompt(prompt, prompt_2, None, num_images_per_prompt, do_classifier_free_guidance,
                               negative_prompt, negative_prompt_2, prompt_embeds, negative_prompt_embeds,
                               pooled_prompt_embeds, negative_pooled_prompt_embeds)
        batch = prompt_embeds.shape[0]
        self.scheduler.set_timesteps(num_inference_steps)
        sigma = float(self.scheduler.sigmas[t_start])                   # add_noise at the begin index t_start
        lat, size = self.prepare_img2img_latents(image, batch, generator, sigma)
        return self._denoise_and_decode(
            lat, t_start, num_inference_steps, (prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds,
                                                negative_pooled_prompt_embeds),
            guidance_scale=guidance_scale, denoising_end=denoising_end, guidance_rescale=guidance_rescale,
            original_size=original_size or size, crops_coords_top_left=crops_coords_top_left,
            target_size=target_size or size, negative_original_size=negative_original_size,
            negative_crops_coords_top_left=negative_crops_coords_top_left, negative_target_size=negative_target_size,
            control_guidance_start=control_guidance_start, control_guidance_end=control_guidance_end,
            callback=callback, callback_steps=callback_steps, output_type=output_type, return_dict=return_dict)

    def _check_edit_args(self, strength: float, num_inference_steps: int, callback, callback_steps) -> int:
        """Validates the editing arguments; -> t_start."""
        if not 0.0 <= strength <= 1.0:
            raise ValueError(f"The value of strength should be in [0.0, 1.0] but is {strength}")
        if callback is not None and (not isinstance(callback_steps, int) or callback_steps <= 0):
            raise ValueError(f"`callback_steps` has to be a positive integer but is {callback_steps}")
        t_start, n_exec = self.get_timesteps(num_inference_steps, strength)
        if n_exec < 1:
            raise ValueError(f"strength {strength} with num_inference_steps {num_inference_steps} leaves no denoising "
                             "step (the number of steps run is min(int(num_inference_steps * strength), num_inference_steps))")
        return t_start

    def _denoise_and_decode(self, lat, t_start: int, num_inference_steps: int, embeds, *, guidance_scale,
                            denoising_end, guidance_rescale, original_size, crops_coords_top_left, target_size,
                            negative_original_size, negative_crops_coords_top_left, negative_target_size,
                            control_guidance_start, control_guidance_end, callback, callback_steps, output_type,
                            return_dict, inpaint=None):
        """The editing loop from t_start (gating and callback counted over the executed steps) and the decode tail;
        `inpaint` is DenoiseEngine.run's."""
        prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds = embeds
        batch = prompt_embeds.shape[0]

        def time_ids(size, crop, target):
            return torch.tensor([list(size) + list(crop) + list(target)], dtype=torch.float32).repeat(batch, 1)
        add_time_ids = time_ids(original_size, crops_coords_top_left, target_size)
        negative_add_time_ids = None
        if negative_original_size is not None and negative_target_size is not None:
            negative_add_time_ids = time_ids(negative_original_size, negative_crops_coords_top_left, negative_target_size)
        loop_steps = num_inference_steps                                # denoising_end cuts the full schedule's list
        if denoising_end is not None and isinstance(denoising_end, float) and 0 < denoising_end < 1:
            n_train = self.scheduler.num_train_timesteps
            cutoff = int(round(n_train - denoising_end * n_train))
            loop_steps = int(sum(1 for t in self.scheduler.timesteps if t >= cutoff))
        conditioning_scale = 1.0
        for attn_processor in self.unet.attn_processors.values():
            if isinstance(attn_processor, IPAttnProcessor):
                conditioning_scale = attn_processor.scale
                break
        if loop_steps > t_start:
            out = self.engine.run(lat, prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds,
                                  negative_pooled_prompt_embeds, add_time_ids, num_inference_steps,
                                  guidance_scale=guidance_scale, ip_scale=conditioning_scale,
                                  control_guidance_start=control_guidance_start,
                                  control_guidance_end=control_guidance_end, guidance_rescale=guidance_rescale,
                                  start_step=t_start, num_loop_steps=loop_steps, callback=callback,
                                  callback_steps=callback_steps, negative_time_ids=negative_add_time_ids,
                                  count_from_start=True, inpaint=inpaint)
        else:
            out = lat
        self.set_scale(conditioning_scale)
        if output_type == "latent":
            image = out
        elif self.vae_decode is not None:
            image = self.vae_decode(out / 0.13025, output_type)
        elif self.vae is not None:
            from imagharmony_b200.vae import postprocess
            image = postprocess(self.vae.decode(out), output_type)
        else:
            raise IHError("this pipeline has no VAE decoder: call with output_type='latent', build it with a `vae` "
                          "(from_random(vae_cfg=...), from_pretrained with a vae/ folder) or pass a vae_decode callable")
        if not return_dict:
            return (image,)
        return StableDiffusionXLPipelineOutput(images=image)


class StableDiffusionXLInpaintCustomPipeline(StableDiffusionXLImg2ImgCustomPipeline):
    """Masked inpainting on the img2img call surface: `image=` (the source), `mask_image=` (white = regenerate) and
    `strength=`, following [3P] diffusers==0.30.0 `StableDiffusionXLInpaintPipeline` with the 4-channel SDXL-base UNet
    (the rules are stated in oracle/inpaint_ref.py).  Unlike img2img, the output size is `height` x `width` (default
    unet sample_size * 8) and the source image is resized to it.  After every denoising step the latents outside the
    mask are replaced by the source image's latents noised to the next sigma; the replacement runs inside the Euler
    kernel of the CUDA-graph loop (`DenoiseEngine.run(inpaint=...)`).  IPAdapterXL.generate(image=..., mask_image=...)
    reaches this call through its **kwargs; `pil_image` stays the IP reference."""

    def preprocess_mask(self, mask_image, height: int, width: int) -> torch.Tensor:
        """-> uint8 grayscale mask [Bm, height, width] on the device.  PIL masks are converted to "L" and
        Lanczos-resized to (width, height); a float tensor [H, W], [B, H, W] or [B, 1, H, W] with values in [0, 1] must
        already be (height, width) and is binarized at 0.5 here (to 255 / 0)."""
        import numpy as np
        from PIL import Image
        if isinstance(mask_image, torch.Tensor):
            m = mask_image.float()
            m = m[None] if m.dim() == 2 else (m[:, 0] if m.dim() == 4 and m.shape[1] == 1 else m)
            if m.dim() != 3 or tuple(m.shape[1:]) != (height, width):
                raise ValueError(f"a tensor mask must be [H, W], [B, H, W] or [B, 1, H, W] with (H, W) = "
                                 f"({height}, {width}), got {tuple(mask_image.shape)}")
            if m.numel() and (m.min() < 0 or m.max() > 1):
                raise ValueError("a tensor mask must have values in [0, 1]")
            return torch.where(m >= 0.5, 255, 0).to(device=self.device, dtype=torch.uint8).contiguous()
        if isinstance(mask_image, Image.Image) or (isinstance(mask_image, (list, tuple)) and mask_image
                                                   and all(isinstance(m, Image.Image) for m in mask_image)):
            arrs = []
            for im in [mask_image] if isinstance(mask_image, Image.Image) else list(mask_image):
                im = im.convert("L")
                if im.size != (width, height):
                    im = im.resize((width, height), resample=Image.LANCZOS)
                arrs.append(np.asarray(im, dtype=np.uint8))
            return torch.from_numpy(np.stack(arrs)).to(self.device)
        raise TypeError(f"mask_image must be a PIL image, a list of PIL images or a torch tensor, got {type(mask_image)}")

    def prepare_inpaint_latents(self, image, mask_image, batch: int, generator, height: int, width: int, t_start: int,
                                is_strength_max: bool):
        """-> (start latents [batch, 4, h, w] fp16, (latent mask uint8 {0, 1} [Bm, h, w], z0, noise)), the second item
        being DenoiseEngine.run's `inpaint`.  Call after scheduler.set_timesteps.

        Draw order ([3P] prepare_latents with a 4-channel UNet): the posterior eps (fp32) and then the noise (fp16).  With
        a generator list, source image i draws its eps from generator[i] for i < n_img only -- the images are encoded as
        they are, not replicated to the batch as in img2img -- and batch slot b then draws its noise from generator[b]."""
        from PIL import Image
        if isinstance(image, (Image.Image, list, tuple)):
            images = [image] if isinstance(image, Image.Image) else list(image)
            if not all(isinstance(im, Image.Image) for im in images):
                raise TypeError("image must be a PIL image, a list of PIL images or a torch tensor")
            image = [im if im.size == (width, height) else im.convert("RGB").resize((width, height), resample=Image.LANCZOS)
                     for im in images]                          # preprocess_image converts the rest to RGB
        kind, x = self.preprocess_image(image)
        h, w = height // self.vae_scale_factor, width // self.vae_scale_factor
        have = tuple(x.shape[2:]) if kind != "pixels" else tuple(x.shape[1:3])
        if have != ((h, w) if kind == "latents" else (height, width)):
            raise ValueError(f"a tensor image must match height x width = {height} x {width}, got {tuple(x.shape)}")
        n_img = x.shape[0]
        if batch % n_img:
            raise ValueError(f"cannot duplicate {n_img} source images to a batch of {batch}")
        if isinstance(generator, list) and len(generator) != batch:
            raise ValueError(f"got {len(generator)} generators for a batch of {batch}")
        mask_u8 = self.preprocess_mask(mask_image, height, width)
        if batch % mask_u8.shape[0]:
            raise ValueError(f"{mask_u8.shape[0]} masks do not divide the batch of {batch}")
        L = self.unet.config.in_channels

        def randn(shape, g, dtype):
            return torch.randn(shape, generator=g, device=g.device if g is not None else "cpu", dtype=dtype)
        if kind == "latents":
            moments, eps = x.permute(0, 2, 3, 1).contiguous(), None
        else:
            if self.vae_encoder is None:
                raise IHError("this pipeline has no VAE encoder: build it with from_random(vae_cfg=...) or from_pretrained "
                              "with a vae/ folder, or pass latents as a 4-channel image tensor")
            moments = self.vae_encoder.encode(x)
            if isinstance(generator, list):
                eps = torch.cat([randn((1, L, h, w), generator[i], torch.float32).to(self.device) for i in range(n_img)])
            else:
                eps = randn((n_img, L, h, w), generator, torch.float32).to(self.device)
        if isinstance(generator, list):
            noise = torch.cat([randn((1, L, h, w), g, torch.float16).to(self.device) for g in generator], dim=0)
        else:
            noise = randn((batch, L, h, w), generator, torch.float16).to(self.device)
        from imagharmony_b200 import ops
        sf = 1.0 if eps is None else self.vae_encoder.config.scaling_factor
        sigma = float(self.scheduler.init_noise_sigma if is_strength_max else self.scheduler.sigmas[t_start])
        lat, z0 = ops.vae_sample_inpaint(moments, eps, noise, L, sf, sigma, is_strength_max)
        return lat, (ops.latent_mask(mask_u8), z0, noise)

    @torch.no_grad()
    def __call__(self, prompt: Optional[Union[str, List[str]]] = None, prompt_2=None, image=None, mask_image=None,
                 height: Optional[int] = None, width: Optional[int] = None, strength: float = 0.9999,
                 num_inference_steps: int = 50, denoising_end: Optional[float] = None, guidance_scale: float = 5.0,
                 negative_prompt=None, negative_prompt_2=None, num_images_per_prompt: Optional[int] = 1,
                 eta: float = 0.0, generator=None, latents: Optional[torch.Tensor] = None,
                 prompt_embeds: Optional[torch.Tensor] = None, negative_prompt_embeds: Optional[torch.Tensor] = None,
                 pooled_prompt_embeds: Optional[torch.Tensor] = None,
                 negative_pooled_prompt_embeds: Optional[torch.Tensor] = None, output_type: Optional[str] = "pil",
                 return_dict: bool = True, callback=None, callback_steps: int = 1,
                 cross_attention_kwargs: Optional[Dict[str, Any]] = None, guidance_rescale: float = 0.0,
                 original_size: Optional[Tuple[int, int]] = None, crops_coords_top_left: Tuple[int, int] = (0, 0),
                 target_size: Optional[Tuple[int, int]] = None, negative_original_size=None,
                 negative_crops_coords_top_left=(0, 0), negative_target_size=None,
                 control_guidance_start: float = 0.0, control_guidance_end: float = 1.0, aesthetic_score: float = 6.0,
                 negative_aesthetic_score: float = 2.5, **ignored):
        """The img2img parameters plus `mask_image`, `height` and `width` (default unet sample_size * 8, multiples of
        8).  `strength` = 1.0 starts from pure noise; the source latents are still used by the blend.  `latents` is not
        used; `aesthetic_score*` are accepted and ignored, as in img2img."""
        if image is None or mask_image is None:
            raise ValueError("inpainting needs a source `image` and a `mask_image`")
        height = height or self.default_sample_size * self.vae_scale_factor
        width = width or self.default_sample_size * self.vae_scale_factor
        if height % self.vae_scale_factor or width % self.vae_scale_factor:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        t_start = self._check_edit_args(strength, num_inference_steps, callback, callback_steps)
        do_classifier_free_guidance = guidance_scale > 1.0
        embeds = self.encode_prompt(prompt, prompt_2, None, num_images_per_prompt, do_classifier_free_guidance,
                                    negative_prompt, negative_prompt_2, prompt_embeds, negative_prompt_embeds,
                                    pooled_prompt_embeds, negative_pooled_prompt_embeds)
        self.scheduler.set_timesteps(num_inference_steps)
        lat, inpaint = self.prepare_inpaint_latents(image, mask_image, embeds[0].shape[0], generator, height, width,
                                                    t_start, strength == 1.0)
        return self._denoise_and_decode(
            lat, t_start, num_inference_steps, embeds, guidance_scale=guidance_scale, denoising_end=denoising_end,
            guidance_rescale=guidance_rescale, original_size=original_size or (height, width),
            crops_coords_top_left=crops_coords_top_left, target_size=target_size or (height, width),
            negative_original_size=negative_original_size, negative_crops_coords_top_left=negative_crops_coords_top_left,
            negative_target_size=negative_target_size, control_guidance_start=control_guidance_start,
            control_guidance_end=control_guidance_end, callback=callback, callback_steps=callback_steps,
            output_type=output_type, return_dict=return_dict, inpaint=inpaint)
