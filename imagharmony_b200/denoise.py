"""The denoise loop of custom_pipelines.py:325-363 as a device-resident loop.

One step = UNet forward on the scaled (CFG) batch + the fused guidance/Euler kernel; everything a step needs (timestep,
sigma pair, step index) is read from device memory, so the step is captured ONCE as a CUDA graph and replayed T times
with no host work in between.  Step-invariant work (cross-attention K/V of all 70 attn2 layers, the text_time
embedding) runs once per call in `prepare`.

Loop options of the reference that are honoured here (all graph-replayed; a callback only breaks the replay sequence,
not the graph): classifier-free guidance on or off (`guidance_scale <= 1`, :223,:332,:348), `guidance_rescale`
(:352-354), `denoising_end` (:307-316, via `num_loop_steps`), `callback` / `callback_steps` (:359-363),
`control_guidance_start/end` IP-scale gating (:326-329), negative micro-conditioning time ids (:286-300).
Inpainting (`inpaint=`) blends the latents with the source image's inside the same Euler kernel, so a masked step
launches as many kernels as a plain one.

Graph lifetime: a captured graph holds raw pointers.  Everything it reads lives in buffers that are owned per shape
and never freed while the graph exists -- the engine's static inputs (`_static`, and `_inpaint_static` for the
mask, z0, noise and last-step index), the processors' K/V buffers and the UNet's add-embedding buffer (per-shape
dicts inside those objects), and the library's grow-only scratch buffers whose re-allocation bumps
`ops.workspace_generation()`.  A graph is replayed only if it was captured under the current UNet `graph_epoch`
(weights / processors unchanged) and the current workspace generation; otherwise it is re-captured.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional, Tuple

import torch

from . import ops
from ._lib import IHError
from .scheduler import EulerDiscreteScheduler
from .unet import UNet2DConditionModel


class DenoiseEngine:
    def __init__(self, unet: UNet2DConditionModel, use_cuda_graph: bool = True,
                 scheduler: Optional[EulerDiscreteScheduler] = None):
        self.unet = unet
        self.device = unet.conv_in.weight.device
        self.scheduler = scheduler or EulerDiscreteScheduler()      # the pipeline's own scheduler object when given
        self.use_cuda_graph = use_cuda_graph and self.device.type == "cuda"
        self._graphs: Dict[Tuple, Tuple[torch.cuda.CUDAGraph, int]] = {}   # key -> (graph, workspace generation)
        self._static: Dict[Tuple, dict] = {}
        self._inpaint_static: Dict[Tuple, dict] = {}
        self._tables: Dict[int, Tuple[torch.Tensor, torch.Tensor, float]] = {}
        self._epoch = getattr(unet, "graph_epoch", 0)
        self.last_launches_per_step = 0
        self.graphs_captured = 0

    # ------------------------------------------------------------------------------------------------------------
    def tables(self, num_steps: int):
        t = self._tables.get(num_steps)
        if t is None:
            s = self.scheduler.set_timesteps(num_steps)
            t = (torch.from_numpy(s.timesteps).to(self.device), torch.from_numpy(s.sigmas).to(self.device),
                 s.init_noise_sigma)
            self._tables[num_steps] = t
        return t

    def set_scale(self, scale: float) -> None:
        """IPAdapter.set_scale / pipeline.set_scale (ip_adapter.py:179-182, custom_pipelines.py:17-20)."""
        for p in self.unet.attn_processors.values():
            if hasattr(p, "to_k_ip"):
                p.scale = scale

    def invalidate_graphs(self) -> None:
        self._graphs.clear()

    def _buffers(self, n: int, h: int, w: int, L: int, use_cfg: bool = True):
        key = (n, h, w, L, use_cfg)
        st = self._static.get(key)
        if st is None:
            cfg = self.unet.config
            dev = self.device
            b = 2 * n if use_cfg else n
            st = {
                "latents": torch.empty((n, cfg.in_channels, h, w), dtype=torch.float16, device=dev),
                "model_in": torch.empty((b, cfg.in_channels, h, w), dtype=torch.float16, device=dev),
                "ehs": torch.empty((b, L, cfg.cross_attention_dim), dtype=torch.float16, device=dev),
                "text_embeds": torch.empty((b, cfg.pooled_embed_dim), dtype=torch.float16, device=dev),
                "time_ids": torch.empty((b, 6), dtype=torch.float32, device=dev),
                "step": torch.zeros((1,), dtype=torch.int32, device=dev),
            }
            self._static[key] = st
        return st

    def _inpaint_buffers(self, n: int, h: int, w: int, n_masks: int):
        key = (n, h, w, n_masks)
        bs = self._inpaint_static.get(key)
        if bs is None:
            dev = self.device
            L = self.unet.config.in_channels
            bs = {
                "mask": torch.empty((n_masks, h, w), dtype=torch.uint8, device=dev),
                "z0": torch.empty((n, L, h, w), dtype=torch.float16, device=dev),
                "noise": torch.empty((n, L, h, w), dtype=torch.float16, device=dev),
                "last": torch.zeros((1,), dtype=torch.int32, device=dev),
            }
            self._inpaint_static[key] = bs
        return bs

    def _step(self, st, timesteps, sigmas, guidance, use_cfg=True, rescale=0.0, blend=None):
        noise = self.unet(st["model_in"], timesteps, st["ehs"], st["text_embeds"], st["time_ids"], step=st["step"])
        if blend is None:
            ops.euler_step(noise, st["latents"], st["model_in"], sigmas, st["step"], guidance, use_cfg=use_cfg,
                           guidance_rescale=rescale)
        else:
            ops.euler_step_inpaint(noise, st["latents"], st["model_in"], sigmas, st["step"], guidance, blend["mask"],
                                   blend["z0"], blend["noise"], blend["last"], use_cfg=use_cfg, guidance_rescale=rescale)

    # ------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def run(self, latents: torch.Tensor, prompt_embeds: torch.Tensor, negative_prompt_embeds: Optional[torch.Tensor],
            pooled: torch.Tensor, negative_pooled: Optional[torch.Tensor], time_ids: torch.Tensor,
            num_inference_steps: int, guidance_scale: float = 5.0, ip_scale: float = 1.0,
            control_guidance_start: float = 0.0, control_guidance_end: float = 1.0, stop_after: Optional[int] = None,
            start_step: int = 0, guidance_rescale: float = 0.0, num_loop_steps: Optional[int] = None,
            callback: Optional[Callable] = None, callback_steps: int = 1,
            negative_time_ids: Optional[torch.Tensor] = None, count_from_start: bool = False,
            inpaint: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None) -> torch.Tensor:
        """latents [n,4,h,w] (already scaled by init_noise_sigma; host or device); embeds host or device tensors.
        Returns the latents after the last executed step as a new device tensor.

        `stop_after` stops after step index k - 1 (PNS preview); `start_step` = k resumes a trajectory whose `latents`
        are the output of a `stop_after=k` call with the same schedule (two-phase PNS: preview all candidates,
        continue only the winner).  `num_loop_steps` = k truncates the timestep list to its first k entries the way
        `denoising_end` does (custom_pipelines.py:307-316: the gating fractions of :326 then use k, the sigma table
        stays the full schedule's).  `guidance_scale <= 1` runs the UNet on the positive branch only (:223).

        `count_from_start=True` is img2img (`start_step` = t_start of `strength`, the latents noised to sigma[t_start]):
        the control_guidance_start/end fractions and the callback's step index then count the executed steps from 0 over
        the truncated list (steps start_step .. loop end), as `enumerate(timesteps)` does in [3P] diffusers' img2img
        loop.  The default counts from the start of the full schedule (a resumed PNS trajectory).

        `inpaint=(mask, z0, noise)` is masked inpainting ([3P] diffusers StableDiffusionXLInpaintPipeline, 4-channel
        UNet): mask uint8 {0, 1} [Bm, h, w] (1 = regenerate; latent image b uses mask b % Bm), z0 and noise fp16
        [n, 4, h, w].  After every step the latents outside the mask become z0 noised to the next sigma, and z0 itself
        after the last step of the loop (num_loop_steps - 1); the next model_in and the callback see the blended
        latents."""
        use_cfg = guidance_scale > 1.0                                            # :223
        if use_cfg and (negative_prompt_embeds is None or negative_pooled is None):
            raise IHError("classifier-free guidance needs negative_prompt_embeds / negative_pooled")
        n, _, h, w = latents.shape
        L = prompt_embeds.shape[1]
        T = num_inference_steps
        loop_T = T if num_loop_steps is None else int(num_loop_steps)
        if not 0 < loop_T <= T:
            raise IHError(f"num_loop_steps {num_loop_steps} outside the {T}-step schedule")
        rescale = float(guidance_rescale or 0.0) if use_cfg else 0.0              # :352 needs CFG
        timesteps, sigmas, _ = self.tables(T)
        st = self._buffers(n, h, w, L, use_cfg)
        # inputs -> static device buffers (H2D copies when the caller hands over pinned host tensors)
        st["latents"].copy_(latents, non_blocking=True)
        neg_tid = time_ids if negative_time_ids is None else negative_time_ids
        if use_cfg:
            st["ehs"][:n].copy_(negative_prompt_embeds, non_blocking=True)    # CFG order [negative, positive], :296
            st["ehs"][n:].copy_(prompt_embeds, non_blocking=True)
            st["text_embeds"][:n].copy_(negative_pooled, non_blocking=True)
            st["text_embeds"][n:].copy_(pooled, non_blocking=True)
            st["time_ids"][:n].copy_(neg_tid, non_blocking=True)              # :298
            st["time_ids"][n:].copy_(time_ids, non_blocking=True)
        else:
            st["ehs"].copy_(prompt_embeds, non_blocking=True)
            st["text_embeds"].copy_(pooled, non_blocking=True)
            st["time_ids"].copy_(time_ids, non_blocking=True)
        if not 0 <= start_step <= loop_T:
            raise IHError(f"start_step {start_step} outside the {loop_T}-step loop")
        st["step"].fill_(start_step)
        blend = None
        if inpaint is not None:
            mask, z0, noise = inpaint
            if mask.dim() != 3 or tuple(mask.shape[1:]) != (h, w) or n % mask.shape[0] \
                    or tuple(z0.shape) != tuple(latents.shape) or tuple(noise.shape) != tuple(latents.shape):
                raise IHError(f"inpaint: mask [Bm, {h}, {w}] with {n} % Bm == 0, z0 and noise {tuple(latents.shape)} "
                              "required")
            blend = self._inpaint_buffers(n, h, w, mask.shape[0])
            blend["mask"].copy_(mask, non_blocking=True)
            blend["z0"].copy_(z0, non_blocking=True)
            blend["noise"].copy_(noise, non_blocking=True)
            blend["last"].fill_(loop_T - 1)
        self.unet.prepare_conditioning(st["ehs"], st["text_embeds"], st["time_ids"])
        ops.scale_model_input(st["latents"], st["model_in"], sigmas, st["step"], duplicate=use_cfg)   # :332-334

        steps = loop_T if stop_after is None else min(stop_after, loop_T)
        origin = start_step if count_from_start else 0                            # index of the first counted step
        n_counted = loop_T - origin

        def scale_at(i: int) -> float:
            j = i - origin
            off = (j / n_counted < control_guidance_start) or ((j + 1) / n_counted > control_guidance_end)   # :326-329
            return 0.0 if off else float(ip_scale)

        def gkey(scale: float):
            key = (n, h, w, L, T, use_cfg, float(guidance_scale), rescale, scale)
            return key if blend is None else key + ("inpaint", blend["mask"].shape[0])

        if self.use_cuda_graph:
            if self._epoch != getattr(self.unet, "graph_epoch", 0):       # weights / processors changed since capture
                self._graphs.clear()
                self._epoch = getattr(self.unet, "graph_epoch", 0)
            needed = sorted({scale_at(i) for i in range(start_step, steps)})
            captured = False
            for _ in range(4):      # a warm-up may grow a scratch buffer, which invalidates graphs captured before it
                gen = ops.workspace_generation()
                missing = [sc for sc in needed if self._graphs.get(gkey(sc), (None, -1))[1] != gen]
                if not missing:
                    break
                for sc in missing:
                    self.set_scale(sc)
                    g = self._capture(st, timesteps, sigmas, guidance_scale, use_cfg, rescale, blend)
                    self._graphs[gkey(sc)] = (g, ops.workspace_generation())
                    captured = True
            else:
                raise IHError("scratch buffers kept growing during graph capture")
            if captured:
                # the warm-up pass of a capture advances the state once: restore the initial state
                st["latents"].copy_(latents, non_blocking=True)
                st["step"].fill_(start_step)
                ops.scale_model_input(st["latents"], st["model_in"], sigmas, st["step"], duplicate=use_cfg)
        for i in range(start_step, steps):
            sc = scale_at(i)
            if self.use_cuda_graph:
                self._graphs[gkey(sc)][0].replay()
            else:
                self.set_scale(sc)
                self._step(st, timesteps, sigmas, guidance_scale, use_cfg, rescale, blend)
            if callback is not None and (i - origin) % callback_steps == 0:       # :359-363 (Euler: order 1, no warm-up)
                callback(i - origin, timesteps[i], st["latents"])
        self.set_scale(ip_scale)
        return st["latents"].clone()

    def _capture(self, st, timesteps, sigmas, guidance, use_cfg=True, rescale=0.0, blend=None):
        # warm-up on a side stream (sets kernel attributes, fills the TMA descriptor cache, sizes the allocator and
        # the library's scratch buffers)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            st["step"].zero_()
            self._step(st, timesteps, sigmas, guidance, use_cfg, rescale, blend)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        st["step"].zero_()
        g = torch.cuda.CUDAGraph()
        before = ops.launch_count()
        with torch.cuda.graph(g):
            self._step(st, timesteps, sigmas, guidance, use_cfg, rescale, blend)
        self.last_launches_per_step = ops.launch_count() - before
        self.graphs_captured += 1
        return g
