"""Masked inpainting cost on one GPU, SDXL architecture with random-init weights (no checkpoints offline).

1. IPAdapterXL.generate(image=src, mask_image=mask, num_inference_steps=50) to PIL at 1024^2: inpainting at the default
   strength 0.9999 (49 UNet steps) and at strength 0.6 (30 steps), against the img2img edit at strength 0.6 (30 steps),
   same pipeline weights; wall clock with a device synchronize on both sides, median of 3 after one warm-up call.
2. The graph-replayed denoising step (CFG, batch 1, 128^2 latents) with and without the mask blend: the two captured
   graphs are replayed alternately, 10 rounds of 20 replays each, CUDA events around each window; per-step medians.

The card's name and power limit are read in the same run.  Usage: python tools/inpaint_latency.py [--out PATH]
(default profiles/inpaint_latency.json)."""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from img2img_latency import card  # noqa: E402
from imagharmony_b200.config import HARMONY_DEFAULT as h, SDXL_BASE, SDXL_VAE  # noqa: E402
from imagharmony_b200.weights import random_state_dict, shapes_of  # noqa: E402


def build():
    from ip_adapter import IPAdapterXL
    from ip_adapter.custom_pipelines import StableDiffusionXLInpaintCustomPipeline
    from train import HarmonyAttention
    pipe = StableDiffusionXLInpaintCustomPipeline.from_random(SDXL_BASE, seed=0, device="cuda", vae_cfg=SDXL_VAE)
    ha = HarmonyAttention(image_hidden_size=h.image_hidden_size, text_context_dim=h.text_context_dim, inter_dim=h.inter_dim,
                          cross_heads=h.cross_heads, reshape_blocks=h.reshape_blocks, cross_value_dim=h.cross_value_dim,
                          scale=1.0, fusion_method="cross_attention")
    ip = IPAdapterXL(pipe, None, None, "cuda", num_tokens=4, target_blocks=["down_blocks.2.attentions.1"], inference=True,
                     number_class_crossattention=ha)
    ip.image_proj_model.load_state_dict({k: v.cuda() for k, v in random_state_dict(shapes_of(ip.image_proj_model), 3).items()})
    ip.number_class_crossattention.load_state_dict({k: v.cuda() for k, v in random_state_dict(shapes_of(ha), 4).items()})
    procs = torch.nn.ModuleList(pipe.unet.attn_processors.values())
    procs.load_state_dict({k: v.cuda() for k, v in random_state_dict(shapes_of(procs), 5).items()})
    pipe.unet.finalize()
    return pipe, ip


def edit_section(out, pipe, ip, steps=50):
    from PIL import Image
    from ip_adapter.custom_pipelines import StableDiffusionXLImg2ImgCustomPipeline
    img = torch.randn(1, h.image_hidden_size, generator=torch.Generator("cpu").manual_seed(5)).half()
    src = Image.fromarray((torch.rand(1024, 1024, 3, generator=torch.Generator("cpu").manual_seed(6)) * 255).byte().numpy())
    mask = Image.new("L", (1024, 1024), 0)
    mask.paste(255, (256, 384, 768, 896))
    kw = dict(pil_image=None, clip_image_embeds=img, prompt="lions", negative_prompt="blurry", scale=1.0, guidance_scale=5.0,
              num_samples=1, num_inference_steps=steps, extra_text="eight sheep", image=src)
    img2img = StableDiffusionXLImg2ImgCustomPipeline(pipe.unet, vae=pipe.vae, scheduler=pipe.scheduler,
                                                     vae_encoder=pipe.vae_encoder)            # same weights
    runs = {"inpaint_default_strength": (pipe, dict(mask_image=mask)),
            "inpaint_strength_0.6": (pipe, dict(mask_image=mask, strength=0.6)),
            "img2img_strength_0.6": (img2img, dict(strength=0.6))}
    res = {"steps": steps, "image": [1024, 1024], "mask_box_xyxy": [256, 384, 768, 896]}
    for name, (p, extra) in runs.items():
        ip.pipe = p
        counted = []
        pil = ip.generate(seed=[1], callback=lambda i, t, x: counted.append(i), **kw, **extra)   # warm-up: graphs
        ts = []
        for s in (2, 3, 4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ip.generate(seed=[s], **kw, **extra)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        res[name] = {"latency_s_pil": sorted(ts)[1], "all_s": ts, "unet_steps": len(counted),
                     "pil": [list(pil[0].size), pil[0].mode]}
    ip.pipe = pipe
    out["edit"] = res


def step_section(out, pipe, rounds=10, reps=20):
    """Replays the two captured step graphs (the plain one and the masked one) alternately."""
    eng = pipe.engine
    g = torch.Generator("cpu").manual_seed(7)
    n, lat, T = 1, 128, 50
    latents = torch.randn(n, 4, lat, lat, generator=g).half()
    ehs = torch.randn(n, 77 + pipe.unet.config.num_ip_tokens, pipe.unet.config.cross_attention_dim, generator=g).half()
    pooled = torch.randn(n, pipe.unet.config.pooled_embed_dim, generator=g).half()
    tid = torch.tensor([[1024.0, 1024.0, 0.0, 0.0, 1024.0, 1024.0]])
    mask = torch.zeros(1, lat, lat, dtype=torch.uint8)
    mask[:, 48:112, 32:96] = 1
    inpaint = (mask, torch.randn(n, 4, lat, lat, generator=g).half(), torch.randn(n, 4, lat, lat, generator=g).half())
    launches = {}
    for name, extra in (("plain", {}), ("masked", {"inpaint": inpaint})):
        eng.run(latents, ehs, torch.zeros_like(ehs), pooled, torch.zeros_like(pooled), tid, T, stop_after=1, **extra)
        launches[name] = eng.last_launches_per_step
    torch.cuda.synchronize()
    plain_key = (n, lat, lat, ehs.shape[1], T, True, 5.0, 0.0, 1.0)       # DenoiseEngine.run's graph key (gkey)
    key_of = {"plain": plain_key, "masked": plain_key + ("inpaint", 1)}
    st = eng._static[(n, lat, lat, ehs.shape[1], True)]
    times = {"plain": [], "masked": []}
    for r in range(rounds + 1):                                  # round 0 is a warm-up
        for name in ("plain", "masked") if r % 2 else ("masked", "plain"):
            graph = eng._graphs[key_of[name]][0]
            st["step"].fill_(5)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                graph.replay()
            b.record()
            b.synchronize()
            if r:
                times[name].append(a.elapsed_time(b) / reps)
    res = {"batch": n, "latent": [lat, lat], "cfg": True, "rounds": rounds, "replays_per_round": reps,
           "launches_per_step": launches}
    for name, ts in times.items():
        ts = sorted(ts)
        res[name] = {"median_ms_per_step": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1]}
    res["masked_minus_plain_ms"] = res["masked"]["median_ms_per_step"] - res["plain"]["median_ms_per_step"]
    out["step"] = res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "inpaint_latency.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("inpaint_latency.py measures on a GPU; none is visible")
    out = {"gpu": card(), "torch": torch.__version__}
    pipe, ip = build()
    edit_section(out, pipe, ip)
    step_section(out, pipe)
    print(json.dumps(out), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
