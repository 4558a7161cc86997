"""Image-to-image editing cost on one GPU, SDXL architecture with random-init weights (no checkpoints offline).

1. VAE encoder, one 1024^2 image: the native encoder (uint8 pixels in, moments out) against the oracle encoder
   (oracle/vae_encoder_ref.py) in torch eager fp32 -- what the reference runs when `force_upcast` is set, with torch's
   default math settings (cuDNN may use TF32 for fp32 convolutions) -- and in torch eager fp16.  CUDA events around each
   call, 3 warm-up calls, median of 20.  The encoder's FLOPs are computed from the shapes below.
2. IPAdapterXL.generate(image=src, strength=0.6, num_inference_steps=50) to PIL (img2img: 30 UNet steps) against the
   text-to-image edit of tools/edit_latency.py (50 steps), same pipeline weights; wall clock with a device synchronize
   on both sides, median of 3.

The card's name and power limit are read in the same run.  Usage: python tools/img2img_latency.py [--out PATH]
(default profiles/img2img_latency.json)."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from imagharmony_b200.config import HARMONY_DEFAULT as h, SDXL_BASE, SDXL_VAE, VAEConfig  # noqa: E402
from imagharmony_b200.weights import random_state_dict, shapes_of  # noqa: E402


def encoder_flops(cfg: VAEConfig, H: int, W: int) -> int:
    """Multiply-adds x 2 of the encoder + quant_conv on an H x W image (convolutions, the mid-block attention's four
    projections and its two N x N x C products); norms and elementwise work are not counted."""
    macs = 0
    conv = lambda hw, cin, cout, k: hw * cin * cout * k * k  # noqa: E731
    hw = H * W
    ch = cfg.block_out_channels
    macs += conv(hw, cfg.in_channels, ch[0], 3)
    prev = ch[0]
    for i, c in enumerate(ch):
        for j in range(cfg.layers_per_block):
            cin = prev if j == 0 else c
            macs += conv(hw, cin, c, 3) + conv(hw, c, c, 3) + (conv(hw, cin, c, 1) if cin != c else 0)
        prev = c
        if i < len(ch) - 1:
            hw //= 4
            macs += conv(hw, c, c, 3)                         # stride 2: output pixels x 9 taps
    C = ch[-1]
    macs += 2 * (2 * conv(hw, C, C, 3))                       # mid resnets
    macs += 4 * hw * C * C + 2 * hw * hw * C                  # attention projections, q k^T and P v
    L2 = 2 * cfg.latent_channels
    macs += conv(hw, C, L2, 3) + conv(hw, L2, L2, 1)
    return 2 * macs


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001 -- the figure is reported as missing, the measurement goes on
        info["power_limit_and_max_sm_clock"] = f"unavailable ({type(e).__name__})"
    return info


def time_events(fn, warmup=3, reps=20):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1], "reps": reps}


def encoder_section(out):
    from imagharmony_b200.vae import AutoencoderKLEncoder
    from oracle.vae_encoder_ref import VAEEncoderRef, preprocess_ref
    cfg = SDXL_VAE
    with torch.device("meta"):
        shapes = shapes_of(VAEEncoderRef(cfg))
    sd = random_state_dict(shapes, 21, device="cuda")
    native = AutoencoderKLEncoder.from_state_dict(cfg, sd, device="cuda")
    g = torch.Generator("cpu").manual_seed(1)
    u8 = (torch.rand(1, 1024, 1024, 3, generator=g) * 255).round().to(torch.uint8)
    u8_dev = u8.cuda()
    x32 = preprocess_ref(u8.numpy()).cuda()
    x16 = x32.half()
    flops = encoder_flops(cfg, 1024, 1024)
    res = {"image": [1024, 1024], "batch": 1, "flops": flops}
    with torch.no_grad():
        res["native"] = time_events(lambda: native.encode(u8_dev))
        for name, dt, x in (("oracle_eager_fp32", torch.float32, x32), ("oracle_eager_fp16", torch.float16, x16)):
            ref = VAEEncoderRef(cfg)
            ref.load_state_dict({k: v.float() for k, v in sd.items()})
            ref = ref.to(device="cuda", dtype=dt).eval()
            res[name] = time_events(lambda: ref.encode(x))
            del ref
            torch.cuda.empty_cache()
    for k in ("native", "oracle_eager_fp32", "oracle_eager_fp16"):
        res[k]["tflops_per_s"] = flops / (res[k]["median_ms"] * 1e-3) / 1e12
    res["speedup_vs_eager_fp32"] = res["oracle_eager_fp32"]["median_ms"] / res["native"]["median_ms"]
    res["speedup_vs_eager_fp16"] = res["oracle_eager_fp16"]["median_ms"] / res["native"]["median_ms"]
    out["encoder"] = res
    del native, sd
    torch.cuda.empty_cache()


def edit_section(out, steps=50, strength=0.6):
    from PIL import Image
    from ip_adapter import IPAdapterXL
    from ip_adapter.custom_pipelines import StableDiffusionXLCustomPipeline, StableDiffusionXLImg2ImgCustomPipeline
    from train import HarmonyAttention
    pipe = StableDiffusionXLImg2ImgCustomPipeline.from_random(SDXL_BASE, seed=0, device="cuda", vae_cfg=SDXL_VAE)
    t2i = StableDiffusionXLCustomPipeline(pipe.unet, vae=pipe.vae, scheduler=pipe.scheduler)   # same weights
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
    img = torch.randn(1, h.image_hidden_size, generator=torch.Generator("cpu").manual_seed(5)).half()
    src = Image.fromarray((torch.rand(1024, 1024, 3, generator=torch.Generator("cpu").manual_seed(6)) * 255).byte().numpy())
    kw = dict(pil_image=None, clip_image_embeds=img, prompt="lions", negative_prompt="blurry", scale=1.0, guidance_scale=5.0,
              num_samples=1, num_inference_steps=steps, extra_text="eight sheep")
    runs = {"text_to_image": (t2i, dict(height=1024, width=1024)), "img2img": (pipe, dict(image=src, strength=strength))}
    res = {"steps": steps, "strength": strength, "image": [1024, 1024]}
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
    res["img2img_over_text_to_image"] = res["img2img"]["latency_s_pil"] / res["text_to_image"]["latency_s_pil"]
    out["edit"] = res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "img2img_latency.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("img2img_latency.py measures on a GPU; none is visible")
    out = {"gpu": card(), "torch": torch.__version__,
           "tf32": {"cudnn": torch.backends.cudnn.allow_tf32, "matmul": torch.backends.cuda.matmul.allow_tf32}}
    encoder_section(out)
    edit_section(out)
    print(json.dumps(out), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
