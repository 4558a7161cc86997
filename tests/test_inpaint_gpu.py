"""GPU tests of masked inpainting through the C ABI kernels: the masked Euler step (all three step variants) and the
inpainting front end bit for bit against fp16 torch restatements, the 512^2 inpainting trajectory against the fp32 and
eager-fp16 oracles (oracle/inpaint_ref.py), the all-zero / all-one mask invariants, graph replay, and the IPAdapterXL
surface."""
import numpy as np
import pytest
import torch

from test_img2img_gpu import _bar, _smooth_u8, _tiny_pipe

pytestmark = pytest.mark.gpu


def _bits(x):
    return x.contiguous().view(torch.int16)


def _inpaint_pipe(seed=0):
    from ip_adapter.custom_pipelines import StableDiffusionXLInpaintCustomPipeline
    p, sd, ip_sd = _tiny_pipe(seed)
    return (StableDiffusionXLInpaintCustomPipeline(p.unet, vae=p.vae, scheduler=p.scheduler, vae_encoder=p.vae_encoder),
            sd, ip_sd)


@pytest.mark.parametrize("variant", ["cfg", "no_cfg", "rescale"])
@pytest.mark.parametrize("n", [1, 2, 4])
def test_masked_step_bit_exact(variant, n):
    """ih_euler_step_inpaint == the plain step (ih_euler_cfg_step / ih_euler_step_ex) followed by the blend restated in
    fp16 torch, at 1024^2 latents, Bm in {1, n}, on an intermediate step, on the schedule's last step and on a last
    step cut short (sigma[k + 1] != 0).  Compared bit for bit, so the sign of zero counts: where the mask keeps z0 = -0,
    the last step gives -0 (with a negative update) where add_noise at sigma 0 would give -0 + 0 = +0."""
    from imagharmony_b200 import ops
    from imagharmony_b200.scheduler import EulerDiscreteScheduler
    from oracle.img2img_ref import add_noise_ref
    use_cfg, rescale = variant != "no_cfg", (0.7 if variant == "rescale" else 0.0)
    T, h, w = 50, 128, 128
    s = EulerDiscreteScheduler().set_timesteps(T)
    sigmas = torch.from_numpy(s.sigmas).cuda()
    g = torch.Generator("cpu").manual_seed(n)
    b = 2 * n if use_cfg else n
    pred = torch.randn(b, 4, h, w, generator=g).half().cuda()
    lat0 = (torch.randn(n, 4, h, w, generator=g) * 4).half().cuda()
    z0 = torch.randn(n, 4, h, w, generator=g).half()
    noise = torch.randn(n, 4, h, w, generator=g).half()
    z0[:, :, :4] = -0.0                                                   # -0 where the mask keeps the source
    noise[:, :, :4] = noise[:, :, :4].abs()
    z0, noise = z0.cuda(), noise.cuda()
    for Bm in sorted({1, n}):
        mask = (torch.rand(Bm, h, w, generator=g) < 0.5).to(torch.uint8)
        mask[:, :4] = 0
        mask = mask.cuda()
        m = mask[torch.arange(n) % Bm][:, None].half()
        for k, last in ((20, 49), (49, 49), (30, 30)):
            step = torch.tensor([k], dtype=torch.int32, device="cuda")
            lat, mi = lat0.clone(), torch.empty_like(pred)
            ops.euler_step_inpaint(pred, lat, mi, sigmas, step, 5.0, mask, z0, noise,
                                   torch.tensor([last], dtype=torch.int32, device="cuda"), use_cfg=use_cfg,
                                   guidance_rescale=rescale)
            ref_lat, ref_mi = lat0.clone(), torch.empty_like(pred)
            ref_step = torch.tensor([k], dtype=torch.int32, device="cuda")
            ops.euler_step(pred, ref_lat, ref_mi, sigmas, ref_step, 5.0, use_cfg=use_cfg, guidance_rescale=rescale)
            proper = z0 if k == last else add_noise_ref(z0, noise, float(sigmas[k + 1]))
            ref_lat = (1 - m) * proper + m * ref_lat
            ops.scale_model_input(ref_lat, ref_mi, sigmas, ref_step, duplicate=use_cfg)   # model_in at sigma[k + 1]
            torch.cuda.synchronize()
            assert int(step.item()) == k + 1
            assert torch.equal(_bits(lat), _bits(ref_lat)), (variant, n, Bm, k)
            assert torch.equal(_bits(mi), _bits(ref_mi)), (variant, n, Bm, k)
            negz = (_bits(ref_lat) == -32768).sum().item()
            assert (negz > 0) == (k == last), (k, last, negz)


def test_front_end_bit_exact():
    """ih_latent_mask_u8 against numpy, ih_vae_sample_inpaint_f16 (z0, noised start, pure-noise start) against the fp16
    torch restatement; z0 equals the img2img kernel's output with sigma 0 except in the sign of zero."""
    from imagharmony_b200 import ops
    from oracle.img2img_ref import add_noise_ref
    from oracle.vae_encoder_ref import posterior_sample_ref
    g = torch.Generator("cpu").manual_seed(3)
    u8 = torch.randint(0, 256, (3, 48, 80), generator=g, dtype=torch.uint8)
    u8[0, 0, :16] = torch.tensor([127, 0, 0, 0, 0, 0, 0, 0, 128, 0, 0, 0, 0, 0, 0, 0], dtype=torch.uint8)
    got = ops.latent_mask(u8.cuda()).cpu()
    assert got.dtype == torch.uint8 and got.shape == (3, 6, 10)
    assert np.array_equal(got.numpy(), (u8.numpy()[:, ::8, ::8] >= 128).astype(np.uint8))
    assert got[0, 0, :2].tolist() == [0, 1]
    C, h, w = 4, 12, 20
    mom = torch.zeros(2, h, w, 16)
    mom[..., :C] = torch.randn(2, h, w, C, generator=g) * 20
    mom[..., C:2 * C] = torch.randn(2, h, w, C, generator=g) * 12 - 4
    mom[0, 0, 0, :C] = -0.0
    mom[0, 0, 0, C:2 * C] = -30.0
    mom = mom.half().cuda()
    eps = torch.randn(2, C, h, w, generator=g).cuda()
    eps[0, :, 0, 0] = -0.0                                                # mean -0 + std * -0 = -0
    for B in (2, 4):
        noise = torch.randn(B, C, h, w, generator=g).half().cuda()
        idx = torch.arange(B, device="cuda")
        m = mom.float().permute(0, 3, 1, 2)[idx % 2]
        z = 0.13025 * posterior_sample_ref(m[:, :2 * C], eps[idx % 2]).half()
        for sigma, pure in ((3.7, False), (14.6146, True)):
            lat, z0 = ops.vae_sample_inpaint(mom, eps, noise, C, 0.13025, sigma, pure)
            want = (noise.float() * torch.tensor(sigma, dtype=torch.float32)).half() if pure else add_noise_ref(z, noise, sigma)
            assert torch.equal(_bits(z0), _bits(z)) and torch.equal(_bits(lat), _bits(want)), (B, sigma)
        assert (_bits(z0) == -32768).any()
        via_sigma0 = ops.vae_sample_add_noise(mom, eps, noise.abs(), C, 0.13025, 0.0)
        assert torch.equal(via_sigma0, z0) and not torch.equal(_bits(via_sigma0), _bits(z0))


def _emb():
    from imagharmony_b200.config import TINY
    g = torch.Generator("cpu").manual_seed(11)
    return dict(prompt_embeds=torch.randn(1, 81, TINY.cross_attention_dim, generator=g).half(),
                negative_prompt_embeds=torch.randn(1, 81, TINY.cross_attention_dim, generator=g).half(),
                pooled_prompt_embeds=torch.randn(1, TINY.pooled_embed_dim, generator=g).half(),
                negative_pooled_prompt_embeds=torch.randn(1, TINY.pooled_embed_dim, generator=g).half())


def _mask(size=512):
    from PIL import Image
    m = Image.new("L", (size, size), 0)
    m.paste(255, (size // 4, size // 8, 3 * size // 4, size // 2))
    return m


@pytest.mark.parametrize("strength", [0.6, 1.0])
def test_inpaint_trajectory_512_matches_oracle(strength):
    """512^2, 4 steps on the SDXL-shaped miniature UNet: the native CUDA-graph loop against the CPU fp32 oracle loop and
    the eager-fp16 one from the same start latents, mask, z0 and noise; outside the mask the result is z0 exactly."""
    from PIL import Image
    from imagharmony_b200.config import TINY
    from oracle import adapter_ref as A
    from oracle.inpaint_ref import inpaint_denoise_loop
    from oracle.unet_ref import UNetRef
    pipe, sd, ip_sd = _inpaint_pipe()
    T = 4
    src = Image.fromarray(_smooth_u8(1, 512, 512, seed=7)[0].numpy())
    emb = _emb()
    o = pipe(image=src, mask_image=_mask(), strength=strength, num_inference_steps=T, height=512, width=512,
             output_type="latent", generator=torch.Generator("cuda").manual_seed(5), **emb).images
    pipe.scheduler.set_timesteps(T)
    t_start, _ = pipe.get_timesteps(T, strength)
    lat, (mask, z0, noise) = pipe.prepare_inpaint_latents(src, _mask(), 1, torch.Generator("cuda").manual_seed(5), 512,
                                                          512, t_start, strength == 1.0)
    torch.cuda.synchronize()
    keep = (mask == 0)[:, None].expand_as(o)
    assert keep.any() and (~keep).any() and torch.equal(o[keep], z0[keep])
    tid = torch.tensor([[512.0, 512.0, 0.0, 0.0, 512.0, 512.0]])
    mask16 = mask[:, None].half()

    def oracle(device, dtype):
        m = UNetRef(TINY)
        m.load_state_dict(sd)
        pr = A.install_processors(m, TINY, dtype=torch.float32)
        torch.nn.ModuleList(pr.values()).load_state_dict(ip_sd)
        return m.to(device=device, dtype=dtype).eval()

    def run_oracle(m, dev, dt):
        fn = lambda s_, t_, e_, te_, ti_: m(s_.to(dt), t_, e_, te_, ti_).to(torch.float16)  # noqa: E731
        return inpaint_denoise_loop(fn, lat.to(dev), emb["prompt_embeds"].to(dev, dt),
                                    emb["negative_prompt_embeds"].to(dev, dt), emb["pooled_prompt_embeds"].to(dev, dt),
                                    emb["negative_pooled_prompt_embeds"].to(dev, dt), tid.to(dev), T, strength,
                                    mask16.to(dev), z0.to(dev), noise.to(dev))
    r = run_oracle(oracle("cpu", torch.float32), "cpu", torch.float32)
    e = run_oracle(oracle("cuda", torch.float16), "cuda", torch.float16)
    _bar(f"inpaint trajectory 512^2 strength {strength}", o, r, e)


def test_mask_invariants():
    """An all-zero mask returns z0; an all-one mask at strength < 1 with one generator is the img2img result."""
    from PIL import Image
    from ip_adapter.custom_pipelines import StableDiffusionXLImg2ImgCustomPipeline
    pipe, _, _ = _inpaint_pipe(seed=1)
    src = Image.fromarray(_smooth_u8(1, 256, 256, seed=8)[0].numpy())
    emb = _emb()
    kw = dict(image=src, strength=0.7, num_inference_steps=6, output_type="latent", **emb)
    zero = pipe(mask_image=Image.new("L", (256, 256), 0), height=256, width=256,
                generator=torch.Generator("cuda").manual_seed(2), **kw).images
    pipe.scheduler.set_timesteps(6)
    _, (_, z0, _) = pipe.prepare_inpaint_latents(src, Image.new("L", (256, 256), 0), 1,
                                                 torch.Generator("cuda").manual_seed(2), 256, 256, 2, False)
    one = pipe(mask_image=Image.new("L", (256, 256), 255), height=256, width=256,
               generator=torch.Generator("cuda").manual_seed(2), **kw).images
    i2i = StableDiffusionXLImg2ImgCustomPipeline.__call__(pipe, generator=torch.Generator("cuda").manual_seed(2), **kw).images
    torch.cuda.synchronize()
    assert torch.equal(zero, z0)
    assert torch.equal(one, i2i)


def test_graph_replay_and_launch_count():
    """Two replayed calls are bit-identical, and a masked step launches as many kernels as a text-to-image step."""
    from PIL import Image
    from ip_adapter.custom_pipelines import StableDiffusionXLCustomPipeline
    pipe, _, _ = _inpaint_pipe(seed=2)
    emb = _emb()
    t2i = StableDiffusionXLCustomPipeline(pipe.unet, vae=pipe.vae, scheduler=pipe.scheduler)
    t2i(height=256, width=256, num_inference_steps=3, output_type="latent", **emb)
    plain = t2i.engine.last_launches_per_step
    src = Image.fromarray(_smooth_u8(1, 256, 256, seed=9)[0].numpy())
    calls = []
    run = lambda: pipe(image=src, mask_image=_mask(256), height=256, width=256, num_inference_steps=5,  # noqa: E731
                       output_type="latent", generator=torch.Generator("cuda").manual_seed(4),
                       callback=lambda i, t, x: calls.append(i), **emb).images
    o1 = run()
    masked = pipe.engine.last_launches_per_step
    o2 = run()
    torch.cuda.synchronize()
    assert torch.equal(_bits(o1), _bits(o2)) and calls == [0, 1, 2, 3] * 2      # strength 0.9999: 4 of 5 steps
    assert plain > 0 and masked == plain, (plain, masked)


def test_ip_adapter_generate_inpaint_on_gpu():
    from PIL import Image
    from imagharmony_b200.config import HARMONY_TINY as h
    from ip_adapter import IPAdapterXL
    from train import HarmonyAttention
    pipe, _, _ = _inpaint_pipe(seed=3)
    ha = HarmonyAttention(image_hidden_size=h.image_hidden_size, text_context_dim=h.text_context_dim,
                          inter_dim=h.inter_dim, cross_heads=h.cross_heads, reshape_blocks=h.reshape_blocks,
                          cross_value_dim=h.cross_value_dim, scale=1.0, fusion_method="cross_attention")
    ip = IPAdapterXL(pipe, None, None, "cuda", num_tokens=4, inference=True, number_class_crossattention=ha)
    src = Image.fromarray(_smooth_u8(1, 256, 384, seed=9)[0].numpy())
    calls = []
    pil = ip.generate(pil_image=None, clip_image_embeds=torch.randn(1, h.image_hidden_size), image=src,
                      mask_image=_mask(256), prompt="lions", num_samples=2, num_inference_steps=10, seed=[3, 4],
                      extra_text="eight sheep", height=256, width=384, callback=lambda i, t, x: calls.append(i))
    assert isinstance(pil, list) and len(pil) == 2 and pil[0].size == (384, 256) and pil[0].mode == "RGB"
    assert calls == list(range(9))                   # default strength 0.9999: 9 of 10 steps
