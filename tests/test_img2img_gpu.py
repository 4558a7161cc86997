"""GPU tests of image-to-image editing through the C ABI kernels: the stride-2 conv with bottom / right padding, the
image front end, the posterior-sample + add_noise kernel, the native SDXL VAE encoder against the fp32 oracle
(oracle/vae_encoder_ref.py), and the img2img pipeline (trajectory, replay determinism, IPAdapterXL surface).

Encoder bar (SURVEY.md section 7, as tests/test_vae_gpu.py): the native fp16 encoder may not be further from the fp32
oracle than 2x the same oracle evaluated in torch-eager fp16 on the GPU, with a floor of 2e-3 * max|ref|.  The fp32
oracle runs on the GPU with TF32 disabled (a 1024^2 SDXL encode is ~5 TFLOP per image: minutes on a CPU)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture()
def no_tf32():
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.parametrize("cin,cout", [(64, 64), (128, 128), (128, 256), (256, 256), (512, 512), (256, 64)])
def test_conv_s2_padbr_kernel(cin, cout):
    """ih_conv2d_s2_padbr_f16 vs F.conv2d(F.pad(x, (0, 1, 0, 1)), stride=2) in fp32; spatial sizes leave partial tiles."""
    from imagharmony_b200 import ops
    for B, H, W in [(2, 14, 22), (1, 34, 18), (1, 96, 64)]:
        g = torch.Generator("cpu").manual_seed(cin + cout + H)
        x = torch.randn(B, H, W, cin, generator=g).half()
        w = (torch.randn(cout, cin, 3, 3, generator=g) * (9 * cin) ** -0.5).half()
        b = (torch.randn(cout, generator=g) * 0.1).half()
        o = ops.conv3x3_s2_padbr(x.cuda(), ops.pack_conv3x3_weight(w).cuda(), b.cuda()).float().cpu()
        want = F.conv2d(F.pad(x.float().permute(0, 3, 1, 2), (0, 1, 0, 1)), w.float(), b.float(), stride=2)
        want = want.permute(0, 2, 3, 1)
        assert o.shape == want.shape == (B, H // 2, W // 2, cout)
        assert torch.allclose(o, want, rtol=1e-3, atol=1e-3), ((B, H, W), (o - want).abs().max())


def test_image_front_end_is_exact():
    """uint8 NHWC -> im2col rows of fp16(2 * (v / 255) - 1): bit-identical to the torch computation."""
    from imagharmony_b200 import ops
    u8 = torch.randint(0, 256, (2, 24, 40, 3), generator=torch.Generator().manual_seed(0), dtype=torch.uint8)
    u8[0, 0, :4] = torch.tensor([[0, 255, 127], [128, 1, 254], [64, 191, 3], [255, 255, 0]], dtype=torch.uint8)
    got = ops.image_im2col3x3(u8.cuda(), 32).cpu()
    x = (2.0 * (torch.from_numpy(u8.numpy().astype(np.float32) / 255.0)) - 1.0).half().float().permute(0, 3, 1, 2)
    want = F.pad(F.unfold(x, kernel_size=3, padding=1).transpose(1, 2).reshape(2 * 24 * 40, 27), (0, 5)).half()
    assert got.dtype == torch.float16 and torch.equal(got, want)


def _restate(moments, eps, noise, C, sf, sigma):
    """The fp16 torch restatement of diffusers' rounding points (sample fp32 -> fp16 -> * sf in fp16 -> add_noise)."""
    from oracle.img2img_ref import add_noise_ref
    from oracle.vae_encoder_ref import posterior_sample_ref
    B = noise.shape[0]
    idx = torch.arange(B, device=moments.device)
    m = moments.float().permute(0, 3, 1, 2)[idx % moments.shape[0]]
    z = m[:, :C].half() if eps is None else sf * posterior_sample_ref(m[:, :2 * C], eps[idx % eps.shape[0]]).half()
    return add_noise_ref(z, noise, sigma)


def test_posterior_add_noise_kernel_bit_exact():
    from imagharmony_b200 import ops
    g = torch.Generator("cpu").manual_seed(1)
    Bm, h, w, C = 2, 12, 20, 4
    mom = torch.zeros(Bm, h, w, 16)
    mom[..., :C] = torch.randn(Bm, h, w, C, generator=g) * 20
    mom[..., C:2 * C] = torch.randn(Bm, h, w, C, generator=g) * 12 - 4       # reaches beyond the clamp at -30 / 20
    mom[0, 0, 0, C:2 * C] = torch.tensor([-45.0, 27.0, 20.5, -30.5])
    mom = mom.half().cuda()
    assert mom[..., C:2 * C].min() < -30 and mom[..., C:2 * C].max() > 20
    for B, Be in [(2, 2), (4, 2), (4, 4), (6, 2)]:
        eps = torch.randn(Be, C, h, w, generator=g).cuda()
        noise = torch.randn(B, C, h, w, generator=g).half().cuda()
        for sigma in (14.614642, 0.6986, 0.0292):
            got = ops.vae_sample_add_noise(mom, eps, noise, C, 0.13025, sigma)
            want = _restate(mom, eps, noise, C, 0.13025, sigma)
            assert got.dtype == torch.float16 and torch.equal(got, want), (B, Be, sigma)
    lat = torch.randn(1, h, w, C, generator=g).half().cuda()                 # latents given as they are (no posterior)
    noise = torch.randn(3, C, h, w, generator=g).half().cuda()
    assert torch.equal(ops.vae_sample_add_noise(lat, None, noise, C, 1.0, 3.5), _restate(lat, None, noise, C, 1.0, 3.5))


def _enc_models(cfg, seed, scale_conv_in=1.0):
    """(native encoder, fp32 oracle on the GPU, fp16 eager oracle on the GPU) with identical fp16-representable weights."""
    from imagharmony_b200.vae import AutoencoderKLEncoder
    from imagharmony_b200.weights import random_state_dict, shapes_of
    from oracle.vae_encoder_ref import VAEEncoderRef
    with torch.device("meta"):
        shapes = shapes_of(VAEEncoderRef(cfg))
    sd = {k: v.float() for k, v in random_state_dict(shapes, seed).items()}
    for k in ("encoder.conv_in.weight", "encoder.conv_in.bias"):
        sd[k] = (sd[k] * scale_conv_in).half().float()
    native = AutoencoderKLEncoder.from_state_dict(cfg, sd, device="cuda")
    ref32 = VAEEncoderRef(cfg)
    ref32.load_state_dict(sd)
    eager16 = VAEEncoderRef(cfg)
    eager16.load_state_dict(sd)
    return native, ref32.cuda().eval(), eager16.half().cuda().eval()


def _smooth_u8(B, H, W, seed):
    g = torch.Generator("cpu").manual_seed(seed)
    x = F.interpolate(torch.rand(B, 3, H // 32, W // 32, generator=g), size=(H, W), mode="bilinear", align_corners=False)
    x = x + 0.1 * torch.rand(B, 3, H, W, generator=g)
    return (x.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def _bar(tag, o, r, e):
    o, r, e = o.float().cpu(), r.float().cpu(), e.float().cpu()
    e_nat, e_eag, mx = (o - r).abs().max().item(), (e - r).abs().max().item(), r.abs().max().item()
    print(f"[{tag}] native max|err| {e_nat:.3e}  eager-fp16 {e_eag:.3e}  max|ref| {mx:.3e}")
    assert torch.isfinite(o).all()
    assert e_nat <= max(2.0 * e_eag, 2e-3 * mx), (e_nat, e_eag, mx)


@pytest.mark.parametrize("B", [1, 2])
def test_sdxl_encoder_1024_matches_oracle(no_tf32, B):
    """The full SDXL VAE encoder (34 M parameters) on 1024^2 pixels, from the uint8 PIL pixels."""
    from imagharmony_b200.config import SDXL_VAE
    from oracle.vae_encoder_ref import preprocess_ref
    native, ref32, eager16 = _enc_models(SDXL_VAE, seed=21)
    u8 = _smooth_u8(B, 1024, 1024, seed=B)
    x = preprocess_ref(u8.numpy()).cuda()
    with torch.no_grad():
        r = ref32.encode(x)
        e = eager16.encode(x.half())
        o = native.encode(u8.cuda())
    torch.cuda.synchronize()
    assert o.shape == (B, 128, 128, 16)
    _bar(f"SDXL encoder 1024^2 B{B}", o[..., :8].permute(0, 3, 1, 2), r, e)


def test_encoder_scaled_stream_survives_fp16_overflow(no_tf32):
    """A model whose residual stream exceeds 6.5e4 (conv_in scaled up): the scaled stream (2^-7) stays finite and matches
    the fp32 oracle."""
    from imagharmony_b200.config import TINY_VAE as cfg
    native, ref32, _ = _enc_models(cfg, seed=22, scale_conv_in=50000.0)
    assert native.stream_scale == 2.0 ** -7
    x = torch.rand(2, 3, 64, 64, generator=torch.Generator("cpu").manual_seed(3)) * 2 - 1
    x = x.half().float().cuda()
    with torch.no_grad():
        r = ref32.encode(x)
        stream = ref32.encoder.conv_in(x)
        o = native.encode(x)[..., :8].permute(0, 3, 1, 2).float()
    torch.cuda.synchronize()
    assert stream.abs().max() > 65504, "the test model must overflow fp16"
    err, mx = (o - r).abs().max().item(), r.abs().max().item()
    print(f"[encoder scaled stream] stream max {stream.abs().max().item():.3e}: max|err| {err:.3e} (max|ref| {mx:.3e})")
    assert torch.isfinite(o).all() and err <= 1e-2 * mx, (err, mx)


def test_sdxl_tiled_encode_1280x1024(no_tf32):
    """enable_vae_tiling(): 1024-pixel tiles every 768 pixels of a 1024 x 1280 image (ragged 256 / 512 edge tiles)."""
    from imagharmony_b200.config import SDXL_VAE
    from oracle.vae_encoder_ref import preprocess_ref, tiled_encode_ref
    native, ref32, eager16 = _enc_models(SDXL_VAE, seed=23)
    native.use_tiling = True
    u8 = _smooth_u8(1, 1024, 1280, seed=5)
    x = preprocess_ref(u8.numpy()).cuda()
    with torch.no_grad():
        r = tiled_encode_ref(ref32, x)
        e = tiled_encode_ref(eager16, x.half())
        o = native.encode(u8.cuda())
    torch.cuda.synchronize()
    assert o.shape == (1, 128, 160, 16) and r.shape == (1, 8, 128, 160)
    _bar("SDXL tiled encode 1024x1280", o[..., :8].permute(0, 3, 1, 2), r, e)


def _tiny_pipe(seed=0):
    """The img2img pipeline on the SDXL-shaped miniature UNet and VAE (random weights, IP processors loaded), and the
    UNet / processor state dicts it was built from (for the oracle)."""
    from imagharmony_b200.config import TINY, TINY_VAE
    from imagharmony_b200.unet import UNet2DConditionModel
    from imagharmony_b200.weights import random_state_dict, shapes_of
    from ip_adapter.custom_pipelines import StableDiffusionXLImg2ImgCustomPipeline
    pipe = StableDiffusionXLImg2ImgCustomPipeline.from_random(TINY, seed=seed, device="cuda", vae_cfg=TINY_VAE)
    procs = torch.nn.ModuleList(pipe.unet.attn_processors.values())
    ip_sd = random_state_dict(shapes_of(procs), seed + 1)
    procs.load_state_dict({k: v.cuda() for k, v in ip_sd.items()})
    pipe.unet.finalize()
    with torch.device("meta"):
        shapes = shapes_of(UNet2DConditionModel(TINY))
    sd = random_state_dict(shapes, seed, device="cuda")                # what from_random drew
    return pipe, {k: v.float().cpu() for k, v in sd.items()}, {k: v.float() for k, v in ip_sd.items()}


def test_img2img_trajectory_512_matches_oracle():
    """512^2 source image, 4 steps at strength 0.6 (2 executed) on the SDXL-shaped miniature UNet: native CUDA-graph loop
    vs the CPU fp32 oracle loop and the eager-fp16 one on the same noised latents; the pipeline result equals
    engine.run(start_step=t_start) on those latents bit for bit, and two replayed calls are bit-identical."""
    from PIL import Image
    from imagharmony_b200.config import TINY
    from oracle import adapter_ref as A
    from oracle.img2img_ref import img2img_denoise_loop
    from oracle.unet_ref import UNetRef
    pipe, sd, ip_sd = _tiny_pipe()
    T, strength = 4, 0.6
    t_start, n_exec = pipe.get_timesteps(T, strength)
    assert (t_start, n_exec) == (2, 2)
    src = Image.fromarray(_smooth_u8(1, 512, 512, seed=7)[0].numpy())
    g = torch.Generator("cpu").manual_seed(11)
    emb = dict(prompt_embeds=torch.randn(1, 81, TINY.cross_attention_dim, generator=g).half(),
               negative_prompt_embeds=torch.randn(1, 81, TINY.cross_attention_dim, generator=g).half(),
               pooled_prompt_embeds=torch.randn(1, TINY.pooled_embed_dim, generator=g).half(),
               negative_pooled_prompt_embeds=torch.randn(1, TINY.pooled_embed_dim, generator=g).half())
    calls = []
    run = lambda: pipe(image=src, strength=strength, num_inference_steps=T, output_type="latent",  # noqa: E731
                       generator=torch.Generator("cuda").manual_seed(5), callback=lambda i, t, x: calls.append(i),
                       **emb).images
    o1 = run()
    o2 = run()
    torch.cuda.synchronize()
    assert calls == [0, 1, 0, 1] and torch.equal(o1, o2)
    pipe.scheduler.set_timesteps(T)
    lat, _ = pipe.prepare_img2img_latents(src, 1, torch.Generator("cuda").manual_seed(5), float(pipe.scheduler.sigmas[t_start]))
    tid = torch.tensor([[512.0, 512.0, 0.0, 0.0, 512.0, 512.0]])
    direct = pipe.engine.run(lat, emb["prompt_embeds"], emb["negative_prompt_embeds"], emb["pooled_prompt_embeds"],
                             emb["negative_pooled_prompt_embeds"], tid, T, start_step=t_start, count_from_start=True)
    assert torch.equal(direct, o1)

    def oracle(device, dtype):
        m = UNetRef(TINY)
        m.load_state_dict(sd)
        pr = A.install_processors(m, TINY, dtype=torch.float32)
        torch.nn.ModuleList(pr.values()).load_state_dict(ip_sd)
        return m.to(device=device, dtype=dtype).eval()

    def run_oracle(m, dev, dt):
        fn = lambda s_, t_, e_, te_, ti_: m(s_.to(dt), t_, e_, te_, ti_).to(torch.float16)  # noqa: E731
        return img2img_denoise_loop(fn, lat.to(dev), emb["prompt_embeds"].to(dev, dt),
                                    emb["negative_prompt_embeds"].to(dev, dt), emb["pooled_prompt_embeds"].to(dev, dt),
                                    emb["negative_pooled_prompt_embeds"].to(dev, dt), tid.to(dev), T, strength)
    r = run_oracle(oracle("cpu", torch.float32), "cpu", torch.float32)
    e = run_oracle(oracle("cuda", torch.float16), "cuda", torch.float16)
    _bar("img2img trajectory 512^2 strength 0.6", o1, r, e)


def test_ip_adapter_generate_img2img_on_gpu():
    """IPAdapterXL.generate(image=src, strength=...) returns PIL images and runs T - t_start steps (callback count)."""
    from PIL import Image
    from imagharmony_b200.config import HARMONY_TINY as h
    from ip_adapter import IPAdapterXL
    from train import HarmonyAttention
    pipe, _, _ = _tiny_pipe(seed=3)
    ha = HarmonyAttention(image_hidden_size=h.image_hidden_size, text_context_dim=h.text_context_dim,
                          inter_dim=h.inter_dim, cross_heads=h.cross_heads, reshape_blocks=h.reshape_blocks,
                          cross_value_dim=h.cross_value_dim, scale=1.0, fusion_method="cross_attention")
    ip = IPAdapterXL(pipe, None, None, "cuda", num_tokens=4, inference=True, number_class_crossattention=ha)
    src = Image.fromarray(_smooth_u8(1, 256, 384, seed=9)[0].numpy())
    calls = []
    pil = ip.generate(pil_image=None, clip_image_embeds=torch.randn(1, h.image_hidden_size), image=src, strength=0.6,
                      prompt="lions", num_samples=2, num_inference_steps=10, seed=[3, 4], extra_text="eight sheep",
                      callback=lambda i, t, x: calls.append(i))
    assert isinstance(pil, list) and len(pil) == 2 and pil[0].size == (384, 256) and pil[0].mode == "RGB"
    assert calls == list(range(6))
