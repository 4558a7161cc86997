"""CPU tests of image-to-image editing: the native VAE encoder's wiring (key names, scaled residual stream, folded
quant_conv, tiled encode), the img2img schedule arithmetic, the generator draw order of the initial latents and the
truncated denoise trajectory, against the fp32 oracle with stand-in ops (no kernels involved; those are
tests/test_img2img_gpu.py)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_wiring_cpu import _build, _Empty32, _fp32_engine, _inputs, patched  # noqa: F401  (fixture)


def _conv3x3_s2_padbr(x, w_packed, bias=None, *, out=None):
    B, H, W, Cin = x.shape
    w = w_packed.reshape(w_packed.shape[0], 3, 3, Cin).permute(0, 3, 1, 2).float()
    y = F.conv2d(F.pad(x.float().permute(0, 3, 1, 2), (0, 1, 0, 1)), w, None if bias is None else bias.float(), stride=2)
    return y.permute(0, 2, 3, 1).to(x.dtype).contiguous()


def _image_im2col3x3(rgb_u8, kpad=32, out=None):
    """fp16-rounded 2 v / 255 - 1 as the kernel computes it, kept in fp32 (the wiring tests run in fp32)."""
    x = (2.0 * (rgb_u8.float() / 255.0) - 1.0).half().float().permute(0, 3, 1, 2)
    B, C, H, W = x.shape
    a = F.unfold(x, kernel_size=3, padding=1).transpose(1, 2).reshape(B * H * W, C * 9)
    return F.pad(a, (0, kpad - C * 9))


def _vae_sample_add_noise(moments, eps, noise, channels, scaling_factor, sigma, out=None):
    from oracle.img2img_ref import add_noise_ref
    from oracle.vae_encoder_ref import posterior_sample_ref
    B, C = noise.shape[0], channels
    m = moments.float().permute(0, 3, 1, 2)[torch.arange(B) % moments.shape[0]]
    if eps is None:
        z = m[:, :C].half()
    else:
        z = scaling_factor * posterior_sample_ref(m[:, :2 * C], eps[torch.arange(B) % eps.shape[0]]).half()
    return add_noise_ref(z, noise.half(), sigma)


@pytest.fixture()
def patched_enc(patched, monkeypatch):  # noqa: F811
    import imagharmony_b200.ops as real_ops
    monkeypatch.setattr(real_ops, "conv3x3_s2_padbr", _conv3x3_s2_padbr)
    monkeypatch.setattr(real_ops, "image_im2col3x3", _image_im2col3x3)
    monkeypatch.setattr(real_ops, "vae_sample_add_noise", _vae_sample_add_noise)
    yield


def _pair(cfg, seed=0, scale_conv_in=1.0):
    from imagharmony_b200.vae import AutoencoderKLEncoder
    from imagharmony_b200.weights import random_state_dict, shapes_of
    from oracle.vae_encoder_ref import VAEEncoderRef
    with torch.device("meta"):
        shapes = shapes_of(VAEEncoderRef(cfg))
    sd = {k: v.float() for k, v in random_state_dict(shapes, seed).items()}
    for k in ("encoder.conv_in.weight", "encoder.conv_in.bias"):
        sd[k] = sd[k] * scale_conv_in
    ref = VAEEncoderRef(cfg)
    ref.load_state_dict(sd)
    with torch.device("meta"):
        native = AutoencoderKLEncoder(cfg)
    native.load_state_dict(sd, assign=True)
    native.finalize()
    return native, ref.eval()


def _nchw(moments, L=4):
    return moments[..., :2 * L].permute(0, 3, 1, 2)


def test_encoder_wiring_matches_oracle_for_all_stream_scales(patched_enc):
    """diffusers key names, and the same function for stream scales 1, 2^-7, 2^-10 (fp32 stand-in ops), on a model
    whose residual stream reaches ~1e5 (it would overflow fp16 without the scaling)."""
    from imagharmony_b200.config import TINY_VAE
    native, ref = _pair(TINY_VAE, seed=3, scale_conv_in=50000.0)
    assert list(native.state_dict().keys()) == list(ref.state_dict().keys())
    assert native.stream_scale == 2.0 ** -7
    x = torch.rand(2, 3, 24, 40, generator=torch.Generator().manual_seed(1)) * 2 - 1
    with torch.no_grad():
        r = ref.encode(x)
        stream = ref.encoder.conv_in(x)
    assert stream.abs().max() > 65504
    for k in (0, 7, 10):
        native.stream_scale = 2.0 ** -k
        native.finalize()
        with torch.no_grad():
            o = native.encode(x)
        assert o.shape == (2, 3, 5, 16) and torch.all(o[..., 8:] == 0)
        assert torch.allclose(_nchw(o), r, rtol=2e-4, atol=2e-4), (k, (_nchw(o) - r).abs().max())


def test_encoder_pixel_front_end_matches_oracle_preprocess(patched_enc):
    """uint8 PIL pixels -> [3P] VaeImageProcessor normalisation (fp32 / 255, 2 x - 1) -> encoder."""
    from imagharmony_b200.config import TINY_VAE
    from oracle.vae_encoder_ref import preprocess_ref
    native, ref = _pair(TINY_VAE, seed=4)
    u8 = torch.randint(0, 256, (1, 16, 32, 3), generator=torch.Generator().manual_seed(2), dtype=torch.uint8)
    with torch.no_grad():
        r = ref.encode(preprocess_ref(u8.numpy()).half().float())      # the kernel rounds the normalised pixel to fp16
        o = native.encode(u8)
    assert torch.allclose(_nchw(o), r, rtol=1e-4, atol=1e-4), (_nchw(o) - r).abs().max()


def test_folded_quant_conv_equals_conv_out_then_quant_conv(patched_enc):
    from imagharmony_b200.config import TINY_VAE
    native, ref = _pair(TINY_VAE, seed=5)
    C = TINY_VAE.block_out_channels[-1]
    h = torch.randn(2, C, 5, 7, generator=torch.Generator().manual_seed(3))
    want = ref.quant_conv(ref.encoder.conv_out(h))
    w = native._w_out.reshape(16, 3, 3, C).permute(0, 3, 1, 2)
    got = F.conv2d(h, w, native._b_out, padding=1)
    assert torch.allclose(got[:, :8], want, rtol=1e-5, atol=1e-5) and torch.all(got[:, 8:] == 0)


def test_tiled_encode_matches_oracle(patched_enc):
    """enable_vae_tiling(): a non-square image larger than one 64-pixel tile (ragged edge tiles) through tiles + blend."""
    from imagharmony_b200.config import TINY_VAE
    from oracle.vae_encoder_ref import tiled_encode_ref
    native, ref = _pair(TINY_VAE, seed=6)
    native.use_tiling = True
    x = torch.rand(1, 3, 112, 88, generator=torch.Generator().manual_seed(4)) * 2 - 1
    with torch.no_grad():
        r = tiled_encode_ref(ref, x)
        o = native.encode(x)
    assert _nchw(o).shape == r.shape == (1, 8, 14, 11)
    assert torch.allclose(_nchw(o), r, rtol=1e-4, atol=1e-4), (_nchw(o) - r).abs().max()
    small = x[:, :, :64, :48].contiguous()                               # fits one tile: the plain path
    with torch.no_grad():
        assert torch.allclose(_nchw(native.encode(small)), ref.encode(small), rtol=1e-4, atol=1e-4)


def test_encoder_and_decoder_load_from_one_full_checkpoint(patched_enc):
    from imagharmony_b200.config import TINY_VAE
    from imagharmony_b200.vae import AutoencoderKLDecoder, AutoencoderKLEncoder
    from imagharmony_b200.weights import random_state_dict, shapes_of
    from oracle.vae_encoder_ref import VAEEncoderRef
    from oracle.vae_ref import VAEDecoderRef
    with torch.device("meta"):
        shapes = {**shapes_of(VAEEncoderRef(TINY_VAE)), **shapes_of(VAEDecoderRef(TINY_VAE))}
    full = random_state_dict(shapes, 7)
    assert any(k.startswith("encoder.") for k in full) and any(k.startswith("post_quant_conv.") for k in full)
    enc = AutoencoderKLEncoder.from_state_dict(TINY_VAE, full, device="cpu")
    dec = AutoencoderKLDecoder.from_state_dict(TINY_VAE, full, device="cpu")
    assert set(enc.state_dict()) | set(dec.state_dict()) == set(full)
    assert torch.equal(enc.quant_conv.weight, full["quant_conv.weight"].half())
    missing = {k: v for k, v in full.items() if k != "encoder.conv_out.bias"}
    with pytest.raises(KeyError):
        AutoencoderKLEncoder.from_state_dict(TINY_VAE, missing, device="cpu")


@pytest.mark.parametrize("T,strength,t_start,n_exec", [
    (50, 0.6, 20, 30), (50, 0.3, 35, 15), (50, 1.0, 0, 50), (4, 0.6, 2, 2), (3, 0.5, 2, 1), (25, 0.99, 1, 24),
    (50, 0.01, 50, 0), (7, 0.0, 7, 0)])
def test_schedule_arithmetic(T, strength, t_start, n_exec):
    from ip_adapter.custom_pipelines import StableDiffusionXLImg2ImgCustomPipeline as P
    from oracle.img2img_ref import get_timesteps
    assert P.get_timesteps(T, strength) == get_timesteps(T, strength) == (t_start, n_exec)


def _pipe():
    from imagharmony_b200.config import TINY, TINY_VAE
    from ip_adapter.custom_pipelines import StableDiffusionXLImg2ImgCustomPipeline
    return StableDiffusionXLImg2ImgCustomPipeline.from_random(TINY, seed=0, device="cpu", vae_cfg=TINY_VAE)


def _embeds(n=1):
    from imagharmony_b200.config import TINY
    g = torch.Generator().manual_seed(11)
    return dict(prompt_embeds=torch.randn(n, 81, TINY.cross_attention_dim, generator=g).half(),
                negative_prompt_embeds=torch.randn(n, 81, TINY.cross_attention_dim, generator=g).half(),
                pooled_prompt_embeds=torch.randn(n, TINY.pooled_embed_dim, generator=g).half(),
                negative_pooled_prompt_embeds=torch.randn(n, TINY.pooled_embed_dim, generator=g).half())


def test_empty_schedule_and_bad_strength_raise(patched_enc):
    from PIL import Image
    pipe = _pipe()
    src = Image.new("RGB", (64, 64), (10, 200, 30))
    for strength, T in ((0.0, 10), (0.2, 3), (1.5, 10), (-0.1, 10)):
        with pytest.raises(ValueError):
            pipe(image=src, strength=strength, num_inference_steps=T, output_type="latent", **_embeds())
    with pytest.raises(ValueError):
        pipe(strength=0.5, num_inference_steps=4, output_type="latent", **_embeds())


@pytest.mark.parametrize("gen_kind", ["single", "list"])
def test_draw_order_matches_oracle(patched_enc, gen_kind):
    """Posterior eps first, then noise; a generator list draws per batch slot (the image replicated to the batch)."""
    from PIL import Image
    from oracle.img2img_ref import init_latents_ref
    pipe = _pipe()
    rng = np.random.default_rng(3)
    src = Image.fromarray(rng.integers(0, 256, (44, 70, 3), dtype=np.uint8))      # resized down to 40 x 64
    pipe.scheduler.set_timesteps(10)
    sigma = float(pipe.scheduler.sigmas[4])

    def gens():
        if gen_kind == "list":
            return [torch.Generator().manual_seed(s) for s in (5, 6, 7)]
        return torch.Generator().manual_seed(5)
    lat, size = pipe.prepare_img2img_latents(src, 3, gens(), sigma)
    assert size == (40, 64) and lat.shape == (3, 4, 5, 8) and lat.dtype == torch.float16
    kind, x = pipe.preprocess_image(src)
    assert kind == "pixels" and tuple(x.shape) == (1, 40, 64, 3)
    moments = _nchw(pipe.vae_encoder.encode(x)).float()
    want = init_latents_ref(moments, 3, gens(), pipe.vae_encoder.config.scaling_factor, sigma)
    assert torch.equal(lat, want)
    if gen_kind == "list":                       # a candidate does not depend on its batch slot
        alone, _ = pipe.prepare_img2img_latents(src, 1, [torch.Generator().manual_seed(7)], sigma)
        assert torch.equal(alone[0], lat[2])
    else:                                        # one posterior sample shared by the copies, different noise
        assert not torch.equal(lat[0], lat[1])


def test_image_tensor_inputs(patched_enc):
    """A float tensor in [0, 1] is normalised 2 x - 1, one with negative values is used as it is, and a 4-channel tensor
    is taken as latents without encoding."""
    pipe = _pipe()
    x01 = torch.rand(1, 3, 16, 24, generator=torch.Generator().manual_seed(1))
    k1, a = pipe.preprocess_image(x01)
    k2, b = pipe.preprocess_image(x01 * 2 - 1)
    assert k1 == k2 == "image" and torch.equal(a, b)
    lat = torch.randn(2, 4, 2, 3)
    k3, c = pipe.preprocess_image(lat)
    assert k3 == "latents" and torch.equal(c, lat.half())
    out, size = pipe.prepare_img2img_latents(lat, 2, None, 0.0)
    assert size == (16, 24) and torch.equal(out, lat.half())            # sigma 0: the latents unchanged


@pytest.mark.parametrize("strength", [0.3, 0.6, 1.0])
@pytest.mark.parametrize("opts", [dict(guidance_scale=5.0, control_guidance_start=0.3),
                                  dict(guidance_scale=1.0, control_guidance_end=0.6)])
def test_img2img_trajectory_matches_oracle(patched, strength, opts):
    """engine.run(start_step=t_start, count_from_start=True) on the noised latents vs the oracle's img2img loop: the
    same latents, gating and callback indices counted over the executed steps."""
    from imagharmony_b200.config import TINY
    from oracle.img2img_ref import get_timesteps, img2img_denoise_loop
    native, ref = _build(TINY, 4)
    T, n, lat = 10, 2, 8
    t_start, n_exec = get_timesteps(T, strength)
    latents = torch.randn(n, 4, lat, lat, generator=torch.Generator().manual_seed(8)) * 3
    _, ehs, te, tid = _inputs(TINY, n, lat, seed=9)
    te = te.half().float()
    procs = [p for p in ref.attn_processors.values() if hasattr(p, "to_k_ip")]
    scales_ref = []

    def set_scale(s):
        scales_ref.append(s)
        for p in procs:
            p.scale = s
    seen_ref, seen = [], []
    r = img2img_denoise_loop(lambda s, t, e, x, y: ref(s, t, e, x, y), latents.clone(), ehs[n:], ehs[:n], te[n:], te[:n],
                             tid[:n], T, strength, set_scale=set_scale, conditioning_scale=0.8,
                             callback=lambda i, t, x: seen_ref.append((i, float(t), x.clone())), callback_steps=2, **opts)
    eng = _fp32_engine(native)
    scales = []
    orig = eng.set_scale

    def record(s):
        scales.append(s)
        orig(s)
    eng.set_scale = record
    with _Empty32():
        o = eng.run(latents.clone(), ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T, ip_scale=0.8, start_step=t_start,
                    count_from_start=True, callback=lambda i, t, x: seen.append((i, float(t), x.clone())),
                    callback_steps=2, **opts)
    assert torch.allclose(o, r, rtol=3e-4, atol=1e-3), (o - r).abs().max()
    assert [s[0] for s in seen] == [s[0] for s in seen_ref] == list(range(0, n_exec, 2))
    assert [s[1] for s in seen] == [s[1] for s in seen_ref]
    assert scales[:-1] == scales_ref                  # the last set_scale restores ip_scale after the loop
    assert 0.0 in scales_ref and 0.8 in scales_ref


def test_pipeline_and_ip_adapter_surface(patched_enc):
    """StableDiffusionXLImg2ImgCustomPipeline runs T - t_start steps (callback count), original / target size default to
    the image size, and IPAdapterXL.generate(image=..., strength=...) reaches it through **kwargs."""
    from PIL import Image
    from imagharmony_b200.config import HARMONY_TINY as h
    from ip_adapter import IPAdapterXL
    from train import HarmonyAttention
    pipe = _pipe()
    src = Image.fromarray(np.random.default_rng(5).integers(0, 256, (64, 32, 3), dtype=np.uint8))
    calls = []
    out = pipe(image=src, strength=0.5, num_inference_steps=6, output_type="latent",
               callback=lambda i, t, x: calls.append(i), generator=torch.Generator().manual_seed(1), **_embeds()).images
    assert out.shape == (1, 4, 8, 4) and calls == [0, 1, 2] and torch.isfinite(out.float()).all()
    calls.clear()
    pipe(image=src, strength=0.5, num_inference_steps=6, output_type="latent", denoising_end=0.8,
         callback=lambda i, t, x: calls.append(i), **_embeds())
    assert calls == [0]                  # denoising_end keeps 4 of the 6 timesteps (t >= 200); from t_start = 3 one runs
    pipe.enable_vae_tiling()
    assert pipe.vae.use_tiling and pipe.vae_encoder.use_tiling
    ha = HarmonyAttention(image_hidden_size=h.image_hidden_size, text_context_dim=h.text_context_dim,
                          inter_dim=h.inter_dim, cross_heads=h.cross_heads, reshape_blocks=h.reshape_blocks,
                          cross_value_dim=h.cross_value_dim, scale=1.0, fusion_method="cross_attention")
    ip = IPAdapterXL(pipe, None, None, "cpu", num_tokens=4, inference=True, number_class_crossattention=ha)
    calls.clear()
    pil = ip.generate(pil_image=None, clip_image_embeds=torch.randn(1, h.image_hidden_size), image=src, strength=0.6,
                      prompt="lions", num_samples=2, num_inference_steps=5, seed=[3, 4], extra_text="eight sheep",
                      callback=lambda i, t, x: calls.append(i))
    assert isinstance(pil, list) and len(pil) == 2 and pil[0].size == (32, 64) and calls == [0, 1, 2]
