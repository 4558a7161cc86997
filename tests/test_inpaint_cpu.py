"""CPU tests of masked inpainting: the mask front end, the start latents and their generator draw order, and the
blended denoise trajectory, against the fp32 oracle (oracle/inpaint_ref.py) with stand-in ops (no kernels involved;
those are tests/test_inpaint_gpu.py)."""
import numpy as np
import pytest
import torch

import fake_ops
from test_img2img_cpu import _embeds, _nchw, patched_enc  # noqa: F401  (fixture)
from test_wiring_cpu import _build, _Empty32, _fp32_engine, _inputs, patched  # noqa: F401  (fixture)


def _vae_sample_inpaint(moments, eps, noise, channels, scaling_factor, sigma, pure_noise):
    from oracle.vae_encoder_ref import posterior_sample_ref
    from oracle.img2img_ref import add_noise_ref
    B, C = noise.shape[0], channels
    m = moments.float().permute(0, 3, 1, 2)[torch.arange(B) % moments.shape[0]]
    if eps is None:
        z0 = m[:, :C].half()
    else:
        z0 = scaling_factor * posterior_sample_ref(m[:, :2 * C], eps[torch.arange(B) % eps.shape[0]]).half()
    if pure_noise:
        return (noise.float() * torch.tensor(sigma, dtype=torch.float32)).half(), z0
    return add_noise_ref(z0, noise.half(), sigma), z0


def _latent_mask(mask_u8):
    return (mask_u8[:, ::8, ::8] >= 128).to(torch.uint8)


def _euler_step_inpaint(noise_pred, latents, model_in, sigmas, step, guidance, mask, z0, noise, last, *, use_cfg=True,
                        guidance_rescale=0.0):
    from oracle.inpaint_ref import blend_ref
    k = int(step.item())
    fake_ops.euler_step(noise_pred, latents, model_in, sigmas, step, guidance, use_cfg=use_cfg,
                        guidance_rescale=guidance_rescale)
    sn = float(sigmas[k + 1])
    latents.copy_(blend_ref(latents, mask[:, None], z0, noise, sn, last=k == int(last.item())))
    mi = (latents.float() / (sn * sn + 1) ** 0.5).to(model_in.dtype)
    model_in.copy_(torch.cat([mi, mi]) if use_cfg else mi)


@pytest.fixture()
def patched_inp(patched_enc, monkeypatch):  # noqa: F811
    import imagharmony_b200.ops as real_ops
    monkeypatch.setattr(real_ops, "vae_sample_inpaint", _vae_sample_inpaint, raising=True)
    monkeypatch.setattr(real_ops, "latent_mask", _latent_mask, raising=True)
    monkeypatch.setattr(real_ops, "euler_step_inpaint", _euler_step_inpaint, raising=True)
    yield


def _pipe():
    from imagharmony_b200.config import TINY, TINY_VAE
    from ip_adapter.custom_pipelines import StableDiffusionXLInpaintCustomPipeline
    return StableDiffusionXLInpaintCustomPipeline.from_random(TINY, seed=0, device="cpu", vae_cfg=TINY_VAE)


def _src(h, w, seed=3):
    from PIL import Image
    return Image.fromarray(np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8))


@pytest.mark.parametrize("mode,size,target", [("L", (48, 80), (48, 80)), ("RGB", (48, 80), (48, 80)),
                                              ("L", (61, 37), (48, 80)), ("RGB", (100, 100), (64, 40))])
def test_mask_front_end_matches_pil_numpy(patched_inp, mode, size, target):
    """PIL mask -> "L" -> Lanczos resize to (width, height) -> v / 255 >= 0.5 -> nearest latent mask (pixel (8y, 8x))."""
    from PIL import Image
    from oracle.inpaint_ref import latent_mask_ref, mask_ref
    H, W = target
    rng = np.random.default_rng(sum(size))
    arr = rng.integers(0, 256, size if mode == "L" else size + (3,), dtype=np.uint8)
    arr[..., :2, :] = 127                                                   # the threshold edge
    arr[..., 2:4, :] = 128
    im = Image.fromarray(arr, mode)
    pipe = _pipe()
    got = pipe.preprocess_mask([im, im.transpose(Image.FLIP_LEFT_RIGHT)], H, W)
    L = im.convert("L")
    want = np.asarray(L if L.size == (W, H) else L.resize((W, H), resample=Image.LANCZOS))
    assert got.dtype == torch.uint8 and got.shape == (2, H, W) and np.array_equal(got[0].numpy(), want)
    lat = _latent_mask(got)
    ref = latent_mask_ref(mask_ref([im, im.transpose(Image.FLIP_LEFT_RIGHT)], H, W), H // 8, W // 8)
    assert lat.shape == (2, H // 8, W // 8) and torch.equal(lat.half(), ref[:, 0])
    if size == target and mode == "L":
        assert torch.all(lat[0, 0] == 0)                                       # row 0 is 127: kept
        assert torch.equal(pipe.preprocess_mask(im, H, W)[0, 2:4], torch.full((2, W), 128, dtype=torch.uint8))
        assert torch.all(_latent_mask(pipe.preprocess_mask(Image.fromarray(np.full((H, W), 128, np.uint8)), H, W)) == 1)


def test_tensor_mask_binarized_and_size_checked(patched_inp):
    from oracle.inpaint_ref import mask_ref
    pipe = _pipe()
    m = torch.rand(2, 16, 24, generator=torch.Generator().manual_seed(1))
    m[0, 0, :3] = torch.tensor([0.4999, 0.5, 1.0])
    for t in (m, m[:, None], m[0]):
        got = pipe.preprocess_mask(t, 16, 24)
        want = (mask_ref(t, 16, 24)[:, 0] * 255).to(torch.uint8)
        assert got.dtype == torch.uint8 and torch.equal(got, want)
    assert got.shape == (1, 16, 24) and got[0, 0, :3].tolist() == [0, 255, 255]
    for bad in (m[:, :8], torch.rand(16, 32), torch.rand(2, 3, 16, 24)):
        with pytest.raises(ValueError):
            pipe.preprocess_mask(bad, 16, 24)
    with pytest.raises(ValueError):
        pipe.preprocess_mask(m * 2, 16, 24)


def test_default_size_is_unet_sample_size(patched_inp):
    """height / width default to sample_size * 8 (256 for the miniature UNet) whatever the image size; time ids follow."""
    from PIL import Image
    pipe = _pipe()
    assert pipe.default_sample_size * 8 == 256
    tids = []
    orig = pipe.engine.run

    def run(*a, **k):
        tids.append(a[5])
        return orig(*a, **k)
    pipe.engine.run = run
    out = pipe(image=_src(40, 72), mask_image=Image.new("L", (72, 40), 255), strength=0.5, num_inference_steps=2,
               output_type="latent", **_embeds()).images
    assert out.shape == (1, 4, 32, 32) and tids[0].tolist() == [[256.0, 256.0, 0.0, 0.0, 256.0, 256.0]]
    out = pipe(image=_src(40, 72), mask_image=Image.new("L", (72, 40), 255), strength=0.5, num_inference_steps=2,
               height=64, width=128, output_type="latent", **_embeds()).images
    assert out.shape == (1, 4, 8, 16) and tids[1].tolist() == [[64.0, 128.0, 0.0, 0.0, 64.0, 128.0]]


@pytest.mark.parametrize("batch", [2, 4])
@pytest.mark.parametrize("gen_kind", ["single", "list"])
def test_draw_order_matches_oracle(patched_inp, gen_kind, batch):
    """eps first (fp32; per source image only, also with a generator list), then the noise (fp16, per batch slot)."""
    from PIL import Image
    from oracle.inpaint_ref import init_latents_ref
    pipe = _pipe()
    src = _src(44, 70)
    pipe.scheduler.set_timesteps(10)
    sigma = float(pipe.scheduler.sigmas[4])

    def gens():
        if gen_kind == "list":
            return [torch.Generator().manual_seed(s) for s in range(5, 5 + batch)]
        return torch.Generator().manual_seed(5)
    lat, (mask, z0, noise) = pipe.prepare_inpaint_latents(src, Image.new("L", (64, 40), 200), batch, gens(), 40, 64, 4,
                                                          False)
    assert lat.shape == z0.shape == noise.shape == (batch, 4, 5, 8) and lat.dtype == torch.float16
    assert mask.shape == (1, 5, 8) and torch.all(mask == 1)
    kind, x = pipe.preprocess_image(src.resize((64, 40), resample=Image.LANCZOS))
    moments = _nchw(pipe.vae_encoder.encode(x)).float()
    want = init_latents_ref(moments, batch, gens(), pipe.vae_encoder.config.scaling_factor, sigma)
    assert torch.equal(lat, want[0]) and torch.equal(z0, want[1]) and torch.equal(noise, want[2])
    assert all(torch.equal(z0[0], z0[b]) for b in range(batch))           # one source image, repeated
    if gen_kind == "list":                       # generator[0] draws eps and then its noise; the others only noise
        g = torch.Generator().manual_seed(5 + batch - 1)
        assert torch.equal(noise[-1], torch.randn((1, 4, 5, 8), generator=g, dtype=torch.float16)[0])
        g = torch.Generator().manual_seed(5)
        torch.randn((1, 4, 5, 8), generator=g)
        assert torch.equal(noise[0], torch.randn((1, 4, 5, 8), generator=g, dtype=torch.float16)[0])
    else:
        assert not torch.equal(noise[0], noise[1])


def test_strength_one_starts_from_pure_noise(patched_inp):
    from PIL import Image
    from oracle.inpaint_ref import init_latents_ref
    pipe = _pipe()
    src = _src(40, 64)
    pipe.scheduler.set_timesteps(10)
    s0 = pipe.scheduler.init_noise_sigma
    lat, (_, z0, noise) = pipe.prepare_inpaint_latents(src, Image.new("L", (64, 40), 0), 2,
                                                       torch.Generator().manual_seed(2), 40, 64, 0, True)
    assert torch.equal(lat, (noise.float() * torch.tensor(s0, dtype=torch.float32)).half())
    kind, x = pipe.preprocess_image(src)
    want = init_latents_ref(_nchw(pipe.vae_encoder.encode(x)).float(), 2, torch.Generator().manual_seed(2),
                            pipe.vae_encoder.config.scaling_factor, 0.0, is_strength_max=True, init_noise_sigma=s0)
    assert torch.equal(lat, want[0]) and torch.equal(z0, want[1])        # z0 is still the encoded image


@pytest.mark.parametrize("opts", [dict(guidance_scale=5.0, control_guidance_start=0.3, strength=0.6),
                                  dict(guidance_scale=1.0, control_guidance_end=0.6, strength=1.0),
                                  dict(guidance_scale=5.0, guidance_rescale=0.7, strength=0.9999),
                                  dict(guidance_scale=5.0, denoising_end=0.7, strength=0.8)])
def test_inpaint_trajectory_matches_oracle(patched_inp, opts):
    """engine.run(inpaint=...) on the stand-in ops vs the oracle's inpaint loop: latents, gating, callback indices
    (counted over the executed steps) and the clean z0 outside the mask after the last step."""
    from imagharmony_b200.config import TINY
    from oracle.img2img_ref import get_timesteps
    from oracle.inpaint_ref import inpaint_denoise_loop
    from oracle.scheduler_ref import denoising_end_steps
    opts = dict(opts)
    strength = opts.pop("strength")
    native, ref = _build(TINY, 4)
    T, n, lat = 10, 2, 8
    t_start, _ = get_timesteps(T, strength)
    loop_T = denoising_end_steps(T, opts.get("denoising_end"))
    g = torch.Generator().manual_seed(8)
    latents = torch.randn(n, 4, lat, lat, generator=g) * 3
    z0 = torch.randn(n, 4, lat, lat, generator=g).half()
    noise = torch.randn(n, 4, lat, lat, generator=g).half()
    mask = torch.zeros(1, lat, lat, dtype=torch.uint8)
    mask[:, 2:6, 1:5] = 1
    _, ehs, te, tid = _inputs(TINY, n, lat, seed=9)
    te = te.half().float()
    procs = [p for p in ref.attn_processors.values() if hasattr(p, "to_k_ip")]
    scales_ref = []

    def set_scale(s):
        scales_ref.append(s)
        for p in procs:
            p.scale = s
    seen_ref, seen = [], []
    r = inpaint_denoise_loop(lambda s, t, e, x, y: ref(s, t, e, x, y), latents.clone(), ehs[n:], ehs[:n], te[n:],
                             te[:n], tid[:n], T, strength, mask[:, None].half(), z0, noise, set_scale=set_scale,
                             conditioning_scale=0.8, callback=lambda i, t, x: seen_ref.append((i, float(t), x.clone())),
                             callback_steps=2, **opts)
    eng = _fp32_engine(native)
    scales = []
    orig = eng.set_scale

    def record(s):
        scales.append(s)
        orig(s)
    eng.set_scale = record
    denoising_end = opts.pop("denoising_end", None)
    with _Empty32():
        o = eng.run(latents.clone(), ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T, ip_scale=0.8, start_step=t_start,
                    num_loop_steps=loop_T, count_from_start=True, inpaint=(mask, z0, noise),
                    callback=lambda i, t, x: seen.append((i, float(t), x.clone())), callback_steps=2, **opts)
    assert torch.allclose(o, r, rtol=3e-4, atol=1e-3), (o - r).abs().max()
    assert [s[0] for s in seen] == [s[0] for s in seen_ref] == list(range(0, loop_T - t_start, 2))
    for (_, _, a), (_, _, b) in zip(seen, seen_ref):
        assert torch.allclose(a, b, rtol=3e-4, atol=1e-3)
    assert scales[:-1] == scales_ref
    out = (mask == 0)[:, None].expand_as(o)
    assert torch.equal(o[out], z0.float()[out]) and torch.equal(r[out], z0.float()[out])   # the last step: z0 itself
    if denoising_end is not None:
        assert loop_T < T                                       # the last step is cut short: sigma[k + 1] != 0


def test_errors(patched_inp):
    from PIL import Image
    pipe = _pipe()
    src, m = _src(64, 64), Image.new("L", (64, 64), 255)
    kw = dict(num_inference_steps=4, output_type="latent", height=64, width=64)
    with pytest.raises(ValueError):
        pipe(image=src, **kw, **_embeds())                                   # no mask
    with pytest.raises(ValueError):
        pipe(mask_image=m, **kw, **_embeds())                                # no image
    for strength, T in ((1.5, 4), (-0.1, 4), (0.0, 4), (0.2, 3)):            # bad strength, empty schedules
        with pytest.raises(ValueError):
            pipe(image=src, mask_image=m, strength=strength, **{**kw, "num_inference_steps": T}, **_embeds())
    with pytest.raises(ValueError, match="leaves no denoising"):
        pipe(image=src, mask_image=m, strength=0.2, **{**kw, "num_inference_steps": 3}, **_embeds())
    with pytest.raises(ValueError, match="do not divide"):
        pipe(image=src, mask_image=[m, m, m], num_images_per_prompt=1, **kw, **_embeds(2))
    with pytest.raises(ValueError, match="divisible by 8"):
        pipe(image=src, mask_image=m, **{**kw, "height": 60}, **_embeds())


def test_pipeline_and_ip_adapter_surface(patched_inp):
    """IPAdapterXL.generate(pil_image=..., image=..., mask_image=...) reaches the inpaint pipeline through **kwargs and
    returns PIL images of (width, height); the callback counts the executed steps from 0."""
    from PIL import Image
    from imagharmony_b200.config import HARMONY_TINY as h
    from ip_adapter import IPAdapterXL
    from train import HarmonyAttention
    pipe = _pipe()
    ha = HarmonyAttention(image_hidden_size=h.image_hidden_size, text_context_dim=h.text_context_dim,
                          inter_dim=h.inter_dim, cross_heads=h.cross_heads, reshape_blocks=h.reshape_blocks,
                          cross_value_dim=h.cross_value_dim, scale=1.0, fusion_method="cross_attention")
    ip = IPAdapterXL(pipe, None, None, "cpu", num_tokens=4, inference=True, number_class_crossattention=ha)
    calls = []
    mask = Image.new("L", (48, 40), 0)
    mask.paste(255, (8, 8, 32, 24))
    pil = ip.generate(pil_image=None, clip_image_embeds=torch.randn(1, h.image_hidden_size), image=_src(40, 48),
                      mask_image=mask, strength=0.6, prompt="lions", num_samples=2, num_inference_steps=5, seed=[3, 4],
                      extra_text="eight sheep", height=32, width=64, callback=lambda i, t, x: calls.append(i))
    assert isinstance(pil, list) and len(pil) == 2 and pil[0].size == (64, 32) and calls == [0, 1, 2]
