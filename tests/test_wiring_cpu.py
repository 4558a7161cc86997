"""CPU test of the native UNet / processor / denoise-loop WIRING: imagharmony_b200.ops is swapped for plain-PyTorch fp32
stand-ins (tests/fake_ops.py, test-only) so that layouts, skip-connection order, weight packing, temb offsets and the
K/V cache logic are compared with the oracle to fp32 round-off -- no kernels involved (those are the -m gpu tests)."""
import sys

import pytest
import torch

import fake_ops


@pytest.fixture()
def patched(monkeypatch):
    import imagharmony_b200.ops as real_ops
    for name in dir(fake_ops):
        if not name.startswith("_") and callable(getattr(fake_ops, name)) and hasattr(real_ops, name):
            monkeypatch.setattr(real_ops, name, getattr(fake_ops, name))
    yield


def _build(cfg, seed):
    from imagharmony_b200.unet import UNet2DConditionModel
    from imagharmony_b200.weights import random_state_dict, shapes_of
    from oracle import adapter_ref as A
    from oracle.unet_ref import UNetRef
    with torch.device("meta"):
        shapes = shapes_of(UNetRef(cfg))
    sd = {k: v.float() for k, v in random_state_dict(shapes, seed).items()}
    with torch.device("meta"):
        native = UNet2DConditionModel(cfg)
    native.load_state_dict(sd, assign=True)
    native.install_default_processors()
    procs = torch.nn.ModuleList(native.attn_processors.values()).float()
    ip_sd = {k: v.float() for k, v in random_state_dict(shapes_of(procs), seed + 1).items()}
    procs.load_state_dict(ip_sd)
    native.finalize()
    ref = UNetRef(cfg)
    ref.load_state_dict(sd)
    pr = A.install_processors(ref, cfg)
    torch.nn.ModuleList(pr.values()).load_state_dict(ip_sd)
    return native, ref.eval()


def _inputs(cfg, n, lat, seed=3):
    g = torch.Generator("cpu").manual_seed(seed)
    B = 2 * n
    return (torch.randn(B, 4, lat, lat, generator=g), torch.randn(B, 77 + cfg.num_ip_tokens, cfg.cross_attention_dim, generator=g),
            torch.randn(B, cfg.pooled_embed_dim, generator=g),
            torch.tensor([[lat * 8., lat * 8., 0., 0., lat * 8., lat * 8.]] * B))


def test_native_unet_wiring_matches_oracle(patched):
    from imagharmony_b200.config import TINY
    native, ref = _build(TINY, 0)
    sample, ehs, te, tid = _inputs(TINY, 1, 16)
    with torch.no_grad():
        r = ref(sample, 321.0, ehs, te, tid)
        o = native(sample, torch.full((2,), 321.0), ehs, te, tid)
    assert o.shape == r.shape
    assert torch.allclose(o, r, rtol=1e-4, atol=1e-4), (o - r).abs().max()
    # 140 processors, same names/order as the oracle (and diffusers): the ip_adapter.bin index contract
    from oracle.unet_ref import UNetRef
    assert list(native.attn_processors.keys()) == list(ref.attn_processors.keys())
    assert set(native.state_dict().keys()) == set(ref.state_dict().keys())


def test_native_denoise_loop_wiring_matches_oracle(patched):
    from imagharmony_b200.config import TINY
    from imagharmony_b200.denoise import DenoiseEngine
    from oracle.scheduler_ref import denoise_loop, euler_tables, prepare_latents
    native, ref = _build(TINY, 2)
    T, n, lat = 3, 2, 8
    _, _, ins = euler_tables(T)
    latents = prepare_latents(n, 4, lat, lat, [1, 2], ins, dtype=torch.float32)
    _, ehs, te, tid = _inputs(TINY, n, lat, seed=5)
    # the native UNet takes the pooled embeddings in fp16 (UNet2DConditionModel add_in): fp16-representable values keep
    # the CFG-amplified difference of the 3-step loop at fp32 round-off instead of fp16 input rounding
    te = te.half().float()
    procs = [p for p in ref.attn_processors.values() if hasattr(p, "to_k_ip")]

    def set_scale(s):
        for p in procs:
            p.scale = s
    r = denoise_loop(lambda s, t, e, x, y: ref(s, t, e, x, y), latents.clone(), ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T,
                     guidance_scale=5.0, set_scale=set_scale, conditioning_scale=0.6, control_guidance_start=0.3)
    eng = DenoiseEngine.__new__(DenoiseEngine)
    DenoiseEngine.__init__(eng, native, use_cuda_graph=False)
    # fp32 CPU buffers for the wiring test
    import imagharmony_b200.denoise as dn
    orig_empty = torch.empty

    def empty32(*a, **k):
        if k.get("dtype") == torch.float16:
            k["dtype"] = torch.float32
        return orig_empty(*a, **k)
    dn.torch.empty = empty32
    try:
        o = eng.run(latents.clone(), ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T, guidance_scale=5.0, ip_scale=0.6,
                    control_guidance_start=0.3)
        # two-phase PNS building blocks: a preview (stop_after=k) resumed with start_step=k is the same trajectory
        pre = eng.run(latents.clone(), ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T, guidance_scale=5.0, ip_scale=0.6,
                      control_guidance_start=0.3, stop_after=1)
        res = eng.run(pre, ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T, guidance_scale=5.0, ip_scale=0.6,
                      control_guidance_start=0.3, start_step=1)
    finally:
        dn.torch.empty = orig_empty
    assert torch.allclose(o, r, rtol=2e-4, atol=2e-4), (o - r).abs().max()
    assert torch.equal(res, o), "preview + resume must reproduce the uninterrupted trajectory"
    assert not torch.equal(pre, o)


def test_adapter_modules_wiring_matches_reference_goldens(patched):
    """ImageProjModel / HarmonyAttention / Resampler (native classes, fp32 stand-in ops) vs the golden outputs of the
    reference's own classes; also checks that the state-dict keys are the reference's."""
    import os
    from imagharmony_b200 import adapter as N
    from oracle.check_against_reference import load_golden
    gold = load_golden(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.pt"))
    g = gold["harmony"]
    ha = N.HarmonyAttention(fusion_method="cross_attention", **g["kwargs"])
    ha.load_state_dict(g["state"])          # strict: same keys as train.py's module
    out = ha(g["text"], g["image"])
    assert torch.allclose(out, g["out"], rtol=1e-4, atol=1e-5), (out - g["out"]).abs().max()
    fused = ha(g["text"], g["image"], add_to=g["image"])
    assert torch.allclose(fused, g["image"] + g["out"], rtol=1e-4, atol=1e-5)
    g = gold["imageproj"]
    ip = N.ImageProjModel(128, 64, 4)
    ip.load_state_dict(g["state"])
    assert torch.allclose(ip(g["image"]), g["out"], rtol=1e-4, atol=1e-5)
    g = gold["resampler"]
    r = N.Resampler(**g["kwargs"])
    r.load_state_dict(g["state"])
    fake_ops.FP32 = True
    import imagharmony_b200.adapter as ad
    orig = torch.empty

    def empty32(*a, **k):
        if k.get("dtype") == torch.float16:
            k["dtype"] = torch.float32
        return orig(*a, **k)
    ad.torch.empty = empty32
    try:
        # the native forward casts the latents parameter to fp16; keep fp32 in the wiring test
        lat16 = torch.Tensor.to
        out = None
        import unittest.mock as um
        with um.patch.object(torch.Tensor, "to", lambda self, *a, **k: self if (a and a[0] == torch.float16) else lat16(self, *a, **k)):
            out = r(g["x"])
    finally:
        ad.torch.empty = orig
    assert out.shape == (2, 12, 160)
    assert torch.allclose(out, g["out"], rtol=1e-4, atol=1e-4), (out - g["out"]).abs().max()


def test_ip_adapter_xl_generate_call_surface(patched, tmp_path):
    """The reference's call surface end to end on the CPU stand-in ops: IPAdapterXL(...) with a HarmonyAttention
    module, a 3-key ip_adapter.bin (convert_bin.py layout), generate(...) with the kwargs test.py passes (including
    the stray number_class_crossattention=), list-of-seeds generators, output_type='latent'."""
    from imagharmony_b200.config import HARMONY_TINY, TINY
    from imagharmony_b200.weights import random_state_dict, shapes_of
    from ip_adapter import IPAdapterXL
    from ip_adapter.custom_pipelines import StableDiffusionXLCustomPipeline
    from tutorial_train_sdxl_ori import ComposedAttention, HarmonyAttention   # demo.py:11 / ip_adapter.py:10 import paths
    from train import HarmonyAttention as HA2                                  # test.py:5 import path
    assert HA2 is HarmonyAttention and ComposedAttention is HarmonyAttention
    from shared_models import ImageProjModel as IPM1                           # train.py:23 import path
    from ip_adapter.shared_models import ImageProjModel as IPM2                # the package's identical copy
    from ip_adapter.ip_adapter import ImageProjModel as IPM3                   # ip_adapter.py:26-48
    assert IPM1 is IPM2 is IPM3
    from ip_adapter.attention_processor import Cross_Attention as CA1           # train.py:32 import path
    from imagharmony_b200.adapter import Cross_Attention as CA2
    assert CA1 is CA2 and isinstance(HarmonyAttention(image_hidden_size=8, text_context_dim=8, inter_dim=16, cross_heads=2,
                                                      reshape_blocks=2, cross_value_dim=4).fusion_text_image, CA1)

    from imagharmony_b200.config import TINY_VAE
    pipe = StableDiffusionXLCustomPipeline.from_random(TINY, seed=0, device="cpu", vae_cfg=TINY_VAE)
    assert not hasattr(pipe, "controlnet")
    h = HARMONY_TINY
    ha = HarmonyAttention(image_hidden_size=h.image_hidden_size, text_context_dim=h.text_context_dim,
                          inter_dim=h.inter_dim, cross_heads=h.cross_heads, reshape_blocks=h.reshape_blocks,
                          cross_value_dim=h.cross_value_dim, scale=1.0, fusion_method="cross_attention")
    # build a checkpoint in the reference's 3-key format and load it through the adapter
    probe = IPAdapterXL(pipe, None, None, "cpu", num_tokens=4, target_blocks=["down_blocks.2.attentions.1"],
                        inference=True, number_class_crossattention=ha)
    ck = {"image_proj": random_state_dict(shapes_of(probe.image_proj_model), 3),
          "composed_adapter": random_state_dict(shapes_of(ha), 4),
          "ip_adapter": random_state_dict(shapes_of(torch.nn.ModuleList(pipe.unet.attn_processors.values())), 5)}
    assert len(ck["ip_adapter"]) == 2 * sum(1 for n in pipe.unet.attn_processors if n.endswith("attn2.processor"))
    path = str(tmp_path / "ip_adapter.bin")
    torch.save(ck, path)
    ip_model = IPAdapterXL(pipe, None, path, "cpu", num_tokens=4, inference=True, number_class_crossattention=ha)
    active = [n for n, p in pipe.unet.attn_processors.items() if hasattr(p, "skip") and not p.skip]
    assert active and all("down_blocks.2.attentions.1" in n for n in active)
    img = torch.randn(1, h.image_hidden_size)
    out = ip_model.generate(pil_image=None, clip_image_embeds=img, prompt="lions", negative_prompt="blurry",
                            scale=0.9, guidance_scale=5.0, num_samples=2, num_inference_steps=2, seed=[7, 8],
                            extra_text="eight sheep", number_class_crossattention=ha, output_type="latent",
                            height=128, width=128)
    assert out.shape == (2, 4, 16, 16) and torch.isfinite(out.float()).all()
    # candidate noises are slot-invariant: generating seed 8 alone reproduces the second image
    out8 = ip_model.generate(pil_image=None, clip_image_embeds=img, prompt="lions", negative_prompt="blurry",
                             scale=0.9, guidance_scale=5.0, num_samples=1, num_inference_steps=2, seed=[8],
                             extra_text="eight sheep", output_type="latent", height=128, width=128)
    assert torch.allclose(out8.float(), out[1:2].float(), atol=6e-2)   # fp16 CPU stand-in ops: BLAS blocking differs with batch
    # extra_text=None is tolerated (the reference raises NameError there)
    ip_model.generate(pil_image=None, clip_image_embeds=img, num_samples=1, num_inference_steps=1, seed=1,
                      output_type="latent", height=128, width=128)
    # the reference's default: PIL images out of the VAE decoder + postprocess (ip_adapter.py:330-340, test.py:33-41)
    pil = ip_model.generate(pil_image=None, clip_image_embeds=img, prompt="lions", num_samples=2, num_inference_steps=1,
                            seed=[3, 4], extra_text="eight sheep", height=128, width=128)
    assert isinstance(pil, list) and len(pil) == 2 and pil[0].size == (128, 128) and pil[0].mode == "RGB"
    ip_model.set_scale(0.25)
    assert all(p.scale == 0.25 for p in pipe.unet.attn_processors.values() if hasattr(p, "to_k_ip"))


def test_ip_adapter_plus_xl_generate_call_surface(patched):
    """IPAdapterPlusXL (reference :389-478): Resampler tokens (16) from penultimate CLIP hidden states appended to the 77
    text tokens, list-of-seeds generators, latent output."""
    from imagharmony_b200.config import TINY
    from ip_adapter import IPAdapterPlusXL
    from ip_adapter.custom_pipelines import StableDiffusionXLCustomPipeline
    pipe = StableDiffusionXLCustomPipeline.from_random(TINY, seed=0, device="cpu")
    model = IPAdapterPlusXL(pipe, None, None, "cpu", num_tokens=16)
    assert sum(1 for p in pipe.unet.attn_processors.values() if hasattr(p, "to_k_ip")) == \
        sum(1 for n in pipe.unet.attn_processors if n.endswith("attn2.processor"))
    g = torch.Generator().manual_seed(0)
    hs, un = torch.randn(1, 257, 1664, generator=g).half(), torch.randn(1, 257, 1664, generator=g).half()
    cond, uncond = model.get_image_embeds(None, hs, un)
    assert cond.shape == uncond.shape == (1, 16, TINY.cross_attention_dim)
    out = model.generate(prompt="lions", num_samples=2, num_inference_steps=1, seed=[1, 2], clip_hidden_states=hs,
                         uncond_clip_hidden_states=un, output_type="latent", height=128, width=128)
    assert out.shape == (2, 4, 16, 16) and torch.isfinite(out.float()).all()


def _fp32_engine(native):
    """DenoiseEngine on the CPU stand-in ops with fp32 static buffers (wiring tests compare to fp32 round-off)."""
    from imagharmony_b200.denoise import DenoiseEngine
    return DenoiseEngine(native, use_cuda_graph=False)


class _Empty32:
    """Context manager: torch.empty(dtype=float16) inside imagharmony_b200.denoise allocates fp32 instead."""

    def __enter__(self):
        import imagharmony_b200.denoise as dn
        self.dn, self.orig = dn, torch.empty

        def empty32(*a, **k):
            if k.get("dtype") == torch.float16:
                k["dtype"] = torch.float32
            return self.orig(*a, **k)
        dn.torch.empty = empty32

    def __exit__(self, *a):
        self.dn.torch.empty = self.orig


@pytest.mark.parametrize("opts", [
    dict(guidance_scale=1.0),                                   # custom_pipelines.py:223 -- no classifier-free guidance
    dict(guidance_scale=5.0, guidance_rescale=0.7),             # :352-354
    dict(guidance_scale=5.0, denoising_end=0.5),                # :307-316
    dict(guidance_scale=0.5, denoising_end=0.7),
])
def test_denoise_loop_options_match_oracle(patched, opts):
    """The loop options the reference accepts (no CFG, guidance_rescale, denoising_end, callback) through the native
    engine on the stand-in ops vs the oracle loop."""
    from imagharmony_b200.config import TINY
    from oracle.scheduler_ref import denoise_loop, denoising_end_steps, euler_tables, prepare_latents
    native, ref = _build(TINY, 4)
    T, n, lat = 4, 2, 8
    _, _, ins = euler_tables(T)
    latents = prepare_latents(n, 4, lat, lat, [5, 6], ins, dtype=torch.float32)
    _, ehs, te, tid = _inputs(TINY, n, lat, seed=9)
    procs = [p for p in ref.attn_processors.values() if hasattr(p, "to_k_ip")]

    def set_scale(s):
        for p in procs:
            p.scale = s
    seen_ref, seen = [], []
    r = denoise_loop(lambda s, t, e, x, y: ref(s, t, e, x, y), latents.clone(), ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T,
                     set_scale=set_scale, conditioning_scale=0.8, control_guidance_end=0.75,
                     callback=lambda i, t, x: seen_ref.append((i, float(t), x.clone())), callback_steps=2, **opts)
    eng = _fp32_engine(native)
    kw = dict(opts)
    de = kw.pop("denoising_end", None)
    loop_steps = denoising_end_steps(T, de)
    with _Empty32():
        o = eng.run(latents.clone(), ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T, ip_scale=0.8, control_guidance_end=0.75,
                    num_loop_steps=loop_steps, callback=lambda i, t, x: seen.append((i, float(t), x.clone())),
                    callback_steps=2, **kw)
    assert torch.allclose(o, r, rtol=3e-4, atol=1e-3), (o - r).abs().max()    # fp32 round-off at |latent| ~ 10
    assert [s[0] for s in seen] == [s[0] for s in seen_ref] and [s[1] for s in seen] == [s[1] for s in seen_ref]
    for a, b in zip(seen, seen_ref):
        assert torch.allclose(a[2], b[2], rtol=3e-4, atol=1e-3)


def test_pipeline_forwards_loop_options(patched):
    """StableDiffusionXLCustomPipeline.__call__ accepts what the reference accepts (custom_pipelines.py:23-56):
    guidance_scale <= 1, guidance_rescale, denoising_end, callback, negative micro-conditioning -- no IHError."""
    from imagharmony_b200.config import TINY
    from ip_adapter.custom_pipelines import StableDiffusionXLCustomPipeline
    pipe = StableDiffusionXLCustomPipeline.from_random(TINY, seed=0, device="cpu")
    pe, ne = torch.randn(1, 81, TINY.cross_attention_dim).half(), torch.randn(1, 81, TINY.cross_attention_dim).half()
    pp, npool = torch.randn(1, TINY.pooled_embed_dim).half(), torch.randn(1, TINY.pooled_embed_dim).half()
    calls = []
    common = dict(prompt_embeds=pe, negative_prompt_embeds=ne, pooled_prompt_embeds=pp, negative_pooled_prompt_embeds=npool,
                  num_inference_steps=4, output_type="latent", height=64, width=64,
                  generator=torch.Generator("cpu").manual_seed(1))
    a = pipe(guidance_scale=5.0, guidance_rescale=0.5, callback=lambda i, t, x: calls.append(i), callback_steps=1,
             negative_original_size=(32, 32), negative_target_size=(64, 64), **common).images
    assert calls == [0, 1, 2, 3] and torch.isfinite(a.float()).all()
    common["generator"] = torch.Generator("cpu").manual_seed(1)
    calls.clear()
    b = pipe(guidance_scale=1.0, denoising_end=0.5, callback=lambda i, t, x: calls.append(i), **common).images
    assert calls == [0, 1] and torch.isfinite(b.float()).all() and not torch.equal(a, b)
    with pytest.raises(ValueError):
        pipe(guidance_scale=5.0, callback=lambda *a: None, callback_steps=0, **common)
    # the engine integrates the pipeline's own scheduler object (a replaced scheduler rebuilds the engine)
    from imagharmony_b200.scheduler import EulerDiscreteScheduler
    e0 = pipe.engine
    assert e0.scheduler is pipe.scheduler
    pipe.scheduler = EulerDiscreteScheduler(beta_end=0.02)
    assert pipe.engine is not e0 and pipe.engine.scheduler is pipe.scheduler
    from imagharmony_b200._lib import IHError
    with pytest.raises(IHError):
        pipe.to("cuda:1")


def test_step_invariant_buffers_are_per_shape(patched):
    """ADVICE r1 (high): K/V and add-embedding buffers a captured graph reads must survive a change of batch size.
    n=1 -> n=2 -> n=1 through one engine: every (processor, shape) keeps ONE buffer address, and the trajectory of the
    second n=1 call equals the first."""
    from imagharmony_b200.config import TINY
    from oracle.scheduler_ref import euler_tables, prepare_latents
    native, _ = _build(TINY, 6)
    T, lat = 2, 8
    _, _, ins = euler_tables(T)
    eng = _fp32_engine(native)
    procs = [p for p in native.attn_processors.values() if hasattr(p, "to_k_ip")]

    def run(n, seeds):
        latents = prepare_latents(n, 4, lat, lat, seeds, ins, dtype=torch.float32)
        _, ehs, te, tid = _inputs(TINY, n, lat, seed=11)
        with _Empty32():
            return eng.run(latents, ehs[n:], ehs[:n], te[n:], te[:n], tid[:n], T)
    a = run(1, [3])
    ptr1 = [p._kv[1].data_ptr() for p in procs]
    aug1 = native._aug[1].data_ptr()
    run(2, [3, 4])
    ptr2 = [p._kv[1].data_ptr() for p in procs]
    assert all(x != y for x, y in zip(ptr1, ptr2)) and native._aug[1].data_ptr() != aug1
    b = run(1, [3])
    assert [p._kv[1].data_ptr() for p in procs] == ptr1 and native._aug[1].data_ptr() == aug1
    assert torch.equal(a, b)
    epoch = native.graph_epoch
    native.finalize()
    assert native.graph_epoch > epoch and all(not p._kv_bufs for p in procs)


def test_harmony_attention_groups_text_rows_per_image(patched):
    """ADVICE r1 (medium): encode_prompt(extra_text, num_images_per_prompt=n) returns rows [a,a,b,b]; image i must attend
    to ITS text (the reference's Cross_Attention view(B, -1, D) groups [a,a],[b,b]) -- checked against the oracle
    restatement of train.py:243-266 that is pinned to the reference class."""
    from imagharmony_b200 import adapter as N
    from imagharmony_b200.config import HARMONY_TINY as h
    from imagharmony_b200.weights import random_state_dict, shapes_of
    from oracle.adapter_ref import HarmonyAttentionRef
    kw = dict(image_hidden_size=h.image_hidden_size, text_context_dim=h.text_context_dim, inter_dim=h.inter_dim,
              cross_heads=h.cross_heads, reshape_blocks=h.reshape_blocks, cross_value_dim=h.cross_value_dim)
    ha = N.HarmonyAttention(fusion_method="cross_attention", **kw)
    sd = {k: v.float() for k, v in random_state_dict(shapes_of(ha), 12).items()}
    ha.load_state_dict(sd)
    ref = HarmonyAttentionRef(**kw)
    ref.load_state_dict(sd)
    g = torch.Generator().manual_seed(2)
    img = torch.randn(2, h.image_hidden_size, generator=g)
    ta, tb = torch.randn(1, 7, h.text_context_dim, generator=g), torch.randn(1, 7, h.text_context_dim, generator=g)
    text = torch.cat([ta, ta, tb, tb])                       # num_samples = 2 copies per image, copies adjacent
    with torch.no_grad():
        want = ref(text, img)
        got = ha(text, img)
    assert torch.allclose(got, want, rtol=1e-4, atol=1e-5), (got - want).abs().max()
    # image 1 really uses text b (a wrong grouping -- text[:B] -- gives image 1 the text of image 0)
    with torch.no_grad():
        wrong = ref(torch.cat([ta, ta]), img)
    assert (wrong[1] - want[1]).abs().max() > 1e-3


def test_attention_map_hooks_match_oracle_and_reference_utils(patched):
    """ip_adapter/utils.py diagnostics (utils.py:6-79): register_cross_attention_hook switches `attn_map` on in the active
    IP processors and collects it per attn2 module; the maps equal the oracle processors' (attention_processor.py:443-444,
    pinned against the reference class in oracle/check_against_reference.py); get_net_attn_map / attnmaps2images equal
    the reference's own functions on the maps stored in tests/golden/reference_helpers.pt."""
    import os
    import numpy as np
    from imagharmony_b200.config import TINY
    from ip_adapter import utils
    native, ref = _build(TINY, 4)
    utils.attn_maps.clear()
    epoch = native.graph_epoch
    assert utils.register_cross_attention_hook(native) is native
    assert native.graph_epoch == epoch + 1                            # graphs captured without the maps are stale
    active = {}
    for name, proc in ref.attn_processors.items():
        if getattr(proc, "skip", True) is False:
            proc.keep_attn_map = True
            active[name[:-len(".processor")]] = proc
    assert active
    sample, ehs, te, tid = _inputs(TINY, 1, 16)
    with torch.no_grad():
        ref(sample, 500.0, ehs, te, tid)
        native(sample, torch.full((2,), 500.0), ehs, te, tid)
    assert set(utils.attn_maps) == set(active)                       # skip=True layers produce no map
    for name, proc in active.items():
        got = utils.attn_maps[name]
        assert got.shape == proc.attn_map.shape and got.shape[0] == 2 and got.shape[-1] == TINY.num_ip_tokens
        # the native K/V cache is fp16 also on this fp32 stand-in path: fp16 rounding of k_ip, not fp32 round-off
        assert torch.allclose(got.float(), proc.attn_map, rtol=2e-3, atol=2e-3), (got.float() - proc.attn_map).abs().max()
        assert not hasattr(native.get_submodule(name).processor, "attn_map")      # moved out by the hook (utils.py:10-11)
    net = utils.get_net_attn_map((128, 128), batch_size=2)
    assert net.shape == (TINY.num_ip_tokens, 128, 128)
    assert torch.allclose(net.sum(dim=0), torch.ones(128, 128), atol=1e-5)         # softmax over the tokens, layer mean
    images = utils.attnmaps2images(net)
    assert len(images) == TINY.num_ip_tokens and images[0].size == (128, 128) and images[0].mode == "L"
    # the reference's own functions on stored maps (written by oracle/make_helper_goldens.py)
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_helpers.pt"), map_location="cpu")
    gold = gold["attn_maps"]
    utils.attn_maps.clear()
    utils.attn_maps.update(gold["maps"])
    s = gold["stride"]
    for neg in (False, True):
        net = utils.get_net_attn_map(gold["size"], 2, neg)
        assert torch.equal(net[:, ::s, ::s], gold[f"net_neg{int(neg)}"])
        if not neg:
            assert (np.stack([np.asarray(x) for x in utils.attnmaps2images(net)]) == gold["images"].numpy()).all()
    utils.attn_maps.clear()


def test_resampler_module_helpers(patched):
    """ip_adapter/resampler.py module-level helpers with the reference's names (resampler.py:13-31, 150-158): FeedForward
    keeps the reference's Sequential indices and computes LN -> Linear -> GELU -> Linear; reshape_tensor / masked_mean /
    FeedForward equal the reference's functions on the inputs stored in tests/golden/reference_helpers.pt."""
    import os
    import torch.nn.functional as F
    from ip_adapter import resampler as own
    ff = own.FeedForward(32, mult=2).float()
    assert list(ff.state_dict()) == ["0.weight", "0.bias", "1.weight", "3.weight"]          # resampler.py:15-20
    g = torch.Generator("cpu").manual_seed(0)
    with torch.no_grad():
        for prm in ff.parameters():
            prm.copy_(torch.randn(prm.shape, generator=g) * 0.2 + (1.0 if prm.ndim == 1 else 0.0))
    x = torch.randn(2, 5, 32, generator=g)
    want = F.linear(F.gelu(F.linear(F.layer_norm(x, (32,), ff[0].weight, ff[0].bias, ff[0].eps), ff[1].weight)), ff[3].weight)
    with torch.no_grad():
        got = ff(x)
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-5), (got - want).abs().max()
    t = torch.randn(3, 7, 24, generator=g)
    r = own.reshape_tensor(t, 4)
    assert r.shape == (3, 4, 7, 6) and torch.equal(r[1, 2, 5], t[1, 5, 12:18])
    mask = torch.rand(3, 7, generator=g) > 0.4
    # the reference's outputs for these inputs (written by oracle/make_helper_goldens.py)
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_helpers.pt"), map_location="cpu")
    gold = gold["resampler"]
    assert torch.equal(t, gold["t"]) and torch.equal(mask, gold["mask"]) and torch.equal(x, gold["x"])
    assert torch.equal(r, gold["reshape_tensor"])
    assert torch.equal(own.masked_mean(t, dim=1), gold["masked_mean"])
    assert torch.allclose(own.masked_mean(t, dim=1, mask=mask), gold["masked_mean_mask"])
    assert list(gold["ff_state"]) == list(ff.state_dict())                                   # same keys, same layout
    assert all(torch.equal(v, gold["ff_state"][k]) for k, v in ff.state_dict().items())
    assert torch.allclose(got, gold["ff_out"], rtol=1e-5, atol=1e-5)
