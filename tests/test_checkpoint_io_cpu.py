"""Checkpoint I/O (scope row f3): the reference's 3-key ip_adapter.bin layout (convert_bin.py:21-40), HarmonyAttention
hyper-parameters recovered from tensor shapes (test.py:9-15 re-types them by hand), and the safetensors snapshot layout
`from_pretrained` reads (test.py:68-72) -- on the CPU stand-in ops."""
import os

import torch

from test_wiring_cpu import patched  # noqa: F401  (fixture)


def test_split_ip_adapter_checkpoint_matches_convert_bin_layout():
    from imagharmony_b200.weights import split_ip_adapter_checkpoint
    flat = {"image_proj_model.proj.weight": torch.ones(2, 2), "image_proj_model.norm.bias": torch.zeros(2),
            "adapter_modules.1.to_k_ip.weight": torch.ones(3, 3), "adapter_modules.1.to_v_ip.weight": torch.ones(3, 3),
            "composed_modules.fc1.weight": torch.ones(4, 4), "unet.conv_in.weight": torch.ones(1)}
    got = split_ip_adapter_checkpoint(flat)
    assert set(got) == {"image_proj", "ip_adapter", "composed_adapter"}          # convert_bin.py:34-38
    assert set(got["image_proj"]) == {"proj.weight", "norm.bias"}
    assert set(got["ip_adapter"]) == {"1.to_k_ip.weight", "1.to_v_ip.weight"}
    assert set(got["composed_adapter"]) == {"fc1.weight"}                       # the frozen UNet keys are dropped


def _flat_training_checkpoint():
    g = torch.Generator("cpu").manual_seed(3)
    r = lambda *shape: torch.randn(*shape, generator=g)   # noqa: E731
    return {"image_proj_model.proj.weight": r(8, 4), "image_proj_model.proj.bias": r(8), "image_proj_model.norm.weight": r(4),
            "adapter_modules.1.to_k_ip.weight": r(6, 5), "adapter_modules.1.to_v_ip.weight": r(6, 5),
            "adapter_modules.3.to_k_ip.weight": r(6, 5), "composed_modules.fc1.weight": r(7, 3), "composed_modules.ln.bias": r(7),
            "unet.conv_in.weight": r(2, 2, 3, 3)}


def test_convert_bin_tool(tmp_path, capsys):
    """convert_bin.convert_checkpoint_to_ip_adapter: the reference tool's contract (convert_bin.py:5-49) -- True + a 3-key
    file, False (and no file) for a missing source or a checkpoint without the three prefixes."""
    import convert_bin
    flat = _flat_training_checkpoint()
    src, dst = tmp_path / "pytorch_model.bin", tmp_path / "ip_adapter.bin"
    torch.save(flat, src)
    assert convert_bin.convert_checkpoint_to_ip_adapter(str(src), str(dst)) is True
    got = torch.load(dst, map_location="cpu")
    assert list(got) == ["image_proj", "ip_adapter", "composed_adapter"]           # convert_bin.py:34-38
    assert list(got["ip_adapter"]) == ["1.to_k_ip.weight", "1.to_v_ip.weight", "3.to_k_ip.weight"]   # source order kept
    for part, prefix in (("image_proj", "image_proj_model."), ("ip_adapter", "adapter_modules."),
                         ("composed_adapter", "composed_modules.")):
        for k, v in got[part].items():
            assert torch.equal(v, flat[prefix + k])
    assert sum(len(v) for v in got.values()) == len(flat) - 1                       # the frozen UNet key is dropped
    assert convert_bin.convert_checkpoint_to_ip_adapter(str(tmp_path / "absent.bin"), str(tmp_path / "x.bin")) is False
    torch.save({"unet.conv_in.weight": torch.ones(1)}, tmp_path / "other.bin")
    assert convert_bin.convert_checkpoint_to_ip_adapter(str(tmp_path / "other.bin"), str(tmp_path / "y.bin")) is False
    (tmp_path / "garbage.bin").write_bytes(b"not a checkpoint")
    assert convert_bin.convert_checkpoint_to_ip_adapter(str(tmp_path / "garbage.bin"), str(tmp_path / "z.bin")) is False
    assert not any((tmp_path / n).exists() for n in ("x.bin", "y.bin", "z.bin"))
    # command line: a directory of checkpoint-* folders
    os.makedirs(tmp_path / "run" / "checkpoint-100")
    torch.save(flat, tmp_path / "run" / "checkpoint-100" / "pytorch_model.bin")
    assert convert_bin._main([str(tmp_path / "run")]) == 0
    assert (tmp_path / "run" / "checkpoint-100" / "ip_adapter.bin").exists()
    capsys.readouterr()


def test_convert_bin_tool_agrees_with_the_reference_tool(tmp_path, capsys):
    """The reference's own converter and ours write the same file for the same training checkpoint (the reference's
    output is tests/golden/reference_helpers.pt, written by oracle/make_helper_goldens.py)."""
    import convert_bin
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_helpers.pt"), map_location="cpu")
    src = tmp_path / "pytorch_model.bin"
    torch.save(gold["convert_bin"]["checkpoint"], src)
    assert convert_bin.convert_checkpoint_to_ip_adapter(str(src), str(tmp_path / "own.bin")) is True
    a, b = gold["convert_bin"]["converted"], torch.load(tmp_path / "own.bin", map_location="cpu")
    assert list(a) == list(b)
    for part in a:
        assert list(a[part]) == list(b[part])
        assert all(torch.equal(a[part][k], b[part][k]) for k in a[part])
    capsys.readouterr()


def test_infer_harmony_dims_from_shapes():
    from imagharmony_b200.config import HARMONY_DEFAULT as h
    from imagharmony_b200.weights import infer_harmony_dims, shapes_of
    from train import HarmonyAttention
    with torch.device("meta"):
        ha = HarmonyAttention(image_hidden_size=h.image_hidden_size, text_context_dim=h.text_context_dim,
                              inter_dim=h.inter_dim, cross_heads=h.cross_heads, reshape_blocks=h.reshape_blocks,
                              cross_value_dim=h.cross_value_dim, scale=1.0, fusion_method="cross_attention")
    shapes = {k: torch.empty(v, device="meta") for k, v in shapes_of(ha).items()}
    d = infer_harmony_dims(shapes)
    assert d["image_hidden_size"] == h.image_hidden_size and d["text_context_dim"] == h.text_context_dim
    assert d["inter_dim"] == h.inter_dim and d["reshape_blocks"] == h.reshape_blocks
    assert d["heads_times_value_dim"] == h.cross_heads * h.cross_value_dim          # 8 x 64 (test.py:12-14)


def test_from_pretrained_reads_diffusers_snapshot_layout(patched, tmp_path):  # noqa: F811
    """<path>/unet/diffusion_pytorch_model.safetensors + <path>/vae/... with diffusers key names (a full AutoencoderKL
    checkpoint also carries encoder.* / quant_conv.* keys, which the decoder ignores) -> pipeline -> PIL image."""
    from safetensors.torch import save_file
    from imagharmony_b200.config import TINY, TINY_VAE
    from imagharmony_b200.unet import UNet2DConditionModel
    from imagharmony_b200.vae import AutoencoderKLDecoder
    from imagharmony_b200.weights import random_state_dict, shapes_of
    from ip_adapter.custom_pipelines import StableDiffusionXLCustomPipeline
    with torch.device("meta"):
        ushapes = shapes_of(UNet2DConditionModel(TINY))
        vshapes = shapes_of(AutoencoderKLDecoder(TINY_VAE))
    os.makedirs(tmp_path / "unet")
    os.makedirs(tmp_path / "vae")
    usd = random_state_dict(ushapes, 1)
    vsd = random_state_dict(vshapes, 2)
    vsd_full = dict(vsd)
    vsd_full["encoder.conv_in.weight"] = torch.zeros(8, 3, 3, 3, dtype=torch.float16)        # ignored by the decoder
    vsd_full["quant_conv.weight"] = torch.zeros(8, 8, 1, 1, dtype=torch.float16)
    save_file({k: v.contiguous() for k, v in usd.items()}, str(tmp_path / "unet" / "diffusion_pytorch_model.safetensors"))
    save_file({k: v.contiguous() for k, v in vsd_full.items()}, str(tmp_path / "vae" / "diffusion_pytorch_model.safetensors"))
    pipe = StableDiffusionXLCustomPipeline.from_pretrained(str(tmp_path), torch_dtype=torch.float16, add_watermarker=False,
                                                           device="cpu", cfg=TINY, vae_cfg=TINY_VAE)
    assert pipe.vae is not None and pipe.unet.config is TINY
    got = pipe.unet.state_dict()
    assert all(torch.equal(got[k], usd[k]) for k in usd)
    pipe.enable_vae_tiling()
    assert pipe.vae.use_tiling
    out = pipe(prompt="lions", negative_prompt="blurry", num_inference_steps=1, height=64, width=64,
               generator=torch.Generator("cpu").manual_seed(0))
    img = out.images[0]
    assert img.size == (64, 64) and img.mode == "RGB"
    # a snapshot without vae/ gives a pipeline that can only return latents
    os.rename(tmp_path / "vae", tmp_path / "vae_off")
    pipe2 = StableDiffusionXLCustomPipeline.from_pretrained(str(tmp_path), device="cpu", cfg=TINY)
    assert pipe2.vae is None
    lat = pipe2(prompt="lions", num_inference_steps=1, height=64, width=64, output_type="latent",
                generator=torch.Generator("cpu").manual_seed(0)).images
    assert lat.shape == (1, 4, 8, 8)
