"""ORACLE tooling (runs only in the build container, where /root/reference exists).

Pins the restatements in oracle/adapter_ref.py against the reference's own modules, imported from
/root/reference BY FILE PATH (the package `ip_adapter` there cannot be imported: ip_adapter.py:10 needs the missing
module tutorial_train_sdxl_ori, and diffusers/accelerate are absent -> stubbed in sys.modules), and writes the
golden input/output vectors the committed tests use:  tests/golden/reference_vectors.pt

    python -m oracle.check_against_reference        # verify + (re)generate the fixture

Parameters are not stored: the fixture keeps each module's recipe -- its state-dict key/shape list as the reference class
defines it, and a seed for `imagharmony_b200.weights.random_state_dict` -- and `load_golden()` expands it.

Nothing under tests/ with the `gpu` mark, smoke() or bench.py reads /root/reference.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types
from unittest.mock import MagicMock

import torch

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_vectors.pt")


def _load(path: str, name: str):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def materialize(recipe: dict) -> dict:
    """{"seed", "shapes"} -> fp32 state dict with exactly the stored keys (fp16-representable values, CPU generator)."""
    from imagharmony_b200.weights import random_state_dict
    return {k: v.float() for k, v in random_state_dict(recipe["shapes"], recipe["seed"]).items()}


def load_golden(path: str = GOLDEN) -> dict:
    """The fixture with every parameter recipe expanded into its state dict."""
    gold = torch.load(path, map_location="cpu")
    for case in gold.values():
        for key, val in case.items():
            if isinstance(val, dict) and set(val) == {"seed", "shapes"}:
                case[key] = materialize(val)
    return gold


def load_reference_modules():
    import torchvision  # noqa: F401  (real one is present)
    import transformers  # noqa: F401  (must be imported before accelerate is stubbed)
    from transformers import (CLIPImageProcessor, CLIPTextModel, CLIPTextModelWithProjection,  # noqa: F401
                              CLIPTokenizer, CLIPVisionModelWithProjection)
    for m in ["diffusers", "diffusers.models", "diffusers.models.attention_processor", "diffusers.pipelines",
              "diffusers.pipelines.controlnet", "diffusers.pipelines.stable_diffusion_xl",
              "diffusers.pipelines.stable_diffusion_xl.pipeline_stable_diffusion_xl", "accelerate",
              "accelerate.logging", "accelerate.utils", "tutorial_train_sdxl_ori"]:
        if m not in sys.modules:
            sys.modules[m] = MagicMock()
    ap = _load(os.path.join(REF, "ip_adapter", "attention_processor.py"), "ref_attention_processor")
    rs = _load(os.path.join(REF, "ip_adapter", "resampler.py"), "ref_resampler")
    # train.py does `from ip_adapter.attention_processor import Cross_Attention` and `from shared_models import ...`
    pkg = types.ModuleType("ip_adapter")
    pkg.__path__ = []
    sys.modules["ip_adapter"] = pkg
    sys.modules["ip_adapter.attention_processor"] = ap
    sys.modules["ip_adapter.resampler"] = rs
    sys.modules["ip_adapter.utils"] = _load(os.path.join(REF, "ip_adapter", "utils.py"), "ref_utils")
    sys.modules["shared_models"] = _load(os.path.join(REF, "shared_models.py"), "ref_shared_models")
    sys.modules["baseline"] = _load(os.path.join(REF, "baseline.py"), "ref_baseline")
    sys.path.insert(0, REF)
    try:
        tr = _load(os.path.join(REF, "train.py"), "ref_train")
    finally:
        sys.path.remove(REF)
    return ap, rs, tr


def main():
    import contextlib
    import io

    sys.path.insert(0, ROOT)
    ap, rs, tr = load_reference_modules()
    # the reference modules shadow our own `ip_adapter` package name in sys.modules; import ours explicitly by path
    from imagharmony_b200.weights import shapes_of
    from oracle import adapter_ref as A
    from oracle.unet_ref import Attention

    torch.manual_seed(0)
    out = {}
    report = []

    def seed_params(module, seed):
        recipe = {"seed": seed, "shapes": shapes_of(module)}
        module.load_state_dict(materialize(recipe))
        return recipe

    def cmp(name, a, b, tol=1e-5):
        err = (a - b).abs().max().item()
        report.append((name, err))
        assert err <= tol, (name, err)

    # ---- attention processors (mock attn = the oracle's Attention shell) -----------------------------------------
    B, N, C, H, D, L, NT = 2, 48, 128, 2, 96, 13, 4
    attn = Attention(C, H, D)
    attn_recipe = seed_params(attn, 1)
    hidden = torch.randn(B, N, C)
    ehs = torch.randn(B, L, D)
    for skip in (False, True):
        ref = ap.IPAttnProcessor2_0(C, D, scale=0.7, num_tokens=NT, skip=skip)
        proc_recipe = seed_params(ref, 2)
        mine = A.IPAttnProcessorRef(C, D, scale=0.7, num_tokens=NT, skip=skip, keep_attn_map=True)
        mine.load_state_dict(ref.state_dict())
        y_ref = ref(attn, hidden, encoder_hidden_states=ehs)
        y = mine(attn, hidden, encoder_hidden_states=ehs)
        cmp(f"IPAttnProcessor2_0 skip={skip}", y, y_ref)
        if not skip:
            cmp("attn_map", mine.attn_map, ref.attn_map)
        out[f"ipattn_skip{int(skip)}"] = {"attn": attn_recipe, "proc": proc_recipe, "hidden": hidden,
                                          "ehs": ehs, "scale": 0.7, "num_tokens": NT, "heads": H, "out": y_ref.detach()}
    self_attn = Attention(C, H)
    self_recipe = seed_params(self_attn, 3)
    y_ref = ap.AttnProcessor2_0()(self_attn, hidden)
    cmp("AttnProcessor2_0", A.SelfAttnProcessorRef()(self_attn, hidden), y_ref)
    out["selfattn"] = {"attn": self_recipe, "hidden": hidden, "heads": H, "out": y_ref.detach()}

    # ---- HarmonyAttention / Cross_Attention / ImageProjModel ----------------------------------------------------
    kw = dict(image_hidden_size=64, text_context_dim=128, inter_dim=256, cross_heads=4, reshape_blocks=4,
              cross_value_dim=16, scale=0.5)
    with contextlib.redirect_stdout(io.StringIO()):       # the reference prints inside __init__/forward (train.py:209,258,260)
        ha_ref = tr.HarmonyAttention(fusion_method="cross_attention", **kw)
    ha_recipe = seed_params(ha_ref, 4)
    ha = A.HarmonyAttentionRef(**kw)
    ha.load_state_dict(ha_ref.state_dict())
    text, img = torch.randn(1, 9, 128), torch.randn(1, 64)
    with contextlib.redirect_stdout(io.StringIO()):
        y_ref = ha_ref(text, img)
    cmp("HarmonyAttention", ha(text, img), y_ref)
    out["harmony"] = {"kwargs": kw, "state": ha_recipe, "text": text, "image": img, "out": y_ref.detach()}
    # num_samples > 1 folds the text batch into the key axis (SURVEY C.11): same result as one copy
    with contextlib.redirect_stdout(io.StringIO()):
        y3 = ha_ref(text.repeat(3, 1, 1), img)
    cmp("HarmonyAttention text-batch folding", y3, y_ref, tol=1e-5)

    ip_ref = tr.ImageProjModel(cross_attention_dim=128, clip_embeddings_dim=64, clip_extra_context_tokens=4)
    ip_recipe = seed_params(ip_ref, 5)
    ip = A.ImageProjRef(128, 64, 4)
    ip.load_state_dict(ip_ref.state_dict())
    cmp("ImageProjModel", ip(img), ip_ref(img))
    out["imageproj"] = {"state": ip_recipe, "image": img, "out": ip_ref(img).detach()}

    # ---- Resampler (the reference's own shape test config, ip_adapter/test_resampler.py:18-40, shrunk) ------------
    rkw = dict(dim=128, depth=2, dim_head=64, heads=2, num_queries=8, embedding_dim=96, output_dim=160, ff_mult=2,
               max_seq_len=33, apply_pos_emb=True, num_latents_mean_pooled=4)
    r_ref = rs.Resampler(**rkw)
    r_recipe = seed_params(r_ref, 6)
    r = A.ResamplerRef(**rkw)
    missing = r.load_state_dict(r_ref.state_dict(), strict=True)
    x = torch.randn(2, 33, 96)
    y_ref = r_ref(x)
    assert y_ref.shape == (2, 12, 160)          # the reference's only assertion (test_resampler.py:40), scaled down
    cmp("Resampler", r(x), y_ref)
    out["resampler"] = {"kwargs": rkw, "state": r_recipe, "x": x, "out": y_ref.detach()}

    for name, err in report:
        print(f"{name:45s} max|diff| = {err:.3e}")
    os.makedirs(os.path.dirname(GOLDEN), exist_ok=True)
    out = {k: {kk: (vv.detach().clone() if torch.is_tensor(vv) else
                    ({k3: v3.detach().clone() for k3, v3 in vv.items()} if isinstance(vv, dict) and vv and
                     torch.is_tensor(next(iter(vv.values()))) else vv))
               for kk, vv in v.items()} for k, v in out.items()}
    torch.save(out, GOLDEN)
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes")


if __name__ == "__main__":
    main()
