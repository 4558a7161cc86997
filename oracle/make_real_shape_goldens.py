"""ORACLE tooling (runs only in the build container, where /root/reference exists).

Golden vectors at the REAL SDXL / IMAGHarmony shapes, produced by the reference's OWN classes (imported from
/root/reference by file path, see oracle/check_against_reference.py) in fp32 on fp16-representable parameters and
inputs.  Parameters and inputs are not stored -- they are regenerated from seeds with
`imagharmony_b200.weights.random_state_dict` / seeded `torch.randn` (deterministic CPU generators) -- only the
reference outputs (sub-sampled rows for the big ones) are committed:  tests/golden/reference_real_shapes.pt

    python -m oracle.make_real_shape_goldens        # verify the restatement at these shapes + (re)generate the fixture

Cases (reference file:line):
  ipattn_a1      IPAttnProcessor2_0 skip=False  C=1280 H=20 N=1024 L=77+4 D=2048   attention_processor.py:364-465
  ipattn_a2_l1   IPAttnProcessor2_0 skip=True   C=640  H=10 N=4096 L=77+4          (level-1 layers, :402-411)
  ipattn_a2_l2   IPAttnProcessor2_0 skip=True   C=1280 H=20 N=1024
  selfattn_l2    AttnProcessor2_0               C=1280 H=20 N=1024                 :258-332
  selfattn_l1    AttnProcessor2_0               C=640  H=10 N=4096
  harmony        HarmonyAttention 1280/2048/2560/8 heads/8 blocks/64               train.py:188-266
  imageproj      ImageProjModel 1280 -> 4 x 2048                                   ip_adapter.py:28-48
  resampler      Resampler PlusXL config (dim 1280, depth 4, 20 x 64, 16 queries, 1664 -> 2048)   resampler.py:81-147
"""
from __future__ import annotations

import contextlib
import io
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_real_shapes.pt")

# (name, kind, C, heads, N, skip, row stride of the stored sub-sample: 16 rows per image keeps the fixture under 1 MB)
ATTN_CASES = [
    ("ipattn_a1", "ip", 1280, 20, 1024, False, 64),
    ("ipattn_a2_l1", "ip", 640, 10, 4096, True, 256),
    ("ipattn_a2_l2", "ip", 1280, 20, 1024, True, 64),
    ("selfattn_l2", "self", 1280, 20, 1024, None, 64),
    ("selfattn_l1", "self", 640, 10, 4096, None, 256),
]
HARMONY_KW = dict(image_hidden_size=1280, text_context_dim=2048, inter_dim=2560, cross_heads=8, reshape_blocks=8,
                  cross_value_dim=64, scale=1.0)
RESAMPLER_KW = dict(dim=1280, depth=4, dim_head=64, heads=20, num_queries=16, embedding_dim=1664, output_dim=2048,
                    ff_mult=4)
CROSS_DIM, N_TEXT, N_IP, BATCH, IP_SCALE = 2048, 77, 4, 2, 0.7


def seeded(shape, seed, scale=1.0):
    """fp16-representable N(0, scale^2) tensor from a CPU generator (what the tests regenerate)."""
    return (torch.randn(shape, generator=torch.Generator("cpu").manual_seed(seed)) * scale).half()


def attn_case_inputs(idx: int, C: int, N: int):
    hidden = seeded((BATCH, N, C), 100 + idx, scale=3.0)      # scores ~ N(0, 3^2): a peaked softmax, not a mean
    ehs = seeded((BATCH, N_TEXT + N_IP, CROSS_DIM), 200 + idx)
    return hidden, ehs


def state_for(module: torch.nn.Module, seed: int):
    from imagharmony_b200.weights import random_state_dict, shapes_of
    return random_state_dict(shapes_of(module), seed)          # fp16 values, CPU generator


def main():
    sys.path.insert(0, ROOT)
    from oracle.check_against_reference import load_reference_modules
    ap, rs, tr = load_reference_modules()
    from oracle import adapter_ref as A
    from oracle.unet_ref import Attention

    out, report = {}, []

    def cmp(name, mine, ref, tol):
        err = (mine - ref).abs().max().item()
        report.append((name, err, ref.abs().max().item()))
        assert err <= tol, (name, err)

    with torch.no_grad():
        for idx, (name, kind, C, H, N, skip, stride) in enumerate(ATTN_CASES):
            hidden, ehs = attn_case_inputs(idx, C, N)
            if kind == "ip":
                attn = Attention(C, H, CROSS_DIM)
                attn.load_state_dict({k: v.float() for k, v in state_for(attn, 300 + idx).items()})
                ref = ap.IPAttnProcessor2_0(C, CROSS_DIM, scale=IP_SCALE, num_tokens=N_IP, skip=skip)
                ref.load_state_dict({k: v.float() for k, v in state_for(ref, 400 + idx).items()})
                y_ref = ref(attn, hidden.float(), encoder_hidden_states=ehs.float())
                mine = A.IPAttnProcessorRef(C, CROSS_DIM, scale=IP_SCALE, num_tokens=N_IP, skip=skip)
                mine.load_state_dict(ref.state_dict())
                cmp(name, mine(attn, hidden.float(), encoder_hidden_states=ehs.float()), y_ref, 2e-5)
            else:
                attn = Attention(C, H)
                attn.load_state_dict({k: v.float() for k, v in state_for(attn, 300 + idx).items()})
                y_ref = ap.AttnProcessor2_0()(attn, hidden.float())
                cmp(name, A.SelfAttnProcessorRef()(attn, hidden.float()), y_ref, 2e-5)
            out[name] = {"out": y_ref[:, ::stride].clone(), "stride": stride}

        with contextlib.redirect_stdout(io.StringIO()):       # the reference prints in __init__/forward (train.py:209,258,260)
            ha_ref = tr.HarmonyAttention(fusion_method="cross_attention", **HARMONY_KW)
        ha_ref.load_state_dict({k: v.float() for k, v in state_for(ha_ref, 500).items()})
        text, img = seeded((1, N_TEXT, CROSS_DIM), 501), seeded((1, 1280), 502)
        with contextlib.redirect_stdout(io.StringIO()):
            y_ref = ha_ref(text.float(), img.float())
        ha = A.HarmonyAttentionRef(**HARMONY_KW)
        ha.load_state_dict(ha_ref.state_dict())
        cmp("harmony", ha(text.float(), img.float()), y_ref, 2e-5)
        out["harmony"] = {"out": y_ref.clone()}

        ip_ref = tr.ImageProjModel(cross_attention_dim=CROSS_DIM, clip_embeddings_dim=1280, clip_extra_context_tokens=N_IP)
        ip_ref.load_state_dict({k: v.float() for k, v in state_for(ip_ref, 510).items()})
        y_ref = ip_ref(img.float())
        ipm = A.ImageProjRef(CROSS_DIM, 1280, N_IP)
        ipm.load_state_dict(ip_ref.state_dict())
        cmp("imageproj", ipm(img.float()), y_ref, 2e-5)
        out["imageproj"] = {"out": y_ref.clone()}

        r_ref = rs.Resampler(**RESAMPLER_KW)
        r_ref.load_state_dict({k: v.float() for k, v in state_for(r_ref, 520).items()})
        x = seeded((1, 257, 1664), 521)
        y_ref = r_ref(x.float())
        r = A.ResamplerRef(**RESAMPLER_KW)
        r.load_state_dict(r_ref.state_dict())
        cmp("resampler", r(x.float()), y_ref, 5e-5)
        out["resampler"] = {"out": y_ref.clone()}

    for name, err, mx in report:
        print(f"{name:16s} oracle restatement vs reference class: max|diff| = {err:.3e} (max|ref| {mx:.3e})")
    os.makedirs(os.path.dirname(GOLDEN), exist_ok=True)
    torch.save(out, GOLDEN)
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes")


if __name__ == "__main__":
    main()
