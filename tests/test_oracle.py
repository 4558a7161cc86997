"""CPU tests of the oracle itself: it must reproduce the golden vectors generated from the reference's own modules
(tests/golden/reference_vectors.pt, written by oracle/check_against_reference.py in the build container) and the
scheduler known-answer values of SURVEY.md appendix A.3."""
import os

import pytest
import torch

from imagharmony_b200.config import SDXL_BASE, TINY
from oracle import adapter_ref as A
from oracle.scheduler_ref import euler_tables, prepare_latents
from oracle.unet_ref import Attention, UNetRef

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.pt")


@pytest.fixture(scope="module")
def gold():
    from oracle.check_against_reference import load_golden
    return load_golden(GOLDEN)


def test_ip_attn_processor_matches_reference(gold):
    for skip in (0, 1):
        g = gold[f"ipattn_skip{skip}"]
        C, D = g["hidden"].shape[-1], g["ehs"].shape[-1]
        attn = Attention(C, g["heads"], D)
        attn.load_state_dict(g["attn"])
        proc = A.IPAttnProcessorRef(C, D, scale=g["scale"], num_tokens=g["num_tokens"], skip=bool(skip))
        proc.load_state_dict(g["proc"])
        out = proc(attn, g["hidden"], encoder_hidden_states=g["ehs"])
        assert torch.allclose(out, g["out"], rtol=1e-5, atol=1e-5)


def test_skip_processor_equals_text_only_cross_attention(gold):
    """skip=True still drops the last num_tokens encoder tokens (attention_processor.py:402-406,430)."""
    g = gold["ipattn_skip1"]
    C, D = g["hidden"].shape[-1], g["ehs"].shape[-1]
    attn = Attention(C, g["heads"], D)
    attn.load_state_dict(g["attn"])
    ref = A.SelfAttnProcessorRef()(attn, g["hidden"], encoder_hidden_states=g["ehs"][:, :-g["num_tokens"]])
    assert torch.allclose(ref, g["out"], rtol=1e-5, atol=1e-5)


def test_self_attn_processor_matches_reference(gold):
    g = gold["selfattn"]
    attn = Attention(g["hidden"].shape[-1], g["heads"])
    attn.load_state_dict(g["attn"])
    out = A.SelfAttnProcessorRef()(attn, g["hidden"])
    assert torch.allclose(out, g["out"], rtol=1e-5, atol=1e-5)


def test_harmony_imageproj_resampler_match_reference(gold):
    g = gold["harmony"]
    ha = A.HarmonyAttentionRef(**g["kwargs"])
    ha.load_state_dict(g["state"])
    assert torch.allclose(ha(g["text"], g["image"]), g["out"], rtol=1e-5, atol=1e-5)
    g = gold["imageproj"]
    ip = A.ImageProjRef(128, 64, 4)
    ip.load_state_dict(g["state"])
    assert torch.allclose(ip(g["image"]), g["out"], rtol=1e-5, atol=1e-5)
    # uncond tokens = image_proj_model(zeros) = LayerNorm(bias) (ip_adapter.py:176): a per-model constant
    z = ip(torch.zeros_like(g["image"]))
    assert torch.allclose(z, ip.norm(ip.proj.bias.reshape(1, 4, 128)), atol=1e-6)
    g = gold["resampler"]
    r = A.ResamplerRef(**g["kwargs"])
    r.load_state_dict(g["state"])
    out = r(g["x"])
    assert out.shape == (2, 12, 160)      # the reference's only assertion (ip_adapter/test_resampler.py:40), scaled
    assert torch.allclose(out, g["out"], rtol=1e-5, atol=1e-5)


def test_scheduler_known_answers():
    kat = {50: ((13.1204, 11.6761, 10.4250), 13.15847), 30: ((11.4769, 9.5436, 8.0043), 11.52033),
           20: ((11.0283, 8.3907, 6.5064), 11.07358), 4: ((4.1167, 1.6237, 0.6984), 4.23641)}
    for T, (sig3, ins) in kat.items():
        ts, sig, init = euler_tables(T)
        assert len(ts) == T and len(sig) == T + 1 and sig[-1] == 0.0
        assert abs(sig[-2] - 0.04131) < 1e-4
        for a, b in zip(sig[:3], sig3):
            assert abs(a - b) < 2e-4
        assert abs(init - ins) < 1e-4
    assert list(euler_tables(50)[0][:3]) == [981.0, 961.0, 941.0]
    assert list(euler_tables(4)[0]) == [751.0, 501.0, 251.0, 1.0]


def test_latents_are_placement_invariant():
    a = prepare_latents(3, 4, 8, 8, [5, 6, 7], 2.0)
    b = prepare_latents(1, 4, 8, 8, [6], 2.0)
    assert torch.equal(a[1:2], b)


def test_unet_ref_structure():
    with torch.device("meta"):
        m = UNetRef(SDXL_BASE)
    n = sum(p.numel() for p in m.parameters())
    assert abs(n - 2.567e9) < 5e6                       # SDXL-base UNet
    names = list(m.attn_processors.keys())
    assert len(names) == 140
    assert names[0] == "down_blocks.1.attentions.0.transformer_blocks.0.attn1.processor"
    active = [i for i, nm in enumerate(names) if SDXL_BASE.ip_target_substring in nm and nm.endswith("attn2.processor")]
    assert active == list(range(29, 48, 2))             # SURVEY.md appendix A.1: ip_adapter.bin indices of the 10 IP layers
    assert names[-1].startswith("mid_block")            # down -> up -> mid registration order
    sd = m.state_dict()
    assert sd["up_blocks.0.resnets.2.conv1.weight"].shape == (1280, 1920, 3, 3)
    assert sd["up_blocks.2.resnets.0.conv_shortcut.weight"].shape == (320, 960, 1, 1)
    assert sd["add_embedding.linear_1.weight"].shape == (1280, 2816)


def test_unet_ref_tiny_forward_runs():
    torch.manual_seed(0)
    m = UNetRef(TINY).eval()
    A.install_processors(m, TINY)
    with torch.no_grad():
        out = m(torch.randn(2, 4, 16, 16), 500.0, torch.randn(2, 9 + 4, TINY.cross_attention_dim),
                torch.randn(2, TINY.pooled_embed_dim), torch.tensor([[128., 128, 0, 0, 128, 128]] * 2))
    assert out.shape == (2, 4, 16, 16) and torch.isfinite(out).all()


def test_oracle_matches_reference_at_real_shapes():
    """The oracle restatement against the reference's own classes at the REAL shapes (tests/golden/
    reference_real_shapes.pt, written by oracle/make_real_shape_goldens.py from /root/reference): the a1 layer
    (C 1280, 20 heads, N 1024, 77 + 4 tokens), HarmonyAttention at the shipped sizes, ImageProjModel."""
    import os
    from oracle import adapter_ref as A
    from oracle import make_real_shape_goldens as G
    from oracle.unet_ref import Attention
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_real_shapes.pt"), map_location="cpu")
    idx, (name, _, C, H, N, skip, stride) = 0, G.ATTN_CASES[0]
    assert name == "ipattn_a1" and not skip
    hidden, ehs = G.attn_case_inputs(idx, C, N)
    attn = Attention(C, H, G.CROSS_DIM)
    attn.load_state_dict({k: v.float() for k, v in G.state_for(attn, 300 + idx).items()})
    proc = A.IPAttnProcessorRef(C, G.CROSS_DIM, scale=G.IP_SCALE, num_tokens=G.N_IP, skip=False)
    proc.load_state_dict({k: v.float() for k, v in G.state_for(proc, 400 + idx).items()})
    with torch.no_grad():
        y = proc(attn, hidden.float(), encoder_hidden_states=ehs.float())
    assert (y[:, ::stride] - gold[name]["out"]).abs().max() < 2e-5
    ha = A.HarmonyAttentionRef(**G.HARMONY_KW)
    ha.load_state_dict({k: v.float() for k, v in G.state_for(ha, 500).items()})
    text, img = G.seeded((1, G.N_TEXT, G.CROSS_DIM), 501), G.seeded((1, 1280), 502)
    with torch.no_grad():
        assert (ha(text.float(), img.float()) - gold["harmony"]["out"]).abs().max() < 2e-5
        ip = A.ImageProjRef(G.CROSS_DIM, 1280, G.N_IP)
        ip.load_state_dict({k: v.float() for k, v in G.state_for(ip, 510).items()})
        assert (ip(img.float()) - gold["imageproj"]["out"]).abs().max() < 2e-5
