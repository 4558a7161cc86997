"""ORACLE tooling (runs only where the reference tree is on disk, see oracle/check_against_reference.py).

Outputs of the reference's host-side helpers on fixed inputs, for the CPU tests that hold our restatements to them:
  convert_bin    convert_checkpoint_to_ip_adapter on a small training checkpoint     convert_bin.py:5-49
  attn_maps      get_net_attn_map (both CFG halves) and attnmaps2images              ip_adapter/utils.py:22-79
  resampler      reshape_tensor, masked_mean, FeedForward                            ip_adapter/resampler.py:13-31,150-158
Inputs are stored with the outputs: tests/golden/reference_helpers.pt

    python -m oracle.make_helper_goldens
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_helpers.pt")
MAP_SIZE = (128, 128)
MAP_STRIDE = 4          # get_net_attn_map outputs are stored every 4th pixel per axis; the images in full


def training_checkpoint():
    g = torch.Generator("cpu").manual_seed(3)
    r = lambda *shape: torch.randn(*shape, generator=g)   # noqa: E731
    return {"image_proj_model.proj.weight": r(8, 4), "image_proj_model.proj.bias": r(8), "image_proj_model.norm.weight": r(4),
            "adapter_modules.1.to_k_ip.weight": r(6, 5), "adapter_modules.1.to_v_ip.weight": r(6, 5),
            "adapter_modules.3.to_k_ip.weight": r(6, 5), "composed_modules.fc1.weight": r(7, 3), "composed_modules.ln.bias": r(7),
            "unet.conv_in.weight": r(2, 2, 3, 3)}


def attention_maps():
    """[B=2 (CFG halves), heads, N, 4 tokens] softmax maps of two layers on the 16x16 and 8x8 grids of a 128^2 image."""
    g = torch.Generator("cpu").manual_seed(4)
    return {f"down_blocks.{i}.attentions.0.transformer_blocks.0.attn2": torch.randn(2, 2, n, 4, generator=g).mul(3).softmax(-1)
            for i, n in ((1, 256), (2, 64))}


def main():
    sys.path.insert(0, ROOT)
    from oracle.check_against_reference import REF, _load, load_reference_modules
    _, rs, _ = load_reference_modules()
    ru = sys.modules["ip_adapter.utils"]
    cb = _load(os.path.join(REF, "convert_bin.py"), "ref_convert_bin")
    out = {}

    flat = training_checkpoint()
    with tempfile.TemporaryDirectory() as d, contextlib.redirect_stdout(io.StringIO()):
        torch.save(flat, os.path.join(d, "pytorch_model.bin"))
        assert cb.convert_checkpoint_to_ip_adapter(os.path.join(d, "pytorch_model.bin"), os.path.join(d, "ip_adapter.bin"))
        converted = torch.load(os.path.join(d, "ip_adapter.bin"), map_location="cpu")
    out["convert_bin"] = {"checkpoint": flat, "converted": {k: dict(v) for k, v in converted.items()}}

    maps = attention_maps()
    ru.attn_maps.clear()
    ru.attn_maps.update(maps)
    nets = {neg: ru.get_net_attn_map(MAP_SIZE, 2, neg) for neg in (False, True)}
    images = np.stack([np.asarray(im) for im in ru.attnmaps2images(nets[False])])
    out["attn_maps"] = {"maps": maps, "size": MAP_SIZE, "stride": MAP_STRIDE, "images": torch.from_numpy(images),
                        **{f"net_neg{int(neg)}": v[:, ::MAP_STRIDE, ::MAP_STRIDE].clone() for neg, v in nets.items()}}

    g = torch.Generator("cpu").manual_seed(0)
    ff = rs.FeedForward(32, mult=2)
    with torch.no_grad():
        for prm in ff.parameters():
            prm.copy_(torch.randn(prm.shape, generator=g) * 0.2 + (1.0 if prm.ndim == 1 else 0.0))
    x = torch.randn(2, 5, 32, generator=g)
    t = torch.randn(3, 7, 24, generator=g)
    mask = torch.rand(3, 7, generator=g) > 0.4
    with torch.no_grad():
        out["resampler"] = {"ff_state": ff.state_dict(), "x": x, "t": t, "mask": mask, "ff_out": ff(x),
                            "reshape_tensor": rs.reshape_tensor(t, 4), "masked_mean": rs.masked_mean(t, dim=1),
                            "masked_mean_mask": rs.masked_mean(t, dim=1, mask=mask)}

    torch.save(out, GOLDEN)
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes")


if __name__ == "__main__":
    main()
