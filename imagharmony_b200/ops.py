"""One Python function per C-ABI entry point of libimagharmony_sm100.so (include/ih_api.h).

Tensors are torch CUDA fp16; PyTorch is only used for device memory and the current stream. No op has a
PyTorch/CPU fallback: a CPU tensor or a missing library raises.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import IHError, check

EPI_NONE, EPI_GEGLU, EPI_SILU, EPI_GELU, EPI_QUICK_GELU = 0, 1, 2, 4, 8


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, name: str, dtype=torch.float16) -> None:
    if not t.is_cuda:
        raise IHError(f"{name}: expected a CUDA tensor (the sm_100a path has no CPU fallback)")
    if t.dtype != dtype:
        raise IHError(f"{name}: expected dtype {dtype}, got {t.dtype}")


def _rows(t: torch.Tensor, name: str) -> int:
    """Row stride (elements) of a 2-D view whose last dim is contiguous."""
    if t.dim() != 2 or t.stride(1) != 1:
        raise IHError(f"{name}: expected a 2-D tensor with contiguous last dim, got shape {tuple(t.shape)} "
                      f"strides {t.stride()}")
    return t.stride(0)


def launch_count() -> int:
    return int(_lib.load().ih_launch_count())


def launch_count_reset() -> None:
    _lib.load().ih_launch_count_reset()


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *,
           residual: Optional[torch.Tensor] = None, rowbias: Optional[torch.Tensor] = None,
           rows_per_group: int = 0, geglu: bool = False, silu: bool = False, gelu: bool = False,
           out: Optional[torch.Tensor] = None, tile_n: int = 0, ln=None,
           stats_out: Optional[torch.Tensor] = None, quick_gelu: bool = False, alpha: float = 1.0) -> torch.Tensor:
    """out = epi(x @ w.T + bias + rowbias[row // rows_per_group]) + residual ; x [M,K], w [N,K] (nn.Linear layout).

    LayerNorm folding: `stats_out` (float32 [ceil(N/64), M, 2]) receives per-row / per-64-column (sum, sumsq) of the
    stored values; `ln=(stats, eps)` makes this GEMM consume RAW rows `x` with the gamma-scaled, row-centred weight and
    the constant vector of fold_layernorm (passed as `w`, `bias`) and apply rstd * acc + bias in the epilogue."""
    lib = _lib.load()
    _req(x, "x"); _req(w, "w")
    M, K = x.shape
    N = w.shape[0]
    if w.shape[1] != K or not w.is_contiguous():
        raise IHError(f"linear: weight must be contiguous [N,{K}], got {tuple(w.shape)}")
    n_out = N // 2 if geglu else N
    if out is None:
        out = torch.empty((M, n_out), dtype=torch.float16, device=x.device)
    ldr = _rows(residual, "residual") if residual is not None else 0
    ldrb = _rows(rowbias, "rowbias") if rowbias is not None else 0
    epi = ((EPI_GEGLU if geglu else 0) | (EPI_SILU if silu else 0) | (EPI_GELU if gelu else 0)
           | (EPI_QUICK_GELU if quick_gelu else 0))
    if alpha != 1.0:
        # out = epi(alpha * x w^T + bias) + residual (ih_gemm_scaled_f16: the VAE decoder's scaled residual stream)
        if ln is not None or stats_out is not None or rowbias is not None or tile_n:
            raise IHError("linear: alpha != 1 cannot be combined with ln / stats_out / rowbias / tile_n")
        rc = lib.ih_gemm_scaled_f16(x.data_ptr(), _rows(x, "x"), w.data_ptr(), _p(bias), _p(residual), ldr, out.data_ptr(),
                                    _rows(out, "out"), M, N, K, epi, float(alpha), _stream())
        check(rc, "ih_gemm_scaled_f16")
        return out
    if ln is None and stats_out is None:
        rc = lib.ih_gemm_f16(x.data_ptr(), _rows(x, "x"), w.data_ptr(), _p(bias), _p(rowbias), rows_per_group, ldrb,
                             _p(residual), ldr, out.data_ptr(), _rows(out, "out"), M, N, K, epi, tile_n, _stream())
        check(rc, "ih_gemm_f16")
        return out
    ln_stats = None
    ln_slabs, ln_eps = 0, 0.0
    if ln is not None:
        ln_stats, ln_eps = ln
        _req(ln_stats, "ln_stats", torch.float32)
        if ln_stats.dim() != 3 or ln_stats.shape[1] != M or ln_stats.shape[-1] != 2 or not ln_stats.is_contiguous():
            raise IHError("linear: ln statistics must be contiguous [slabs, M, 2]")
        if ln_stats.shape[0] != (K + 63) // 64:
            raise IHError(f"linear: ln statistics cover {ln_stats.shape[0]} slabs, K={K} needs {(K + 63) // 64}")
        ln_slabs = ln_stats.shape[0]
    if stats_out is not None:
        _req(stats_out, "stats_out", torch.float32)
        if tuple(stats_out.shape) != ((n_out + 63) // 64, M, 2) or not stats_out.is_contiguous():
            raise IHError(f"linear: stats_out must be contiguous float32 [{(n_out + 63) // 64}, {M}, 2]")
    rc = lib.ih_gemm_ln_f16(x.data_ptr(), _rows(x, "x"), w.data_ptr(), _p(bias), _p(rowbias), rows_per_group, ldrb,
                            _p(residual), ldr, out.data_ptr(), _rows(out, "out"), M, N, K, epi, tile_n, _p(ln_stats),
                            ln_slabs, float(ln_eps), _p(stats_out), _stream())
    check(rc, "ih_gemm_ln_f16")
    return out


PREFETCH_WEIGHTS = os.environ.get("IH_PREFETCH", "1") != "0"


def prefetch_next(w: Optional[torch.Tensor]) -> None:
    """Hint for the NEXT linear / conv3x3 call: while it runs, pull `w` (the weight of the launch after it) into L2."""
    if PREFETCH_WEIGHTS and w is not None and w.is_cuda:
        _lib.load().ih_gemm_prefetch_next(w.data_ptr(), w.numel() * w.element_size())


def fold_layernorm(w: torch.Tensor, bias: Optional[torch.Tensor], gamma: torch.Tensor, beta: torch.Tensor):
    """LayerNorm(x) @ w.T + bias == rstd(x) * (x @ w_c.T) + c with
       w_c[n, k] = w[n, k] gamma[k] - mean_k(w[n, :] gamma)   (rows centred: x @ w_c.T = (x - mean(x)) @ (w gamma).T)
       c[n]      = sum_k beta[k] w[n, k] + bias[n].
    Returns (w_c, c) in fp16 for ops.linear(x_raw, w_c, c, ln=(row statistics of x_raw, eps))."""
    w_g = w.double() * gamma.double()[None, :]
    w_c = (w_g - w_g.mean(dim=1, keepdim=True)).to(torch.float16).contiguous()
    c = w.double() @ beta.double()
    if bias is not None:
        c = c + bias.double()
    return w_c, c.to(torch.float16).contiguous()


def conv3x3(x: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor] = None, *,
            rowbias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None, stride: int = 1,
            out: Optional[torch.Tensor] = None, tile_n: int = 0, alpha: float = 1.0, shortcut=None) -> torch.Tensor:
    """3x3 conv, pad 1. x NHWC [B,H,W,Cin]; w_packed [Cout, 9*Cin] (see pack_conv3x3_weight); rowbias [B, >=Cout].
    `shortcut=(s0, s1 | None)`: fused 1x1 shortcut conv over the channel concat of the NHWC tensors s0 [, s1]; then
    w_packed is [Cout, 9*Cin + C(s0) + C(s1)] (3x3 taps followed by the shortcut weight), see ih_conv2d_shortcut_f16."""
    lib = _lib.load()
    _req(x, "x"); _req(w_packed, "w")
    B, H, W, Cin = x.shape
    Cout = w_packed.shape[0]
    if shortcut is not None:
        s0, s1 = shortcut
        c0, c1 = s0.shape[-1], (0 if s1 is None else s1.shape[-1])
        _req(s0, "shortcut[0]")
        if s1 is not None:
            _req(s1, "shortcut[1]")
        if (stride != 1 or residual is not None or alpha != 1.0 or tile_n or not x.is_contiguous() or not s0.is_contiguous()
                or (s1 is not None and not s1.is_contiguous()) or tuple(s0.shape[:3]) != (B, H, W)
                or (s1 is not None and tuple(s1.shape[:3]) != (B, H, W)) or not w_packed.is_contiguous()
                or w_packed.shape[1] != 9 * Cin + c0 + c1):
            raise IHError("conv3x3(shortcut=): stride 1, no residual / alpha / tile_n, contiguous NHWC sources of the same "
                          "spatial size and w_packed [Cout, 9*Cin + C0 + C1] required")
        if out is None:
            out = torch.empty((B, H, W, Cout), dtype=torch.float16, device=x.device)
        ldrb = _rows(rowbias, "rowbias") if rowbias is not None else 0
        rc = lib.ih_conv2d_shortcut_f16(x.data_ptr(), w_packed.data_ptr(), _p(bias), _p(rowbias), ldrb, s0.data_ptr(), c0,
                                        _p(s1), c1, out.data_ptr(), B, H, W, Cin, Cout, _stream())
        check(rc, "ih_conv2d_shortcut_f16")
        return out
    if not x.is_contiguous() or not w_packed.is_contiguous() or w_packed.shape[1] != 9 * Cin:
        raise IHError("conv3x3: x must be contiguous NHWC and w_packed [Cout, 9*Cin]")
    Ho, Wo = H // stride, W // stride
    if out is None:
        out = torch.empty((B, Ho, Wo, Cout), dtype=torch.float16, device=x.device)
    ldrb = _rows(rowbias, "rowbias") if rowbias is not None else 0
    if residual is not None and (not residual.is_contiguous() or residual.shape != out.shape):
        raise IHError("conv3x3: residual must be contiguous and shaped like the output")
    if alpha != 1.0:
        if rowbias is not None or tile_n:
            raise IHError("conv3x3: alpha != 1 cannot be combined with rowbias / tile_n")
        rc = lib.ih_conv2d_scaled_f16(x.data_ptr(), w_packed.data_ptr(), _p(bias), _p(residual), out.data_ptr(), B, H, W,
                                      Cin, Cout, stride, float(alpha), _stream())
        check(rc, "ih_conv2d_scaled_f16")
        return out
    rc = lib.ih_conv2d_f16(x.data_ptr(), w_packed.data_ptr(), _p(bias), _p(rowbias), ldrb, _p(residual),
                           out.data_ptr(), B, H, W, Cin, Cout, 3, stride, tile_n, _stream())
    check(rc, "ih_conv2d_f16")
    return out


def conv3x3_s2_padbr(x: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor] = None, *,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """conv3x3(F.pad(x, (0, 1, 0, 1)), stride=2) + bias: the VAE encoder's Downsample2D(padding=0).  x NHWC [B,H,W,Cin]
    (H, W even), w_packed [Cout, 9*Cin] (pack_conv3x3_weight); returns [B, H/2, W/2, Cout]."""
    lib = _lib.load()
    _req(x, "x"); _req(w_packed, "w")
    B, H, W, Cin = x.shape
    Cout = w_packed.shape[0]
    if not x.is_contiguous() or not w_packed.is_contiguous() or w_packed.shape[1] != 9 * Cin:
        raise IHError("conv3x3_s2_padbr: x must be contiguous NHWC and w_packed [Cout, 9*Cin]")
    if out is None:
        out = torch.empty((B, H // 2, W // 2, Cout), dtype=torch.float16, device=x.device)
    check(lib.ih_conv2d_s2_padbr_f16(x.data_ptr(), w_packed.data_ptr(), _p(bias), out.data_ptr(), B, H, W, Cin, Cout,
                                     _stream()), "ih_conv2d_s2_padbr_f16")
    return out


def image_im2col3x3(rgb_u8: torch.Tensor, kpad: int = 32, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 RGB NHWC [B, H, W, 3] -> A [B*H*W, kpad] of the normalised image 2 * (v / 255) - 1 (k = ci*9 + ky*3 + kx,
    zero padded): the VAE encoder's conv_in as a tensor-core GEMM straight from the PIL pixels."""
    lib = _lib.load()
    _req(rgb_u8, "rgb_u8", torch.uint8)
    B, H, W, C = rgb_u8.shape
    if C != 3 or not rgb_u8.is_contiguous():
        raise IHError("image_im2col3x3: contiguous uint8 RGB NHWC [B, H, W, 3] required")
    if out is None:
        out = torch.empty((B * H * W, kpad), dtype=torch.float16, device=rgb_u8.device)
    check(lib.ih_image_im2col3x3_u8(rgb_u8.data_ptr(), out.data_ptr(), B, H, W, kpad, _stream()), "ih_image_im2col3x3_u8")
    return out


def vae_sample_add_noise(moments: torch.Tensor, eps: Optional[torch.Tensor], noise: torch.Tensor, channels: int,
                         scaling_factor: float, sigma: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """img2img initial latents: moments NHWC [Bm, h, w, ldm] (mean, logvar), eps fp32 NCHW [Be, C, h, w] (None: the
    moments' first C channels are the latents), noise fp16 NCHW [B, C, h, w] -> NCHW fp16
    fp16(fp16(sf * fp16(mean + std * eps)) + fp16(noise * fp16(sigma))); image b uses moments b % Bm, eps b % Be."""
    lib = _lib.load()
    _req(moments, "moments"); _req(noise, "noise")
    Bm, h, w, ldm = moments.shape
    B = noise.shape[0]
    if not moments.is_contiguous() or not noise.is_contiguous() or tuple(noise.shape) != (B, channels, h, w):
        raise IHError(f"vae_sample_add_noise: contiguous moments and noise [B, {channels}, {h}, {w}] required")
    Be = 0
    if eps is not None:
        _req(eps, "eps", torch.float32)
        Be = eps.shape[0]
        if not eps.is_contiguous() or tuple(eps.shape[1:]) != (channels, h, w):
            raise IHError(f"vae_sample_add_noise: eps must be contiguous [Be, {channels}, {h}, {w}]")
    if out is None:
        out = torch.empty((B, channels, h, w), dtype=torch.float16, device=moments.device)
    check(lib.ih_vae_sample_add_noise_f16(moments.data_ptr(), ldm, Bm, _p(eps), Be, noise.data_ptr(), out.data_ptr(), B,
                                          channels, h, w, float(scaling_factor), float(sigma), _stream()),
          "ih_vae_sample_add_noise_f16")
    return out


def vae_sample_inpaint(moments: torch.Tensor, eps: Optional[torch.Tensor], noise: torch.Tensor, channels: int,
                       scaling_factor: float, sigma: float, pure_noise: bool) -> Tuple[torch.Tensor, torch.Tensor]:
    """Inpainting start latents and z0 (both NCHW fp16 [B, C, h, w]), arguments as vae_sample_add_noise:
    z0 = fp16(sf * fp16(mean + std * eps)); latents = fp16(z0 + fp16(noise * fp16(sigma))), or with `pure_noise`
    (strength 1) fp16(noise * sigma) with sigma = init_noise_sigma."""
    lib = _lib.load()
    _req(moments, "moments"); _req(noise, "noise")
    Bm, h, w, ldm = moments.shape
    B = noise.shape[0]
    if not moments.is_contiguous() or not noise.is_contiguous() or tuple(noise.shape) != (B, channels, h, w):
        raise IHError(f"vae_sample_inpaint: contiguous moments and noise [B, {channels}, {h}, {w}] required")
    Be = 0
    if eps is not None:
        _req(eps, "eps", torch.float32)
        Be = eps.shape[0]
        if not eps.is_contiguous() or tuple(eps.shape[1:]) != (channels, h, w):
            raise IHError(f"vae_sample_inpaint: eps must be contiguous [Be, {channels}, {h}, {w}]")
    latents = torch.empty((B, channels, h, w), dtype=torch.float16, device=moments.device)
    z0 = torch.empty_like(latents)
    check(lib.ih_vae_sample_inpaint_f16(moments.data_ptr(), ldm, Bm, _p(eps), Be, noise.data_ptr(), latents.data_ptr(),
                                        z0.data_ptr(), B, channels, h, w, float(scaling_factor), float(sigma),
                                        int(pure_noise), _stream()), "ih_vae_sample_inpaint_f16")
    return latents, z0


def latent_mask(mask_u8: torch.Tensor) -> torch.Tensor:
    """uint8 grayscale mask [Bm, H, W] (H, W multiples of 8) -> uint8 {0, 1} [Bm, H/8, W/8]: pixel (8y, 8x) >= 128."""
    lib = _lib.load()
    _req(mask_u8, "mask_u8", torch.uint8)
    if mask_u8.dim() != 3 or not mask_u8.is_contiguous():
        raise IHError("latent_mask: contiguous uint8 [Bm, H, W] required")
    Bm, H, W = mask_u8.shape
    out = torch.empty((Bm, H // 8, W // 8), dtype=torch.uint8, device=mask_u8.device)
    check(lib.ih_latent_mask_u8(mask_u8.data_ptr(), out.data_ptr(), Bm, H, W, _stream()), "ih_latent_mask_u8")
    return out


def pack_conv3x3_weight(w_oihw: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3] (nn.Conv2d) -> [Cout, 9*Cin] tap-major, the layout ih_conv2d_f16 expects."""
    Cout, Cin, kh, kw = w_oihw.shape
    assert kh == 3 and kw == 3
    return w_oihw.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()


_attn_ws = {}
_ws_generation = 0


def workspace_generation() -> int:
    """Bumped whenever a persistent scratch buffer (attention KV-split parts, GroupNorm statistics) is re-allocated.
    A CUDA graph captured under an older generation may hold a pointer to freed memory: DenoiseEngine compares this
    number with the one it recorded at capture time and re-captures instead of replaying a stale graph."""
    return _ws_generation


def _bump_generation() -> None:
    global _ws_generation
    _ws_generation += 1


def _attn_workspace(device, need: int) -> Optional[torch.Tensor]:
    """Persistent grow-only scratch for the KV-split self-attention parts (one per device; calls are stream-ordered)."""
    if need <= 0:
        return None
    ws = _attn_ws.get(device)
    if ws is None or ws.numel() < need:
        if torch.cuda.is_current_stream_capturing():
            raise IHError("attention workspace must be created before CUDA-graph capture (run one warm-up step)")
        had = ws is not None
        ws = torch.zeros(max(need, 16 << 20), dtype=torch.uint8, device=device)   # arrival counters start at zero
        _attn_ws[device] = ws
        if had:
            _bump_generation()
    return ws


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, B: int, H: int, Nq: int, Nk: int, *,
              n_ip: int = 0, ip_scale: float = 1.0, out: Optional[torch.Tensor] = None,
              kv_split: bool = True) -> torch.Tensor:
    """q [B*Nq, >=H*64] / k, v [B*Nk, >=H*64] 2-D views (row stride arbitrary); returns [B*Nq, H*64].
    kv_split=False withholds the workspace, i.e. every query tile is processed whole (ih_attention_f16 behaviour)."""
    lib = _lib.load()
    _req(q, "q"); _req(k, "k"); _req(v, "v")
    if out is None:
        out = torch.empty((B * Nq, H * 64), dtype=torch.float16, device=q.device)
    ws = _attn_workspace(q.device, int(lib.ih_attention_workspace_bytes(B, H, Nq, Nk, n_ip))) if kv_split else None
    rc = lib.ih_attention_ws_f16(q.data_ptr(), _rows(q, "q"), k.data_ptr(), _rows(k, "k"), v.data_ptr(),
                                 _rows(v, "v"), out.data_ptr(), _rows(out, "out"), B, H, Nq, Nk, n_ip,
                                 float(ip_scale), _p(ws), 0 if ws is None else ws.numel(), _stream())
    check(rc, "ih_attention_ws_f16")
    return out


# Measured on B200 (tools/attn_probe.py cross, profiles/): at UNet batch 2 the fused q-projection + cross-attention
# kernel takes 28.6 us per layer against 25.2 us for projection GEMM + attention kernel -- its per-head attention
# epilogue is a serial latency chain with nothing to overlap (one tile per CTA, TMEM full), while the stand-alone
# kernel hides the same chain behind three co-resident CTAs per SM.  The processors therefore use it only on request.
USE_FUSED_XATTN = os.environ.get("IH_XATTN_FUSED", "0") == "1"


def xattn_q_fused_ok(Nq: int, Nk: int) -> bool:
    """Shapes the fused q-projection + short-key cross-attention kernel covers (else: linear + attention)."""
    return Nq % 128 == 0 and 0 < Nk <= 96


def xattn_q_fused(h: torch.Tensor, wq: torch.Tensor, k: torch.Tensor, v: torch.Tensor, B: int, H: int, Nq: int,
                  Nk: int, *, n_ip: int = 0, ip_scale: float = 1.0, bias: Optional[torch.Tensor] = None, ln=None,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """attention(linear(h, wq, bias, ln=ln), k, v, ...) in one kernel: h [B*Nq, K] raw rows, wq [H*64, K],
    k / v [B*Nk, >=H*64] views; `ln=(stats, eps)` as in linear().  Returns [B*Nq, H*64]."""
    lib = _lib.load()
    _req(h, "h"); _req(wq, "wq"); _req(k, "k"); _req(v, "v")
    M, K = h.shape
    if M != B * Nq or tuple(wq.shape) != (H * 64, K) or not wq.is_contiguous():
        raise IHError(f"xattn_q_fused: h must be [{B * Nq}, K] and wq contiguous [{H * 64}, K]")
    ln_stats, ln_slabs, ln_eps = None, 0, 0.0
    if ln is not None:
        ln_stats, ln_eps = ln
        _req(ln_stats, "ln_stats", torch.float32)
        if ln_stats.dim() != 3 or ln_stats.shape[1] != M or ln_stats.shape[0] != (K + 63) // 64 or not ln_stats.is_contiguous():
            raise IHError("xattn_q_fused: ln statistics must be contiguous [ceil(K/64), M, 2]")
        ln_slabs = ln_stats.shape[0]
    if out is None:
        out = torch.empty((M, H * 64), dtype=torch.float16, device=h.device)
    rc = lib.ih_xattn_q_fused_f16(h.data_ptr(), _rows(h, "h"), wq.data_ptr(), _p(bias), _p(ln_stats), ln_slabs,
                                  float(ln_eps), k.data_ptr(), _rows(k, "k"), v.data_ptr(), _rows(v, "v"),
                                  out.data_ptr(), _rows(out, "out"), B, H, Nq, Nk, n_ip, float(ip_scale), K, _stream())
    check(rc, "ih_xattn_q_fused_f16")
    return out


_gn_ws = {}


def _gn_workspace(device, B: int, groups: int) -> torch.Tensor:
    """Persistent zero-initialised statistics workspace (one per device; GroupNorm calls are stream-ordered)."""
    need = int(_lib.load().ih_groupnorm_workspace_bytes(B, groups))
    ws = _gn_ws.get(device)
    if ws is None or ws.numel() < need:
        if torch.cuda.is_current_stream_capturing():
            raise IHError("groupnorm workspace must be created before CUDA-graph capture (run one warm-up step)")
        had = ws is not None
        ws = torch.zeros(max(need, 1 << 20), dtype=torch.uint8, device=device)
        _gn_ws[device] = ws
        if had:
            _bump_generation()
    return ws


def groupnorm(x0: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, *, x1: Optional[torch.Tensor] = None,
              groups: int = 32, eps: float = 1e-5, silu: bool = False, out: Optional[torch.Tensor] = None,
              ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm over NHWC x0 [B,H,W,C0] (optionally concatenated with x1 [B,H,W,C1] on channels)."""
    lib = _lib.load()
    _req(x0, "x0")
    B, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else x1.shape[-1]
    if not x0.is_contiguous() or (x1 is not None and not x1.is_contiguous()):
        raise IHError("groupnorm: inputs must be contiguous NHWC")
    if out is None:
        out = torch.empty((B, H, W, C0 + C1), dtype=torch.float16, device=x0.device)
    if ws is None:
        ws = _gn_workspace(x0.device, B, groups)
    rc = lib.ih_groupnorm_f16(x0.data_ptr(), C0, _p(x1), C1, gamma.data_ptr(), beta.data_ptr(), out.data_ptr(),
                              ws.data_ptr(), B, H * W, groups, float(eps), int(silu), _stream())
    check(rc, "ih_groupnorm_f16")
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _req(x, "x")
    if not x.is_contiguous():
        raise IHError("layernorm: x must be contiguous")
    C = x.shape[-1]
    rows = x.numel() // C
    if out is None:
        out = torch.empty_like(x)
    rc = lib.ih_layernorm_f16(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), rows, C, float(eps),
                              _stream())
    check(rc, "ih_layernorm_f16")
    return out


def linear_small(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, act_in: bool = False,
                 act_out: bool = False, addend: Optional[torch.Tensor] = None, out_scale: float = 1.0,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Small-M (<= 8 rows) linear with optional SiLU on the input and/or output and an optional fp16 addend."""
    lib = _lib.load()
    _req(x, "x"); _req(w, "w")
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float16, device=x.device)
    if M > 64:
        raise IHError(f"linear_small: M={M} > 64 rows; use ops.linear")
    ld_add = _rows(addend, "addend") if addend is not None else 0
    rc = lib.ih_linear_small_f16(x.data_ptr(), _rows(x, "x"), w.data_ptr(), _p(bias), _p(addend), ld_add,
                                 out.data_ptr(), _rows(out, "out"), M, N, K, int(act_in), int(act_out),
                                 float(out_scale), _stream())
    check(rc, "ih_linear_small_f16")
    return out


def attention_small(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, B: int, H: int, Nq: int, Nk: int, dqk: int,
                    dv: int, scale: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """CUDA-core attention for odd head sizes / few queries: q [B*Nq, H*dqk], k [B*Nk, H*dqk], v [B*Nk, H*dv]."""
    lib = _lib.load()
    _req(q, "q"); _req(k, "k"); _req(v, "v")
    if out is None:
        out = torch.empty((B * Nq, H * dv), dtype=torch.float16, device=q.device)
    rc = lib.ih_attention_small_f16(q.data_ptr(), _rows(q, "q"), k.data_ptr(), _rows(k, "k"), v.data_ptr(),
                                    _rows(v, "v"), out.data_ptr(), _rows(out, "out"), B, H, Nq, Nk, dqk, dv,
                                    float(scale), _stream())
    check(rc, "ih_attention_small_f16")
    return out


def attention_generic(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, B: int, H: int, Nq: int, Nk: int, dqk: int,
                      dv: int, scale: float, causal: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(q k^T * scale (+ causal mask)) v for any head dims that are multiples of 8 (CLIP towers: 64 causal,
    104 for ViT-bigG): q [B*Nq, >=H*dqk], k [B*Nk, >=H*dqk], v [B*Nk, >=H*dv] 2-D views."""
    lib = _lib.load()
    _req(q, "q"); _req(k, "k"); _req(v, "v")
    if out is None:
        out = torch.empty((B * Nq, H * dv), dtype=torch.float16, device=q.device)
    rc = lib.ih_attention_generic_f16(q.data_ptr(), _rows(q, "q"), k.data_ptr(), _rows(k, "k"), v.data_ptr(),
                                      _rows(v, "v"), out.data_ptr(), _rows(out, "out"), B, H, Nq, Nk, dqk, dv,
                                      float(scale), int(causal), _stream())
    check(rc, "ih_attention_generic_f16")
    return out


def embed_tokens(ids: torch.Tensor, tok_emb: torch.Tensor, pos_emb: torch.Tensor,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """ids int32 [B, T] (device) -> tok_emb[ids] + pos_emb[:T]  as [B*T, C] fp16."""
    lib = _lib.load()
    _req(ids, "ids", torch.int32); _req(tok_emb, "tok_emb"); _req(pos_emb, "pos_emb")
    B, T = ids.shape
    C = tok_emb.shape[1]
    if not (ids.is_contiguous() and tok_emb.is_contiguous() and pos_emb.is_contiguous()) or pos_emb.shape[0] < T:
        raise IHError("embed_tokens: contiguous ids / tables and pos_emb with >= T rows required")
    if out is None:
        out = torch.empty((B * T, C), dtype=torch.float16, device=ids.device)
    check(lib.ih_embed_tokens_f16(ids.data_ptr(), tok_emb.data_ptr(), pos_emb.data_ptr(), out.data_ptr(), B * T, T, C,
                                  tok_emb.shape[0], _stream()), "ih_embed_tokens_f16")
    return out


def resize_patchify(img: torch.Tensor, size: int, patch: int, kpad: int, mean, std,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """img NCHW fp16 in [-1, 1] -> area-averaged size x size, [0,1], (v - mean) / std, as patch rows
    [B * (size/patch)^2, kpad] with k = c*patch^2 + py*patch + px (zero padded)."""
    import ctypes
    lib = _lib.load()
    _req(img, "img")
    B, C, H, W = img.shape
    if not img.is_contiguous():
        raise IHError("resize_patchify: contiguous NCHW image required")
    g = size // patch
    if out is None:
        out = torch.empty((B * g * g, kpad), dtype=torch.float16, device=img.device)
    m3 = (ctypes.c_float * 3)(*[float(x) for x in mean])
    s3 = (ctypes.c_float * 3)(*[float(x) for x in std])
    check(lib.ih_resize_patchify_f16(img.data_ptr(), out.data_ptr(), B, C, H, W, size, patch, kpad, m3, s3, _stream()),
          "ih_resize_patchify_f16")
    return out


def softmax_rows_(x: torch.Tensor) -> torch.Tensor:
    """In-place softmax over the last dimension of a 2-D fp16 matrix (row stride arbitrary, cols % 8 == 0, <= 32768)."""
    lib = _lib.load()
    _req(x, "x")
    if x.dim() != 2:
        raise IHError("softmax_rows_: 2-D matrix required")
    check(lib.ih_softmax_rows_f16(x.data_ptr(), _rows(x, "x"), x.shape[0], x.shape[1], _stream()), "ih_softmax_rows_f16")
    return x


def add_bcast(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """a + b where b is broadcast over the leading elements of a (a.numel() % b.numel() == 0), contiguous fp16."""
    lib = _lib.load()
    _req(a, "a"); _req(b, "b")
    if not (a.is_contiguous() and b.is_contiguous()) or a.numel() % b.numel() != 0:
        raise IHError("add_bcast: contiguous tensors with a.numel() % b.numel() == 0 required")
    if out is None:
        out = torch.empty_like(a)
    check(lib.ih_add_bcast_f16(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.numel(), b.numel(), _stream()),
          "ih_add_bcast_f16")
    return out


def mean_tokens(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[B, n, D] -> [B, D] mean over tokens."""
    lib = _lib.load()
    _req(x, "x")
    B, n, D = x.shape
    if not x.is_contiguous():
        raise IHError("mean_tokens: x must be contiguous")
    if out is None:
        out = torch.empty((B, D), dtype=torch.float16, device=x.device)
    check(lib.ih_mean_tokens_f16(x.data_ptr(), out.data_ptr(), B, n, D, _stream()), "ih_mean_tokens_f16")
    return out


def sinusoid(t: torch.Tensor, dim: int, n: int, *, step: Optional[torch.Tensor] = None,
             out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[n, dim] fp16 sinusoidal embedding of fp32 `t` (or of t[step] for every row when `step` is given)."""
    lib = _lib.load()
    _req(t, "t", torch.float32)
    if out is None:
        out = torch.empty((n, dim), dtype=torch.float16, device=t.device)
    rc = lib.ih_sinusoid_f16(t.data_ptr(), _p(step), out.data_ptr(), _rows(out, "out"), n, dim, _stream())
    check(rc, "ih_sinusoid_f16")
    return out


def upsample2x(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _req(x, "x")
    B, H, W, C = x.shape
    if out is None:
        out = torch.empty((B, 2 * H, 2 * W, C), dtype=torch.float16, device=x.device)
    check(lib.ih_upsample2x_f16(x.data_ptr(), out.data_ptr(), B, H, W, C, _stream()), "ih_upsample2x_f16")
    return out


def concat_channels(x0: torch.Tensor, x1: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _req(x0, "x0"); _req(x1, "x1")
    C0, C1 = x0.shape[-1], x1.shape[-1]
    rows = x0.numel() // C0
    if out is None:
        out = torch.empty(tuple(x0.shape[:-1]) + (C0 + C1,), dtype=torch.float16, device=x0.device)
    check(lib.ih_concat_f16(x0.data_ptr(), C0, x1.data_ptr(), C1, out.data_ptr(), rows, _stream()), "ih_concat_f16")
    return out


def conv_in(x_nchw: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, out: Optional[torch.Tensor] = None):
    lib = _lib.load()
    _req(x_nchw, "x")
    B, Cin, H, W = x_nchw.shape
    Cout = w.shape[0]
    if out is None:
        out = torch.empty((B, H, W, Cout), dtype=torch.float16, device=x_nchw.device)
    check(lib.ih_conv_in_f16(x_nchw.data_ptr(), w.data_ptr(), _p(bias), out.data_ptr(), B, H, W, Cin, Cout,
                             _stream()), "ih_conv_in_f16")
    return out


def conv_out(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, out: Optional[torch.Tensor] = None):
    lib = _lib.load()
    _req(x, "x")
    B, H, W, Cin = x.shape
    Cout = w.shape[0]
    if out is None:
        out = torch.empty((B, Cout, H, W), dtype=torch.float16, device=x.device)
    check(lib.ih_conv_out_f16(x.data_ptr(), w.data_ptr(), _p(bias), out.data_ptr(), B, H, W, Cin, Cout, _stream()),
          "ih_conv_out_f16")
    return out


def im2col3x3_nchw(x_nchw: torch.Tensor, kpad: int = 64, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[B, Cin, H, W] -> A [B*H*W, kpad] with k = ci*9 + ky*3 + kx (zero padded): conv_in as a tensor-core GEMM."""
    lib = _lib.load()
    _req(x_nchw, "x")
    B, Cin, H, W = x_nchw.shape
    if out is None:
        out = torch.empty((B * H * W, kpad), dtype=torch.float16, device=x_nchw.device)
    check(lib.ih_im2col3x3_nchw_f16(x_nchw.data_ptr(), out.data_ptr(), B, Cin, H, W, kpad, _stream()),
          "ih_im2col3x3_nchw_f16")
    return out


def softmax_rows_masked_(x: torch.Tensor, valid_cols: int) -> torch.Tensor:
    """softmax_rows_ over the first `valid_cols` columns of each row; the remaining (padding) columns become 0."""
    lib = _lib.load()
    _req(x, "x")
    if x.dim() != 2 or not 0 < valid_cols <= x.shape[1]:
        raise IHError("softmax_rows_masked_: 2-D matrix and 0 < valid_cols <= cols required")
    check(lib.ih_softmax_rows_masked_f16(x.data_ptr(), _rows(x, "x"), x.shape[0], x.shape[1], int(valid_cols), _stream()),
          "ih_softmax_rows_masked_f16")
    return x


def nhwc_to_nchw(x: torch.Tensor, C: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x NHWC [B, H, W, ldc] -> NCHW [B, C, H, W] taking channels [0, C)."""
    lib = _lib.load()
    _req(x, "x")
    B, H, W, ldc = x.shape
    if out is None:
        out = torch.empty((B, C, H, W), dtype=torch.float16, device=x.device)
    check(lib.ih_nhwc_to_nchw_f16(x.data_ptr(), ldc, out.data_ptr(), B, H * W, C, _stream()), "ih_nhwc_to_nchw_f16")
    return out


def euler_cfg_step(noise_pred: torch.Tensor, latents: torch.Tensor, model_in: torch.Tensor, sigmas: torch.Tensor,
                   step: torch.Tensor, guidance: float) -> None:
    lib = _lib.load()
    _req(noise_pred, "noise_pred"); _req(latents, "latents"); _req(model_in, "model_in")
    _req(sigmas, "sigmas", torch.float32); _req(step, "step", torch.int32)
    n = latents.shape[0]
    per = latents.numel() // n
    check(lib.ih_euler_cfg_step(noise_pred.data_ptr(), latents.data_ptr(), model_in.data_ptr(), sigmas.data_ptr(),
                                step.data_ptr(), float(guidance), per, n, _stream()), "ih_euler_cfg_step")


def euler_step(noise_pred: torch.Tensor, latents: torch.Tensor, model_in: torch.Tensor, sigmas: torch.Tensor,
               step: torch.Tensor, guidance: float, *, use_cfg: bool = True, guidance_rescale: float = 0.0) -> None:
    """One scheduler transition with the reference's loop options: the default (CFG, no rescale) is the fused
    grid-stride kernel `ih_euler_cfg_step`; guidance_scale <= 1 and guidance_rescale > 0 (custom_pipelines.py:223,
    :352-354) run `ih_euler_step_ex` (one block per image, per-image std for the rescale)."""
    if use_cfg and not guidance_rescale:
        return euler_cfg_step(noise_pred, latents, model_in, sigmas, step, guidance)
    lib = _lib.load()
    _req(noise_pred, "noise_pred"); _req(latents, "latents"); _req(model_in, "model_in")
    _req(sigmas, "sigmas", torch.float32); _req(step, "step", torch.int32)
    n = latents.shape[0]
    per = latents.numel() // n
    want = (2 * n if use_cfg else n) * per
    if noise_pred.numel() != want or model_in.numel() != want:
        raise IHError(f"euler_step: noise_pred / model_in must hold {want} elements (use_cfg={use_cfg})")
    check(lib.ih_euler_step_ex(noise_pred.data_ptr(), latents.data_ptr(), model_in.data_ptr(), sigmas.data_ptr(),
                               step.data_ptr(), float(guidance), float(guidance_rescale), per, n, int(use_cfg),
                               _stream()), "ih_euler_step_ex")


def euler_step_inpaint(noise_pred: torch.Tensor, latents: torch.Tensor, model_in: torch.Tensor, sigmas: torch.Tensor,
                       step: torch.Tensor, guidance: float, mask: torch.Tensor, z0: torch.Tensor, noise: torch.Tensor,
                       last: torch.Tensor, *, use_cfg: bool = True, guidance_rescale: float = 0.0) -> None:
    """euler_step followed by the inpainting blend, in the same kernel (`ih_euler_step_inpaint`): outside the mask the
    latents become z0 noised to the next sigma (z0 itself on the step index `last`), before model_in is formed.
    mask uint8 {0, 1} [Bm, h, w] (latent image b uses mask b % Bm); z0, noise fp16 like `latents`; last int32 [1]."""
    lib = _lib.load()
    _req(noise_pred, "noise_pred"); _req(latents, "latents"); _req(model_in, "model_in")
    _req(sigmas, "sigmas", torch.float32); _req(step, "step", torch.int32)
    _req(mask, "mask", torch.uint8); _req(z0, "z0"); _req(noise, "noise"); _req(last, "last", torch.int32)
    n, _, h, w = latents.shape
    per = latents.numel() // n
    want = (2 * n if use_cfg else n) * per
    if noise_pred.numel() != want or model_in.numel() != want:
        raise IHError(f"euler_step_inpaint: noise_pred / model_in must hold {want} elements (use_cfg={use_cfg})")
    if z0.shape != latents.shape or noise.shape != latents.shape or mask.dim() != 3 or tuple(mask.shape[1:]) != (h, w) \
            or n % mask.shape[0] or not (mask.is_contiguous() and z0.is_contiguous() and noise.is_contiguous()):
        raise IHError(f"euler_step_inpaint: contiguous z0 / noise {tuple(latents.shape)} and mask [Bm, {h}, {w}] with "
                      f"{n} % Bm == 0 required")
    check(lib.ih_euler_step_inpaint(noise_pred.data_ptr(), latents.data_ptr(), model_in.data_ptr(), sigmas.data_ptr(),
                                    step.data_ptr(), float(guidance), float(guidance_rescale), per, n, int(use_cfg),
                                    mask.data_ptr(), mask.shape[0], h * w, z0.data_ptr(), noise.data_ptr(),
                                    last.data_ptr(), _stream()), "ih_euler_step_inpaint")


def scale_model_input(latents: torch.Tensor, model_in: torch.Tensor, sigmas: torch.Tensor, step: torch.Tensor,
                      duplicate: bool = True) -> None:
    lib = _lib.load()
    _req(latents, "latents"); _req(model_in, "model_in")
    if model_in.numel() != (2 if duplicate else 1) * latents.numel():
        raise IHError("scale_model_input: model_in must hold the CFG pair (duplicate=True) or one copy of the latents")
    check(lib.ih_scale_model_input_ex(latents.data_ptr(), model_in.data_ptr(), sigmas.data_ptr(), step.data_ptr(),
                                      latents.numel(), int(duplicate), _stream()), "ih_scale_model_input_ex")
