"""Native SDXL VAE decoder (scope row f1: custom_pipelines.py:365-386 `vae.decode(latents / scaling_factor)` + postprocess)
and encoder (row f5, image-to-image editing: `AutoencoderKLEncoder`, see its docstring).

Module tree and state-dict keys are those of [3P] diffusers==0.30.0 `AutoencoderKL` (decoder: `post_quant_conv.*`,
`decoder.*`; encoder: `encoder.*`, `quant_conv.*`; each half ignores the other's keys), so
`vae/diffusion_pytorch_model.safetensors` loads without a key map.  Every operator of the decoder runs on the sm_100a
kernels of this package:

* `post_quant_conv` (1x1, 4->4), the division by `scaling_factor` and `decoder.conv_in` (3x3, 4->C) are ONE tensor-core
  GEMM: the latent gets a constant-one fifth channel, `ih_im2col3x3_nchw_f16` builds the [B*h*w, 45 -> 64] patch matrix
  (zero padding applies to the ones channel too, which makes the folded bias exact at the image border) and the folded
  weight W'[o, (c, tap)] = sum_m conv_in[o, m, tap] * pqc[m, c] / scaling_factor multiplies it;
* ResnetBlock2D (no time embedding): GroupNorm+SiLU kernel -> implicit-GEMM conv3x3 (residual fused in conv2);
* mid-block attention (1 head, head_dim = C = 512, N = h*w tokens): q / k GEMMs (1/sqrt(C) folded into q), V^T = W_v h^T
  by a GEMM, then per block of <= 64 MiB of scores: q k^T (GEMM) -> `ih_softmax_rows_masked_f16` -> P V + b_v (GEMM);
  out projection with fused residual;
* nearest 2x upsample + conv3x3; conv_out with Cout padded 3 -> 16 and a gather to NCHW.

Numerics: fp16 storage / fp32 accumulation like the UNet.  The reference upcasts the VAE to fp32 when
`vae.config.force_upcast` is set, because the ORIGINAL SDXL VAE's activations overflow fp16 (custom_pipelines.py:366-371).
The native equivalent is a SCALED RESIDUAL STREAM: the decoder's residual stream (conv_in output, every ResBlock /
attention / upsampler output) is stored as s * x with s = 2^-7.  GroupNorm is scale invariant (GN(s x; eps s^2) = GN(x; eps)),
so each consumer normalises the scaled stream directly; every conv / linear that WRITES the stream scales its
accumulator and bias by s in the GEMM epilogue (`alpha`), shortcuts / upsampler convs are linear in the stream and only
scale their bias.  In real arithmetic this is exact; in fp16 it moves the representable range from 6.5e4 to 8.4e6 while
the weights stay untouched.  `force_upcast = False` configurations (the fp16-fix checkpoint) run with s = 1.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops
from ._lib import IHError
from .config import SDXL_VAE, VAEConfig


def _scaled(t: torch.Tensor, s: float) -> torch.Tensor:
    """bias * s in the parameter dtype (s is a power of two: exact unless the product is subnormal)."""
    return t.detach() if s == 1.0 else (t.detach().float() * s).to(t.dtype).contiguous()


class VAEResnetBlock(nn.Module):
    def __init__(self, cin: int, cout: int, groups: int):
        super().__init__()
        self.cin, self.cout, self.groups = cin, cout, groups
        self.norm1 = nn.GroupNorm(groups, cin, eps=1e-6)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.norm2 = nn.GroupNorm(groups, cout, eps=1e-6)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        self.conv_shortcut = nn.Conv2d(cin, cout, 1) if cin != cout else None
        self._w1 = self._w2 = self._wsc = None
        self._s = 1.0

    def finalize(self, s: float = 1.0):
        self._s = s
        self._w1 = ops.pack_conv3x3_weight(self.conv1.weight.detach())
        self._w2 = ops.pack_conv3x3_weight(self.conv2.weight.detach())
        self._b1, self._b2 = _scaled(self.conv1.bias, s), _scaled(self.conv2.bias, s)
        if self.conv_shortcut is not None:
            self._wsc = self.conv_shortcut.weight.detach().reshape(self.cout, self.cin).contiguous()
            self._bsc = _scaled(self.conv_shortcut.bias, s)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x = s * (residual stream); returns s * (block output).  conv1's output only feeds norm2, so it is kept at the
        same scale s (its magnitude follows the stream's in the original VAE)."""
        B, H, W, _ = x.shape
        s = self._s
        eps = 1e-6 * s * s
        h = ops.groupnorm(x, self.norm1.weight, self.norm1.bias, groups=self.groups, eps=eps, silu=True)
        h = ops.conv3x3(h, self._w1, self._b1, alpha=s)
        h = ops.groupnorm(h, self.norm2.weight, self.norm2.bias, groups=self.groups, eps=eps, silu=True)
        sc = x
        if self.conv_shortcut is not None:       # linear in the (scaled) stream: only the bias is scaled
            sc = ops.linear(x.reshape(B * H * W, self.cin), self._wsc, self._bsc).reshape(B, H, W, self.cout)
        return ops.conv3x3(h, self._w2, self._b2, residual=sc, alpha=s)


class VAEAttention(nn.Module):
    """diffusers `Attention(heads=1, dim_head=C, norm_num_groups, residual_connection=True, bias=True)`.

    One head of width C = 512 over N = h * w tokens.  The N x N score matrix is never materialised whole: queries are
    processed in blocks sized so that a block of fp16 scores stays within 64 MiB (L2-resident on B200: 2048 query rows at
    N = 16384, the 1024^2 image), each block = scores GEMM -> masked row softmax -> P V GEMM on the tensor-core kernel.
    V^T comes straight out of a GEMM (W_v h^T), and the v bias is added after P V (softmax rows sum to one)."""

    SCORE_BLOCK_BYTES = 64 << 20

    def __init__(self, ch: int, groups: int):
        super().__init__()
        self.ch, self.groups = ch, groups
        self.group_norm = nn.GroupNorm(groups, ch, eps=1e-6)
        self.to_q = nn.Linear(ch, ch)
        self.to_k = nn.Linear(ch, ch)
        self.to_v = nn.Linear(ch, ch)
        self.to_out = nn.ModuleList([nn.Linear(ch, ch), nn.Dropout(0.0)])
        self._w_q = self._b_q = None
        self._s = 1.0

    def finalize(self, s: float = 1.0):
        self._s = s
        sc = self.ch ** -0.5                                     # softmax scale folded into the q projection
        dt = self.to_q.weight.dtype
        self._w_q = (self.to_q.weight.detach().float() * sc).to(dt).contiguous()
        self._b_q = (self.to_q.bias.detach().float() * sc).to(dt).contiguous()
        self._b_o = _scaled(self.to_out[0].bias, s)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        B, H, W, C = x.shape
        N = H * W
        Np = (N + 7) // 8 * 8                 # the GEMM / softmax kernels want multiples of 8: pad keys, mask their scores
        if Np > 32768:
            raise IHError(f"VAE mid-block attention: {N} tokens exceed 32768 (enable_vae_tiling() decodes 128x128 tiles)")
        s = self._s
        h = ops.groupnorm(x, self.group_norm.weight, self.group_norm.bias, groups=self.groups, eps=1e-6 * s * s, silu=False)
        h2 = h.reshape(B * N, C)
        q = ops.linear(h2, self._w_q, self._b_q)                                    # [B*N, C], 1/sqrt(C) folded in
        k = ops.linear(h2, self.to_k.weight, self.to_k.bias)
        o = torch.empty((B * N, C), dtype=x.dtype, device=x.device)
        block = max(128, min((N + 127) // 128 * 128, self.SCORE_BLOCK_BYTES // (2 * Np) // 128 * 128))
        scores = torch.empty((block, Np), dtype=x.dtype, device=x.device)           # reused by every block
        vt = (torch.empty if Np == N else torch.zeros)((C, Np), dtype=x.dtype, device=x.device)
        for b in range(B):                                                          # one image at a time
            hb, kb = h2[b * N:(b + 1) * N], k[b * N:(b + 1) * N]
            if Np != N:                                                             # odd edge tiles of a tiled decode
                hp = torch.zeros((Np, C), dtype=x.dtype, device=x.device)
                kp = torch.zeros((Np, C), dtype=x.dtype, device=x.device)
                hp[:N], kp[:N] = hb, kb
                hb, kb = hp, kp
            ops.linear(self.to_v.weight, hb, out=vt)                                # V^T = W_v h^T  [C, Np]
            for r0 in range(0, N, block):
                rows = min(block, N - r0)
                sc = scores[:rows]
                ops.linear(q[b * N + r0: b * N + r0 + rows], kb, out=sc)            # scores (scale already in q)
                ops.softmax_rows_masked_(sc, N)                                     # padded keys get no weight
                ops.linear(sc, vt, self.to_v.bias, out=o[b * N + r0: b * N + r0 + rows])   # P V + b_v
        out = ops.linear(o, self.to_out[0].weight, self._b_o, residual=x.reshape(B * N, C), alpha=s)
        return out.reshape(B, H, W, C)


class VAEUpsample(nn.Module):
    def __init__(self, ch: int):
        super().__init__()
        self.conv = nn.Conv2d(ch, ch, 3, padding=1)
        self._w = None

    def finalize(self, s: float = 1.0):
        self._w = ops.pack_conv3x3_weight(self.conv.weight.detach())
        self._b = _scaled(self.conv.bias, s)

    def forward(self, x):
        return ops.conv3x3(ops.upsample2x(x), self._w, self._b)     # linear in the scaled stream: only the bias scales


class VAEMidBlock(nn.Module):
    def __init__(self, ch: int, groups: int):
        super().__init__()
        self.attentions = nn.ModuleList([VAEAttention(ch, groups)])
        self.resnets = nn.ModuleList([VAEResnetBlock(ch, ch, groups), VAEResnetBlock(ch, ch, groups)])

    def forward(self, x):
        x = self.resnets[0](x)
        x = self.attentions[0](x)
        return self.resnets[1](x)


class VAEUpBlock(nn.Module):
    def __init__(self, cin: int, cout: int, n_res: int, groups: int, add_up: bool):
        super().__init__()
        self.resnets = nn.ModuleList([VAEResnetBlock(cin if j == 0 else cout, cout, groups) for j in range(n_res)])
        if add_up:
            self.upsamplers = nn.ModuleList([VAEUpsample(cout)])
        self.has_up = add_up

    def forward(self, x):
        for r in self.resnets:
            x = r(x)
        return self.upsamplers[0](x) if self.has_up else x


class Decoder(nn.Module):
    def __init__(self, cfg: VAEConfig):
        super().__init__()
        ch = cfg.decoder_channels
        g = cfg.norm_num_groups
        self.conv_in = nn.Conv2d(cfg.latent_channels, ch[0], 3, padding=1)
        self.mid_block = VAEMidBlock(ch[0], g)
        ups: List[nn.Module] = []
        prev = ch[0]
        for i, c in enumerate(ch):
            ups.append(VAEUpBlock(prev, c, cfg.layers_per_block + 1, g, add_up=i < len(ch) - 1))
            prev = c
        self.up_blocks = nn.ModuleList(ups)
        self.conv_norm_out = nn.GroupNorm(g, ch[-1], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[-1], cfg.out_channels, 3, padding=1)


class AutoencoderKLDecoder(nn.Module):
    """`decode(latents)` = diffusers `vae.decode(latents / scaling_factor).sample` (the division is folded in)."""

    def __init__(self, cfg: VAEConfig = SDXL_VAE):
        super().__init__()
        self.config = cfg
        self.post_quant_conv = nn.Conv2d(cfg.latent_channels, cfg.latent_channels, 1)
        self.decoder = Decoder(cfg)
        self._w_in = self._w_out = self._b_out = None
        self.use_tiling = False             # pipeline.enable_vae_tiling() (test.py:73)
        # scale of the stored residual stream (module docstring): 2^-7 when the configuration asks for the fp32 upcast
        self.stream_scale = 2.0 ** -7 if getattr(cfg, "force_upcast", True) else 1.0

    # ---- construction ------------------------------------------------------------------------------------------
    @classmethod
    def from_state_dict(cls, cfg: VAEConfig, sd: Dict[str, torch.Tensor], device="cuda",
                        stream_scale: Optional[float] = None) -> "AutoencoderKLDecoder":
        with torch.device("meta"):
            m = cls(cfg)
        if stream_scale is not None:
            if stream_scale <= 0 or math.log2(stream_scale) != int(math.log2(stream_scale)):
                raise IHError("stream_scale must be a power of two")
            m.stream_scale = float(stream_scale)
        m = m.to_empty(device=device)
        own = m.state_dict()
        missing = [k for k in own if k not in sd]
        if missing:
            raise KeyError(f"VAE checkpoint lacks {len(missing)} decoder keys, e.g. {missing[:3]}")
        m.load_state_dict({k: sd[k].to(device=device, dtype=torch.float16).reshape(own[k].shape) for k in own})
        m = m.half().eval()
        m.finalize()
        return m

    def finalize(self) -> None:
        s = self.stream_scale
        for mod in self.modules():
            if isinstance(mod, (VAEResnetBlock, VAEAttention, VAEUpsample)):
                mod.finalize(s)
        self._b_in = _scaled(self.decoder.conv_in.bias, s)
        cfg = self.config
        L = cfg.latent_channels
        w_in = self.decoder.conv_in.weight.detach().float()                          # [C, L, 3, 3]
        w_pq = self.post_quant_conv.weight.detach().float().reshape(L, L)            # [m, c]
        b_pq = self.post_quant_conv.bias.detach().float()
        C0 = w_in.shape[0]
        folded = torch.zeros((C0, L + 1, 9), dtype=torch.float32, device=w_in.device)
        wt = w_in.reshape(C0, L, 9)                                                  # [o, m, tap]
        folded[:, :L] = torch.einsum("omt,mc->oct", wt, w_pq) / cfg.scaling_factor   # latent channels (z / sf folded)
        folded[:, L] = torch.einsum("omt,m->ot", wt, b_pq)                           # the constant-one channel
        kpad = 64
        w = torch.zeros((C0, kpad), dtype=torch.float32, device=w_in.device)
        w[:, :(L + 1) * 9] = folded.reshape(C0, (L + 1) * 9)                         # k = ci*9 + ky*3 + kx
        self._w_in = w.to(self.decoder.conv_in.weight.dtype).contiguous()
        co = self.decoder.conv_out
        cpad = 16
        w_out = torch.zeros((cpad,) + tuple(co.weight.shape[1:]), dtype=co.weight.dtype, device=co.weight.device)
        w_out[:cfg.out_channels] = co.weight.detach()
        self._w_out = ops.pack_conv3x3_weight(w_out)
        b_out = torch.zeros((cpad,), dtype=co.weight.dtype, device=co.weight.device)
        b_out[:cfg.out_channels] = co.bias.detach()
        self._b_out = b_out

    # ---- forward -----------------------------------------------------------------------------------------------
    @torch.no_grad()
    def decode(self, latents: torch.Tensor) -> torch.Tensor:
        """latents [B, 4, h, w] fp16 straight from the denoise loop -> image [B, 3, 8h, 8w] fp16 in [-1, 1] (nominally).
        With `use_tiling` and a latent larger than one tile (128 x 128 for SDXL) the image is decoded tile by tile and
        blended, [3P] diffusers `AutoencoderKL.tiled_decode`."""
        if self._w_in is None:
            raise IHError("AutoencoderKLDecoder.finalize() has not run (use from_state_dict)")
        t = self.config.tile_latent_min_size
        if self.use_tiling and (latents.shape[-1] > t or latents.shape[-2] > t):
            return self._tiled_decode(latents)
        return self._decode_tile(latents)

    def _tiled_decode(self, z: torch.Tensor) -> torch.Tensor:
        """[3P] tiled_decode: tiles of `tile_latent_min_size` latents every (1 - overlap) tile, each decoded on its own
        (so tile borders see zero padding, as in diffusers), then linearly cross-faded over the overlap with the tile
        above and the tile to the left and cropped to the stride.  The cross-fade is elementwise torch glue."""
        cfg = self.config
        tl = cfg.tile_latent_min_size
        overlap = int(tl * (1 - cfg.tile_overlap_factor))
        blend = int(cfg.sample_size * cfg.tile_overlap_factor)
        limit = cfg.sample_size - blend
        rows = []
        for i in range(0, z.shape[2], overlap):
            rows.append([self._decode_tile(z[:, :, i:i + tl, j:j + tl].contiguous()).float()
                         for j in range(0, z.shape[3], overlap)])

        def blend_v(a, b, ext):
            ext = min(a.shape[2], b.shape[2], ext)
            wgt = (torch.arange(ext, device=b.device, dtype=torch.float32) / ext).view(1, 1, ext, 1)
            b[:, :, :ext, :] = a[:, :, -ext:, :] * (1 - wgt) + b[:, :, :ext, :] * wgt
            return b

        def blend_h(a, b, ext):
            ext = min(a.shape[3], b.shape[3], ext)
            wgt = (torch.arange(ext, device=b.device, dtype=torch.float32) / ext).view(1, 1, 1, ext)
            b[:, :, :, :ext] = a[:, :, :, -ext:] * (1 - wgt) + b[:, :, :, :ext] * wgt
            return b

        out_rows = []
        for i, row in enumerate(rows):
            out_row = []
            for j, tile in enumerate(row):
                if i > 0:
                    tile = blend_v(rows[i - 1][j], tile, blend)
                if j > 0:
                    tile = blend_h(row[j - 1], tile, blend)
                out_row.append(tile[:, :, :limit, :limit])
            out_rows.append(torch.cat(out_row, dim=3))
        return torch.cat(out_rows, dim=2).to(z.dtype if z.dtype != torch.float32 else torch.float32)

    def _decode_tile(self, latents: torch.Tensor) -> torch.Tensor:
        B, L, h, w = latents.shape
        dec = self.decoder
        dt = self._w_in.dtype                                     # fp16 on the GPU (fp32 only in the CPU wiring test)
        ones = torch.ones((B, 1, h, w), dtype=dt, device=latents.device)
        z5 = torch.cat([latents.to(dt), ones], dim=1).contiguous()
        a = ops.im2col3x3_nchw(z5, self._w_in.shape[1])
        s = self.stream_scale
        x = ops.linear(a, self._w_in, self._b_in, alpha=s).reshape(B, h, w, -1)        # s * (post_quant_conv + /sf + conv_in)
        x = dec.mid_block(x)
        for blk in dec.up_blocks:
            x = blk(x)
        g = self.config.norm_num_groups
        x = ops.groupnorm(x, dec.conv_norm_out.weight, dec.conv_norm_out.bias, groups=g, eps=1e-6 * s * s, silu=True)
        x = ops.conv3x3(x, self._w_out, self._b_out)
        return ops.nhwc_to_nchw(x, self.config.out_channels)


class VAEDownsample(nn.Module):
    """diffusers Downsample2D(padding=0): conv3x3(F.pad(x, (0, 1, 0, 1)), stride 2) as one ih_conv2d_s2_padbr_f16."""

    def __init__(self, ch: int):
        super().__init__()
        self.conv = nn.Conv2d(ch, ch, 3, stride=2, padding=0)
        self._w = None

    def finalize(self, s: float = 1.0):
        self._w = ops.pack_conv3x3_weight(self.conv.weight.detach())
        self._b = _scaled(self.conv.bias, s)

    def forward(self, x):
        return ops.conv3x3_s2_padbr(x, self._w, self._b)     # linear in the scaled stream: only the bias scales


class VAEDownBlock(nn.Module):
    def __init__(self, cin: int, cout: int, n_res: int, groups: int, add_down: bool):
        super().__init__()
        self.resnets = nn.ModuleList([VAEResnetBlock(cin if j == 0 else cout, cout, groups) for j in range(n_res)])
        if add_down:
            self.downsamplers = nn.ModuleList([VAEDownsample(cout)])
        self.has_down = add_down

    def forward(self, x):
        for r in self.resnets:
            x = r(x)
        return self.downsamplers[0](x) if self.has_down else x


class Encoder(nn.Module):
    def __init__(self, cfg: VAEConfig):
        super().__init__()
        ch = cfg.block_out_channels
        g = cfg.norm_num_groups
        self.conv_in = nn.Conv2d(cfg.in_channels, ch[0], 3, padding=1)
        downs: List[nn.Module] = []
        prev = ch[0]
        for i, c in enumerate(ch):
            downs.append(VAEDownBlock(prev, c, cfg.layers_per_block, g, add_down=i < len(ch) - 1))
            prev = c
        self.down_blocks = nn.ModuleList(downs)
        self.mid_block = VAEMidBlock(ch[-1], g)
        self.conv_norm_out = nn.GroupNorm(g, ch[-1], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[-1], 2 * cfg.latent_channels, 3, padding=1)


class AutoencoderKLEncoder(nn.Module):
    """`encode(image)` = the moments of diffusers `vae.encode(image).latent_dist` (mean, logvar); the posterior sample,
    `scaling_factor` and the scheduler's `add_noise` follow in one kernel (`ops.vae_sample_add_noise`).

    * conv_in (3 -> C) is a GEMM over the im2col rows of the image: straight from the uint8 PIL pixels
      (`ih_image_im2col3x3_u8`, which also normalises 2 v / 255 - 1) or from a float NCHW tensor in [-1, 1]
      (`ih_im2col3x3_nchw_f16`);
    * down blocks of ResnetBlock2D (the decoder's VAEResnetBlock) and Downsample2D(padding=0) (`ih_conv2d_s2_padbr_f16`),
      the decoder's mid block (resnet, attention, resnet);
    * GroupNorm + SiLU, then conv_out with quant_conv folded in: W' = Wq Wco, b' = Wq bco + bq (exact in real
      arithmetic), Cout padded 8 -> 16.  The moments come out as NHWC [B, h, w, 16], channels [0, L) mean,
      [L, 2L) logvar.

    The residual stream is scaled by `stream_scale` exactly as in the decoder (module docstring); conv_out reads the
    GroupNorm output, so the moments are at scale 1."""

    def __init__(self, cfg: VAEConfig = SDXL_VAE):
        super().__init__()
        self.config = cfg
        self.encoder = Encoder(cfg)
        self.quant_conv = nn.Conv2d(2 * cfg.latent_channels, 2 * cfg.latent_channels, 1)
        self._w_in = self._w_out = self._b_out = None
        self.use_tiling = False             # pipeline.enable_vae_tiling() (test.py:73)
        self.stream_scale = 2.0 ** -7 if getattr(cfg, "force_upcast", True) else 1.0

    KPAD_IN = 32                            # conv_in: 3 * 9 = 27 im2col columns padded to a multiple of 8
    COUT_PAD = 16                           # conv_out: 2 L = 8 moment channels padded to 16

    @classmethod
    def from_state_dict(cls, cfg: VAEConfig, sd: Dict[str, torch.Tensor], device="cuda",
                        stream_scale: Optional[float] = None) -> "AutoencoderKLEncoder":
        """Loads the `encoder.*` / `quant_conv.*` keys of a diffusers AutoencoderKL state dict (other keys ignored)."""
        with torch.device("meta"):
            m = cls(cfg)
        if stream_scale is not None:
            if stream_scale <= 0 or math.log2(stream_scale) != int(math.log2(stream_scale)):
                raise IHError("stream_scale must be a power of two")
            m.stream_scale = float(stream_scale)
        m = m.to_empty(device=device)
        own = m.state_dict()
        missing = [k for k in own if k not in sd]
        if missing:
            raise KeyError(f"VAE checkpoint lacks {len(missing)} encoder keys, e.g. {missing[:3]}")
        m.load_state_dict({k: sd[k].to(device=device, dtype=torch.float16).reshape(own[k].shape) for k in own})
        m = m.half().eval()
        m.finalize()
        return m

    def finalize(self) -> None:
        s = self.stream_scale
        for mod in self.modules():
            if isinstance(mod, (VAEResnetBlock, VAEAttention, VAEDownsample)):
                mod.finalize(s)
        enc = self.encoder
        dt = enc.conv_in.weight.dtype
        w_in = enc.conv_in.weight.detach()
        C0 = w_in.shape[0]
        w = torch.zeros((C0, self.KPAD_IN), dtype=dt, device=w_in.device)
        w[:, :w_in[0].numel()] = w_in.reshape(C0, -1)                                 # k = ci*9 + ky*3 + kx
        self._w_in = w.contiguous()
        self._b_in = _scaled(enc.conv_in.bias, s)
        L2 = 2 * self.config.latent_channels
        wq = self.quant_conv.weight.detach().float().reshape(L2, L2)                    # [o, m]
        wco = enc.conv_out.weight.detach().float()                                     # [m, C, 3, 3]
        folded_w = torch.einsum("om,mcyx->ocyx", wq, wco)
        folded_b = wq @ enc.conv_out.bias.detach().float() + self.quant_conv.bias.detach().float()
        w_out = torch.zeros((self.COUT_PAD,) + tuple(wco.shape[1:]), dtype=dt, device=wco.device)
        w_out[:L2] = folded_w.to(dt)
        self._w_out = ops.pack_conv3x3_weight(w_out)
        b_out = torch.zeros((self.COUT_PAD,), dtype=dt, device=wco.device)
        b_out[:L2] = folded_b.to(dt)
        self._b_out = b_out

    # ---- forward -----------------------------------------------------------------------------------------------
    @torch.no_grad()
    def encode(self, image: torch.Tensor) -> torch.Tensor:
        """image: uint8 RGB NHWC [B, H, W, 3] (PIL pixels) or float NCHW [B, 3, H, W] in [-1, 1]; H, W multiples of 8.
        Returns the moments NHWC [B, H/8, W/8, 16] (fp16; channels [0, L) mean, [L, 2L) logvar, the rest zero).
        With `use_tiling` and an image larger than one tile (`sample_size` pixels) the image is encoded tile by tile and
        the moments are blended, [3P] diffusers `AutoencoderKL.tiled_encode`."""
        if self._w_in is None:
            raise IHError("AutoencoderKLEncoder.finalize() has not run (use from_state_dict)")
        nhwc = image.dtype == torch.uint8
        H, W = (image.shape[1], image.shape[2]) if nhwc else (image.shape[2], image.shape[3])
        if H % 8 or W % 8:
            raise IHError(f"VAE encoder: image size {H}x{W} is not a multiple of 8")
        t = self.config.sample_size
        if self.use_tiling and (H > t or W > t):
            return self._tiled_encode(image, nhwc)
        return self._encode_tile(image, nhwc)

    def _tiled_encode(self, x: torch.Tensor, nhwc: bool) -> torch.Tensor:
        """[3P] tiled_encode: tiles of `sample_size` pixels every (1 - overlap) tile, each encoded on its own, the moments
        cross-faded over `tile_latent_min_size * overlap` latents with the tile above and the tile to the left and
        cropped to the rest of the latent tile.  The cross-fade is elementwise torch glue (NHWC moments)."""
        cfg = self.config
        ts = cfg.sample_size
        stride = int(ts * (1 - cfg.tile_overlap_factor))
        blend = int(cfg.tile_latent_min_size * cfg.tile_overlap_factor)
        limit = cfg.tile_latent_min_size - blend
        H, W = (x.shape[1], x.shape[2]) if nhwc else (x.shape[2], x.shape[3])
        rows = []
        for i in range(0, H, stride):
            row = []
            for j in range(0, W, stride):
                tile = x[:, i:i + ts, j:j + ts, :] if nhwc else x[:, :, i:i + ts, j:j + ts]
                row.append(self._encode_tile(tile.contiguous(), nhwc).float())
            rows.append(row)

        def blend_v(a, b, ext):
            ext = min(a.shape[1], b.shape[1], ext)
            wgt = (torch.arange(ext, device=b.device, dtype=torch.float32) / ext).view(1, ext, 1, 1)
            b[:, :ext] = a[:, -ext:] * (1 - wgt) + b[:, :ext] * wgt
            return b

        def blend_h(a, b, ext):
            ext = min(a.shape[2], b.shape[2], ext)
            wgt = (torch.arange(ext, device=b.device, dtype=torch.float32) / ext).view(1, 1, ext, 1)
            b[:, :, :ext] = a[:, :, -ext:] * (1 - wgt) + b[:, :, :ext] * wgt
            return b

        out_rows = []
        for i, row in enumerate(rows):
            out_row = []
            for j, tile in enumerate(row):
                if i > 0:
                    tile = blend_v(rows[i - 1][j], tile, blend)
                if j > 0:
                    tile = blend_h(row[j - 1], tile, blend)
                out_row.append(tile[:, :limit, :limit])
            out_rows.append(torch.cat(out_row, dim=2))
        return torch.cat(out_rows, dim=1).to(self._w_in.dtype).contiguous()

    def _encode_tile(self, x: torch.Tensor, nhwc: bool) -> torch.Tensor:
        enc = self.encoder
        dt = self._w_in.dtype                                     # fp16 on the GPU (fp32 only in the CPU wiring test)
        if nhwc:
            B, H, W, _ = x.shape
            a = ops.image_im2col3x3(x, self.KPAD_IN)
        else:
            B, _, H, W = x.shape
            a = ops.im2col3x3_nchw(x.to(dt).contiguous(), self.KPAD_IN)
        s = self.stream_scale
        h = ops.linear(a, self._w_in, self._b_in, alpha=s).reshape(B, H, W, -1)       # s * conv_in(image)
        for blk in enc.down_blocks:
            h = blk(h)
        h = enc.mid_block(h)
        g = self.config.norm_num_groups
        h = ops.groupnorm(h, enc.conv_norm_out.weight, enc.conv_norm_out.bias, groups=g, eps=1e-6 * s * s, silu=True)
        return ops.conv3x3(h, self._w_out, self._b_out)                               # quant_conv(conv_out(.)), scale 1



def postprocess(image: torch.Tensor, output_type: str = "pil"):
    """[3P] diffusers VaeImageProcessor.postprocess as used at custom_pipelines.py:383: denormalise to [0, 1], NHWC,
    uint8 rounding, PIL.  `output_type` in {"pt", "np", "pil"}."""
    img = (image.float() / 2 + 0.5).clamp(0, 1)
    if output_type == "pt":
        return img
    arr = img.permute(0, 2, 3, 1).cpu().numpy()
    if output_type == "np":
        return arr
    if output_type != "pil":
        raise IHError(f"unknown output_type {output_type!r}")
    from PIL import Image
    u8 = (arr * 255).round().astype("uint8")
    return [Image.fromarray(a) for a in u8]
