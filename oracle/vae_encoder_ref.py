"""CPU restatement of the encoder half of [3P] diffusers==0.30.0 `AutoencoderKL` as an img2img pipeline calls it:
`vae.encode(image).latent_dist.sample(generator)` (DiagonalGaussianDistribution), with the image normalised by
`VaeImageProcessor` (PIL -> fp32 / 255 -> 2 x - 1).  TEST INFRASTRUCTURE ONLY (tests/, tools).  **Parity unpinned**, as
for the decoder (oracle/vae_ref.py): diffusers is not installable here and no golden vector exists for the VAE.

Structure (public SDXL `vae/config.json`): conv_in (3 -> 128), one DownEncoderBlock2D per block_out_channels entry
(layers_per_block ResnetBlock2D, then a Downsample2D(padding=0) = conv3x3(F.pad(x, (0, 1, 0, 1)), stride 2) on every
block but the last), UNetMidBlock2D (resnet, single-head attention, resnet), GroupNorm + SiLU, conv_out (512 -> 2 L,
`double_z`) and quant_conv (1x1, 2 L -> 2 L).  State-dict keys equal diffusers' (`encoder.*`, `quant_conv.*`)."""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .vae_ref import MidRef, ResnetRef


class DownsampleRef(nn.Module):
    def __init__(self, ch):
        super().__init__()
        self.conv = nn.Conv2d(ch, ch, 3, stride=2, padding=0)

    def forward(self, x):
        return self.conv(F.pad(x, (0, 1, 0, 1)))


class DownBlockRef(nn.Module):
    def __init__(self, cin, cout, n_res, groups, add_down):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetRef(cin if j == 0 else cout, cout, groups) for j in range(n_res)])
        if add_down:
            self.downsamplers = nn.ModuleList([DownsampleRef(cout)])
        self.has_down = add_down

    def forward(self, x):
        for r in self.resnets:
            x = r(x)
        return self.downsamplers[0](x) if self.has_down else x


class EncoderRef(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        ch = cfg.block_out_channels
        g = cfg.norm_num_groups
        self.conv_in = nn.Conv2d(cfg.in_channels, ch[0], 3, padding=1)
        downs, prev = [], ch[0]
        for i, c in enumerate(ch):
            downs.append(DownBlockRef(prev, c, cfg.layers_per_block, g, add_down=i < len(ch) - 1))
            prev = c
        self.down_blocks = nn.ModuleList(downs)
        self.mid_block = MidRef(ch[-1], g)
        self.conv_norm_out = nn.GroupNorm(g, ch[-1], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[-1], 2 * cfg.latent_channels, 3, padding=1)

    def forward(self, x):
        x = self.conv_in(x)
        for b in self.down_blocks:
            x = b(x)
        x = self.mid_block(x)
        return self.conv_out(F.silu(self.conv_norm_out(x)))


class VAEEncoderRef(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.config = cfg
        self.encoder = EncoderRef(cfg)
        self.quant_conv = nn.Conv2d(2 * cfg.latent_channels, 2 * cfg.latent_channels, 1)

    def encode(self, image):
        """image NCHW in [-1, 1] -> moments NCHW [B, 2 L, H/8, W/8] (mean, logvar) = the latent_dist parameters."""
        return self.quant_conv(self.encoder(image))


def preprocess_ref(rgb_u8: np.ndarray) -> torch.Tensor:
    """[3P] VaeImageProcessor.preprocess of PIL pixels: uint8 NHWC -> fp32 / 255 (numpy) -> NCHW -> 2 x - 1 (fp32)."""
    x = torch.from_numpy(np.asarray(rgb_u8).astype(np.float32) / 255.0).permute(0, 3, 1, 2)
    return 2.0 * x - 1.0


def posterior_sample_ref(moments: torch.Tensor, eps: torch.Tensor) -> torch.Tensor:
    """[3P] DiagonalGaussianDistribution(moments).sample with the noise `eps` given: fp32 mean + std * eps."""
    mean, logvar = torch.chunk(moments.float(), 2, dim=1)
    std = torch.exp(0.5 * torch.clamp(logvar, -30.0, 20.0))
    return mean + std * eps.float()


def tiled_encode_ref(vae: "VAEEncoderRef", image: torch.Tensor) -> torch.Tensor:
    """[3P] AutoencoderKL.tiled_encode (enable_vae_tiling(), test.py:73): tiles of `sample_size` pixels every
    sample_size * (1 - overlap) pixels, each through encoder + quant_conv on its own, moments blended with the upper and
    the left neighbour over `tile_latent_min_size * overlap` latents and cropped to the rest of the latent tile."""
    cfg = vae.config
    ts = cfg.sample_size
    tl = cfg.tile_latent_min_size
    overlap_size = int(ts * (1 - cfg.tile_overlap_factor))
    blend_extent = int(tl * cfg.tile_overlap_factor)
    row_limit = tl - blend_extent
    rows = []
    for i in range(0, image.shape[2], overlap_size):
        rows.append([vae.encode(image[:, :, i:i + ts, j:j + ts]) for j in range(0, image.shape[3], overlap_size)])
    result_rows = []
    for i, row in enumerate(rows):
        result_row = []
        for j, tile in enumerate(row):
            if i > 0:
                a, b = rows[i - 1][j], tile
                ext = min(a.shape[2], b.shape[2], blend_extent)
                for y in range(ext):
                    b[:, :, y, :] = a[:, :, -ext + y, :] * (1 - y / ext) + b[:, :, y, :] * (y / ext)
            if j > 0:
                a, b = row[j - 1], tile
                ext = min(a.shape[3], b.shape[3], blend_extent)
                for x in range(ext):
                    b[:, :, :, x] = a[:, :, :, -ext + x] * (1 - x / ext) + b[:, :, :, x] * (x / ext)
            result_row.append(tile[:, :, :row_limit, :row_limit])
        result_rows.append(torch.cat(result_row, dim=3))
    return torch.cat(result_rows, dim=2)
