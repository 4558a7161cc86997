"""Architecture description of the SDXL-base UNet the reference drives (custom_pipelines.py:338-345) plus the
IMAGHarmony adapter hyper-parameters (test.py:12-15, ip_adapter.py:99-123). [3P] values are the public
stabilityai/stable-diffusion-xl-base-1.0 unet/config.json restated in SURVEY.md appendix A.1."""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Tuple


@dataclass(frozen=True)
class UNetConfig:
    in_channels: int = 4
    out_channels: int = 4
    block_out_channels: Tuple[int, ...] = (320, 640, 1280)
    layers_per_block: int = 2
    # transformer depth per resolution level; 0 = no attention at that level (DownBlock2D / UpBlock2D)
    transformer_layers_per_block: Tuple[int, ...] = (0, 2, 10)
    attention_head_dim: int = 64
    cross_attention_dim: int = 2048
    norm_num_groups: int = 32
    addition_time_embed_dim: int = 256
    pooled_embed_dim: int = 1280          # text_embeds width (projection_class_embeddings_input_dim = 6*256 + 1280)
    sample_size: int = 128
    # IMAGHarmony / IP-Adapter
    num_ip_tokens: int = 4
    ip_target_substring: str = "down_blocks.2.attentions.1"   # ip_adapter.py:117 (hard-coded in the reference)

    @property
    def time_embed_dim(self) -> int:
        return self.block_out_channels[0] * 4

    @property
    def add_embed_in(self) -> int:
        return 6 * self.addition_time_embed_dim + self.pooled_embed_dim

    def heads(self, channels: int) -> int:
        return channels // self.attention_head_dim


SDXL_BASE = UNetConfig()

# A structurally identical miniature (same block types, skip wiring, IP layer placement) used by the CPU-side tests
# and the golden fixtures; channels stay multiples of 64 so every sm_100a kernel path is exercised.
TINY = UNetConfig(
    block_out_channels=(64, 128, 256),
    transformer_layers_per_block=(0, 1, 2),
    cross_attention_dim=128,
    addition_time_embed_dim=32,
    pooled_embed_dim=64,
    sample_size=32,
)


@dataclass(frozen=True)
class HarmonyConfig:
    """HarmonyAttention hyper-parameters (train.py:189-197; shipped values run.sh:17-20, test.py:12-15)."""
    image_hidden_size: int = 1280
    text_context_dim: int = 2048
    inter_dim: int = 2560
    cross_heads: int = 8
    reshape_blocks: int = 8
    cross_value_dim: int = 64
    scale: float = 1.0


HARMONY_DEFAULT = HarmonyConfig()
HARMONY_TINY = HarmonyConfig(image_hidden_size=64, text_context_dim=128, inter_dim=256, cross_heads=4,
                             reshape_blocks=4, cross_value_dim=16)


@dataclass(frozen=True)
class VAEConfig:
    """[3P] diffusers AutoencoderKL of SDXL (decoder and encoder): vae/config.json of stabilityai/stable-diffusion-xl-base-1.0."""
    latent_channels: int = 4
    out_channels: int = 3
    block_out_channels: Tuple[int, ...] = (128, 256, 512, 512)
    layers_per_block: int = 2
    norm_num_groups: int = 32
    scaling_factor: float = 0.13025
    sample_size: int = 1024               # tiling: tiles of sample_size pixels (= sample_size / 8 latents), 25 % overlap
    tile_overlap_factor: float = 0.25
    force_upcast: bool = True             # vae/config.json of SDXL-base: the reference upcasts the VAE to fp32 (custom_pipelines.py:366-371)
    in_channels: int = 3                  # image channels the encoder reads (img2img)

    @property
    def tile_latent_min_size(self) -> int:
        return int(self.sample_size / (2 ** (len(self.block_out_channels) - 1)))

    @property
    def decoder_channels(self) -> Tuple[int, ...]:
        return tuple(reversed(self.block_out_channels))


SDXL_VAE = VAEConfig()
# miniature with the same block structure (mid attention, a channel-changing shortcut); channels stay multiples of 64
# because the implicit-GEMM conv kernel needs Cin % 64 == 0
TINY_VAE = VAEConfig(block_out_channels=(64, 64, 128, 128), layers_per_block=1, norm_num_groups=8, sample_size=64)
