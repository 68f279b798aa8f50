"""Model configurations of the edit path (diffusers ``config.json`` equivalents, SURVEY Appendix A.2-A.4).

``sdxl`` / ``ssd-1b`` are the two entries of the reference's ``FastEditor.MODEL_CONFIGS`` (``src/pipeline.py:30-43``);
ControlNet small/full are chosen at ``src/pipeline.py:82-87``; the VAE at ``:94-105``.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Sequence

# ----------------------------------------------------------------------------------------------
# Configurations (diffusers config.json equivalents)
# ----------------------------------------------------------------------------------------------


@dataclass
class UNetConfig:
    name: str
    in_channels: int = 4
    out_channels: int = 4
    block_out_channels: Sequence[int] = (320, 640, 1280)
    layers_per_block: int = 2
    # transformer depth of each attention in each down block ([] = DownBlock2D without attention)
    down_depths: Sequence[Sequence[int]] = ((), (2, 2), (10, 10))
    # mid block: depth of its Transformer2D, or None for a single attention-free ResnetBlock2D
    mid_depth: Optional[int] = 10
    # up blocks listed in execution order (first = deepest); 3 resnets each
    up_depths: Sequence[Sequence[int]] = ((10, 10, 10), (2, 2, 2), ())
    head_dim: int = 64
    cross_attention_dim: int = 2048
    norm_groups: int = 32
    norm_eps: float = 1e-5
    time_embed_dim: int = 1280
    addition_time_embed_dim: int = 256
    projection_class_embeddings_input_dim: int = 2816
    # synthetic-weight recipe (SURVEY 8(d)): gain folded into conv_out so std(eps) ~ 1
    conv_out_gain: float = 1.0
    seed: int = 0


def sdxl_unet_config() -> UNetConfig:
    return UNetConfig(name="sdxl", seed=11, conv_out_gain=3.0)   # gain calibrated on the fp32 oracle: std(eps) 0.333 -> ~1


def ssd1b_unet_config() -> UNetConfig:
    # segmind/SSD-1B: transformer_layers_per_block [1,[2,2],[4,4]], reverse [[4,4,10],[2,1,1],1],
    # mid = UNetMidBlock2D(num_layers=0, add_attention=False) (SURVEY Appendix A.2)
    return UNetConfig(name="ssd-1b", down_depths=((), (2, 2), (4, 4)), mid_depth=None,
                      up_depths=((4, 4, 10), (2, 1, 1), ()), seed=12, conv_out_gain=3.0)   # calibrated: std(eps) 0.35 -> ~1


def tiny_unet_config(name="tiny", mid_depth: Optional[int] = 1) -> UNetConfig:
    """Small same-topology UNet for CPU-sized parity tests (channels stay multiples of 64)."""
    return UNetConfig(name=name, block_out_channels=(64, 128, 256), down_depths=((), (1, 1), (2, 1)),
                      mid_depth=mid_depth, up_depths=((1, 2, 1), (1, 1, 1), ()), cross_attention_dim=128,
                      time_embed_dim=256, addition_time_embed_dim=32, projection_class_embeddings_input_dim=64 + 6 * 32,
                      seed=21)


@dataclass
class ControlNetConfig:
    name: str
    unet: UNetConfig = field(default_factory=sdxl_unet_config)
    full: bool = False  # full: CrossAttn blocks (1,2,10)+mid depth 10; small: attention-free, 1-resnet mid
    cond_channels: Sequence[int] = (16, 32, 96, 256)
    seed: int = 13


def controlnet_config(full: bool = False, base: Optional[UNetConfig] = None) -> ControlNetConfig:
    base = base or sdxl_unet_config()
    if full:
        enc = UNetConfig(name="cn-full", block_out_channels=base.block_out_channels, down_depths=((), (2, 2), (10, 10)),
                         mid_depth=10, up_depths=(), cross_attention_dim=base.cross_attention_dim,
                         time_embed_dim=base.time_embed_dim, addition_time_embed_dim=base.addition_time_embed_dim,
                         projection_class_embeddings_input_dim=base.projection_class_embeddings_input_dim)
        return ControlNetConfig(name="cn-full", unet=enc, full=True, seed=14)
    enc = UNetConfig(name="cn-small", block_out_channels=base.block_out_channels, down_depths=((), (), ()),
                     mid_depth=None, up_depths=(), cross_attention_dim=base.cross_attention_dim,
                     time_embed_dim=base.time_embed_dim, addition_time_embed_dim=base.addition_time_embed_dim,
                     projection_class_embeddings_input_dim=base.projection_class_embeddings_input_dim)
    return ControlNetConfig(name="cn-small", unet=enc, full=False, seed=13)


def tiny_controlnet_config(full=False) -> ControlNetConfig:
    base = tiny_unet_config()
    enc = UNetConfig(name="cn-tiny", block_out_channels=base.block_out_channels,
                     down_depths=((), (1, 1), (2, 1)) if full else ((), (), ()), mid_depth=1 if full else None,
                     up_depths=(), cross_attention_dim=base.cross_attention_dim, time_embed_dim=base.time_embed_dim,
                     addition_time_embed_dim=base.addition_time_embed_dim,
                     projection_class_embeddings_input_dim=base.projection_class_embeddings_input_dim)
    return ControlNetConfig(name="cn-tiny-full" if full else "cn-tiny", unet=enc, full=full,
                            cond_channels=(16, 32, 96, 256), seed=23)


@dataclass
class VAEConfig:
    name: str = "sdxl-vae"
    block_out_channels: Sequence[int] = (128, 256, 512, 512)
    layers_per_block: int = 2
    latent_channels: int = 4
    norm_groups: int = 32
    norm_eps: float = 1e-6
    scaling_factor: float = 0.13025
    conv_out_gain: float = 1.0  # synthetic recipe: decoder conv_out gain so image std ~0.3-0.5
    seed: int = 15
    # diffusers' AutoencoderKL ``force_upcast`` (config.json): True = the VAE's activations do not fit fp16 (the original SDXL VAE);
    # None = the key is absent.  FastEditor(vae_dtype=None) runs such a VAE in bf16.
    force_upcast: Optional[bool] = None


def tiny_vae_config() -> VAEConfig:
    return VAEConfig(name="tiny-vae", block_out_channels=(64, 64, 128, 128), seed=25)


def skip_channels(cfg: UNetConfig) -> List[int]:
    ch = cfg.block_out_channels
    out = [ch[0]]
    for i, c in enumerate(ch):
        out += [c] * cfg.layers_per_block
        if i < len(ch) - 1:
            out.append(c)
    return out


