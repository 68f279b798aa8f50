"""Model assembly for ``FastEditor``: maps the reference's ``MODEL_CONFIGS`` names (``src/pipeline.py:30-43``) and
ControlNet choice (``:82-87``) to configs + weights.  No checkpoints exist offline, so weights come from the seeded
synthetic recipe (:mod:`.synthetic`); a diffusers-style state dict can be passed instead (real-weight loading is
SURVEY 8(f)-3)."""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import configs as C
from . import synthetic as S


def model_configs(model_name: str, full_controlnet: bool = False, tiny: bool = False):
    if tiny:
        return C.tiny_unet_config(), C.tiny_controlnet_config(full_controlnet), C.tiny_vae_config()
    if model_name == "sdxl":
        ucfg = C.sdxl_unet_config()
    elif model_name == "ssd-1b":
        ucfg = C.ssd1b_unet_config()
    else:
        raise ValueError(f"Unknown model: {model_name}. Choose from ['sdxl', 'ssd-1b']")
    return ucfg, C.controlnet_config(full_controlnet), C.VAEConfig()


def synthetic_state(model_name: str, full_controlnet: bool = False, tiny: bool = False) -> Dict:
    """fp32 master weights on the CPU: dict(unet_cfg, unet, cn_cfg, cn, vae_cfg, vae, lora, lora_scale)."""
    ucfg, ccfg, vcfg = model_configs(model_name, full_controlnet, tiny)
    unet = S.make_unet_params(ucfg)
    # the reference applies LCM-LoRA (r=64, alpha=64 -> scale 1.0) to SDXL only; SSD-1B uses a full LCM UNet
    lora = S.make_lora_params(unet, rank=8 if tiny else 64) if model_name == "sdxl" else None
    return dict(unet_cfg=ucfg, unet=unet, cn_cfg=ccfg, cn=S.make_controlnet_params(ccfg), vae_cfg=vcfg, vae=S.make_vae_params(vcfg),
                lora=lora, lora_scale=1.0)


def build_engine(state: Dict, device="cuda", pack_on_host: bool = False):
    from .pipeline import EditEngine
    return EditEngine(state["unet"], state["unet_cfg"], state["cn"], state["cn_cfg"], state["vae"], state["vae_cfg"], device,
                      state.get("lora"), state.get("lora_scale", 1.0), pack_on_host=pack_on_host, vae_scores_f32=bool(state.get("vae_scores_f32", False)),
                      vae_dtype=state.get("vae_dtype", torch.float16))
