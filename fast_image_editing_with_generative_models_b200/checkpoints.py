"""Real-weight loading (SURVEY 8(f)-3): diffusers checkpoint directories -> the engine's state dict.

The reference obtains its weights with ``from_pretrained`` (``ControlNetModel`` ``src/pipeline.py:89-92``, ``AutoencoderKL`` ``:96-105``,
``UNet2DConditionModel`` ``:115-124``, the pipeline ``:128-153``) and ``load_lora_weights`` (``:154``).  No checkpoint or network
exists in this environment, so nothing here can be exercised on the real files; what is implemented and tested (round trip through
the on-disk format, the published SDXL / SSD-1B ``config.json`` contents, kohya- and peft-style LoRA keys) is the mapping:

* ``config.json`` of a diffusers UNet / ControlNet / VAE -> :mod:`.configs` dataclasses;
* ``diffusion_pytorch_model[.fp16].safetensors`` -> fp32 master tensors under diffusers' own parameter names (the engine's packer
  consumes exactly those names);
* LCM-LoRA ``pytorch_lora_weights.safetensors`` (kohya ``lora_unet_*.lora_down/up.weight`` + ``alpha``, or peft ``lora_A/B``) ->
  ``{param}.lora_A.weight`` / ``{param}.lora_B.weight`` with ``alpha / rank`` folded into B."""
from __future__ import annotations

import json
import os
from typing import Dict, Optional, Sequence

import torch

from . import configs as C

Tensor = torch.Tensor


def _per_block(v, n_blocks: int, layers: int):
    """diffusers ``transformer_layers_per_block``: int | [int] | [[int]] -> per block, per layer."""
    if isinstance(v, int):
        v = [v] * n_blocks
    return [list(b) if isinstance(b, (list, tuple)) else [b] * layers for b in v]


def unet_config_from_json(d: Dict, name: str = "unet") -> C.UNetConfig:
    ch = list(d["block_out_channels"])
    lpb = d.get("layers_per_block", 2)
    if not isinstance(lpb, int):
        if len(set(lpb)) != 1:
            raise ValueError("per-block layers_per_block is not supported")
        lpb = lpb[0]
    heads = d.get("attention_head_dim", 8)          # diffusers' misnomer: the number of heads per block
    heads = [heads] * len(ch) if isinstance(heads, int) else list(heads)
    for c, h in zip(ch, heads):
        if c // h != 64:
            raise ValueError(f"attention head size {c // h} != 64 (the flash kernel is specialised for 64)")
    tl = _per_block(d.get("transformer_layers_per_block", 1), len(ch), lpb)
    down_types = d.get("down_block_types", ["CrossAttnDownBlock2D"] * len(ch))
    down = [tuple(tl[i]) if "CrossAttn" in t else () for i, t in enumerate(down_types)]
    mid_type = d.get("mid_block_type", "UNetMidBlock2DCrossAttn")
    if mid_type is None:
        raise ValueError("mid_block_type: null (a UNet without a mid block) is not supported")
    mid = None if mid_type == "UNetMidBlock2D" else int(tl[-1][-1])
    up_types = d.get("up_block_types", ["CrossAttnUpBlock2D"] * len(ch))
    rev = d.get("reverse_transformer_layers_per_block")
    rtl = _per_block(rev, len(ch), lpb + 1) if rev is not None else [[b[-1]] * (lpb + 1) for b in reversed(tl)]
    up = [tuple(rtl[i]) if "CrossAttn" in t else () for i, t in enumerate(up_types)]
    return C.UNetConfig(name=name, in_channels=d.get("in_channels", 4), out_channels=d.get("out_channels", 4), block_out_channels=tuple(ch),
                        layers_per_block=lpb, down_depths=tuple(down), mid_depth=mid, up_depths=tuple(up),
                        cross_attention_dim=d.get("cross_attention_dim", 2048), norm_groups=d.get("norm_num_groups", 32), norm_eps=d.get("norm_eps", 1e-5),
                        time_embed_dim=ch[0] * 4, addition_time_embed_dim=d.get("addition_time_embed_dim", 256),
                        projection_class_embeddings_input_dim=d.get("projection_class_embeddings_input_dim", 2816))


def controlnet_config_from_json(d: Dict, name: str = "controlnet") -> C.ControlNetConfig:
    enc = unet_config_from_json({**d, "up_block_types": []}, name)
    enc.up_depths = ()
    full = any(len(x) for x in enc.down_depths)
    return C.ControlNetConfig(name=name, unet=enc, full=full, cond_channels=tuple(d.get("conditioning_embedding_out_channels", (16, 32, 96, 256))))


def vae_config_from_json(d: Dict, name: str = "vae") -> C.VAEConfig:
    return C.VAEConfig(name=name, block_out_channels=tuple(d["block_out_channels"]), layers_per_block=d.get("layers_per_block", 2),
                       latent_channels=d.get("latent_channels", 4), norm_groups=d.get("norm_num_groups", 32), norm_eps=1e-6,
                       scaling_factor=d.get("scaling_factor", 0.13025),
                       force_upcast=bool(d["force_upcast"]) if d.get("force_upcast") is not None else None)


def _weights_file(folder: str) -> str:
    for f in ("diffusion_pytorch_model.fp16.safetensors", "diffusion_pytorch_model.safetensors"):
        if os.path.exists(os.path.join(folder, f)):
            return os.path.join(folder, f)
    raise FileNotFoundError(f"no diffusion_pytorch_model[.fp16].safetensors in {folder}")


def load_model_dir(folder: str):
    """-> (config.json dict, {name: fp32 CPU tensor})."""
    from safetensors.torch import load_file
    with open(os.path.join(folder, "config.json")) as f:
        cfg = json.load(f)
    return cfg, {k: v.float() for k, v in load_file(_weights_file(folder)).items()}


# model part -> (kohya prefix, peft / diffusers prefix) of the keys of a LoRA file
LORA_PARTS = {"unet": ("lora_unet_", "unet."), "text_encoder": ("lora_te1_", "text_encoder."), "text_encoder_2": ("lora_te2_", "text_encoder_2.")}
_UNSUPPORTED_LORA = ("dora_scale", "hada_", "lokr_")          # DoRA, LyCORIS LoHa / LoKr: not a plain B A delta


def read_lora(src, weight_name: Optional[str] = None) -> Dict[str, Tensor]:
    """``load_lora_weights``' first argument -> a state dict: a dict as it is, a local ``.safetensors`` file, or a folder holding
    ``weight_name`` (default ``pytorch_lora_weights.safetensors``).  Anything else (a hub id) is a ValueError: nothing is downloaded."""
    if isinstance(src, dict):
        return dict(src)
    if not isinstance(src, (str, os.PathLike)):
        raise ValueError(f"LoRA: expected a state dict, a .safetensors file or a folder, not {type(src).__name__}")
    path = os.fspath(src)
    if os.path.isdir(path):
        path = os.path.join(path, weight_name or "pytorch_lora_weights.safetensors")
    if not (path.endswith(".safetensors") and os.path.isfile(path)):
        raise ValueError(f"LoRA: {path!r} is not a local .safetensors file or a folder holding one (hub ids are not supported)")
    from safetensors.torch import load_file
    return load_file(path)


def split_lora(sd: Dict[str, Tensor]) -> Dict[str, Dict[str, Tensor]]:
    """A LoRA state dict -> {part: its keys} for the parts of :data:`LORA_PARTS` that occur.  Keys with no part prefix belong to the UNet
    (peft files saved from a bare UNet).  ValueError for DoRA (``dora_scale``) and LyCORIS LoHa / LoKr keys, and for any key that is not
    a LoRA factor of one of the parts in a layout :func:`lora_to_peft` reads (e.g. SD 1.x ``lora_te_`` keys), or whose partner is missing."""
    bad = [k for k in sd if any(t in k for t in _UNSUPPORTED_LORA)]
    if bad:
        raise ValueError(f"LoRA: unsupported format (DoRA / LyCORIS LoHa / LoKr keys, first: {bad[:2]}); only plain LoRA (B A) deltas are supported")
    parts: Dict[str, Dict[str, Tensor]] = {}
    unknown = []
    for k, v in sd.items():
        part = next((p for p, pre in LORA_PARTS.items() if k.startswith(pre)), "unet")
        if not _lora_key_ok(k, sd, LORA_PARTS[part][0]):
            unknown.append(k)
        parts.setdefault(part, {})[k] = v
    if unknown:             # a key lora_to_peft would skip: a silently dropped tensor would give a quietly different model
        raise ValueError(f"LoRA: {len(unknown)} tensors are not LoRA factors of the UNet or a text encoder in a known layout, or lack their "
                         f"partner (first: {unknown[:3]})")
    return parts


def _lora_key_ok(k: str, sd: Dict[str, Tensor], kohya: str) -> bool:
    """Whether :func:`lora_to_peft` consumes key ``k``: a kohya down / up / alpha key of the part (down and up both present), or a peft
    ``lora_A`` / ``lora_B`` (``lora.down`` / ``lora.up``) weight with its partner.  peft files carry no alpha (it is folded into B)."""
    if k.startswith(kohya):
        for role, other in ((".lora_down.weight", ".lora_up.weight"), (".lora_up.weight", ".lora_down.weight"), (".alpha", ".lora_down.weight")):
            if k.endswith(role):
                return k[: -len(role)] + other in sd
        return False
    for role, other in ((".lora_A.", ".lora_B."), (".lora_B.", ".lora_A."), (".lora.down.", ".lora.up."), (".lora.up.", ".lora.down.")):
        if role in k and k.endswith(".weight"):
            return k.replace(role, other) in sd
    return False


def lora_to_peft(sd: Dict[str, Tensor], param_names: Sequence[str], part: str = "unet") -> Dict[str, Tensor]:
    """LoRA state dict (kohya or peft/diffusers keys) of one model part (:data:`LORA_PARTS`) -> {param}.lora_A.weight /
    {param}.lora_B.weight, ``alpha / rank`` folded into B."""
    kohya, peft = LORA_PARTS[part]
    by_flat = {n[: -len(".weight")].replace(".", "_"): n[: -len(".weight")] for n in param_names if n.endswith(".weight")}
    out: Dict[str, Tensor] = {}
    unmapped = []
    for k, v in sd.items():
        if k.endswith(".lora_down.weight") and k.startswith(kohya):                     # kohya
            flat = k[len(kohya): -len(".lora_down.weight")]
            name = by_flat.get(flat)
            if name is None:
                unmapped.append(k)
                continue
            up = sd[k.replace("lora_down", "lora_up")].float()
            alpha = sd.get(k.replace("lora_down.weight", "alpha"))
            scale = float(alpha) / v.shape[0] if alpha is not None else 1.0
            out[name + ".lora_A.weight"], out[name + ".lora_B.weight"] = v.float(), up * scale
        elif ".lora_A" in k or ".lora.down" in k:                                         # peft / old diffusers
            name = k.split(".lora")[0]
            name = name[len(peft):] if name.startswith(peft) else name
            kb = k.replace(".lora_A", ".lora_B").replace(".lora.down", ".lora.up")
            if name + ".weight" in param_names or name in by_flat.values():
                out[name + ".lora_A.weight"], out[name + ".lora_B.weight"] = v.float(), sd[kb].float()
            else:
                unmapped.append(k)
    if unmapped:            # a silently skipped adapter layer would give a quietly different model
        what = "UNet" if part == "unet" else part
        raise ValueError(f"LoRA: {len(unmapped)} adapter tensors do not match any {what} parameter (first: {unmapped[:3]})")
    return out


def clip_config_from_json(d: Dict, name: str):
    """transformers ``CLIPTextConfig`` JSON (``text_encoder/config.json``) -> :class:`text_encoder.CLIPTextConfig`."""
    from .text_encoder import CLIPTextConfig
    act = d.get("hidden_act", "quick_gelu")
    if act not in ("quick_gelu", "gelu"):
        raise ValueError(f"CLIP text encoder: unsupported hidden_act {act!r}")
    with_proj = "WithProjection" in "".join(d.get("architectures") or [])
    return CLIPTextConfig(name=name, vocab_size=d.get("vocab_size", 49408), hidden_size=d["hidden_size"], num_layers=d["num_hidden_layers"],
                          num_heads=d["num_attention_heads"], intermediate_size=d["intermediate_size"],
                          max_positions=d.get("max_position_embeddings", 77), hidden_act=act, layer_norm_eps=d.get("layer_norm_eps", 1e-5),
                          projection_dim=d.get("projection_dim") if with_proj else None)


def load_clip_dir(folder: str):
    """``text_encoder`` / ``text_encoder_2`` folder of an SDXL pipeline (``config.json`` + ``model[.fp16].safetensors``, transformers
    ``CLIPTextModel`` / ``CLIPTextModelWithProjection`` parameter names) -> (CLIPTextConfig, {name: fp32 CPU tensor})."""
    from safetensors.torch import load_file
    with open(os.path.join(folder, "config.json")) as f:
        cfg = clip_config_from_json(json.load(f), os.path.basename(os.path.normpath(folder)))
    for fn in ("model.fp16.safetensors", "model.safetensors"):
        if os.path.exists(os.path.join(folder, fn)):
            sd = {k: v.float() for k, v in load_file(os.path.join(folder, fn)).items() if "position_ids" not in k}
            if cfg.projection_dim and "text_projection.weight" not in sd:
                raise ValueError(f"{folder}: CLIPTextModelWithProjection checkpoint without text_projection.weight")
            return cfg, sd
    raise FileNotFoundError(f"no model[.fp16].safetensors in {folder}")


def save_clip_dir(folder: str, cfg, params: Dict[str, Tensor], fp16: bool = True):
    """Writes the layout :func:`load_clip_dir` reads (tests, exporting synthetic towers)."""
    from safetensors.torch import save_file
    os.makedirs(folder, exist_ok=True)
    d = {"architectures": ["CLIPTextModelWithProjection" if cfg.projection_dim else "CLIPTextModel"], "vocab_size": cfg.vocab_size,
         "hidden_size": cfg.hidden_size, "num_hidden_layers": cfg.num_layers, "num_attention_heads": cfg.num_heads,
         "intermediate_size": cfg.intermediate_size, "max_position_embeddings": cfg.max_positions, "hidden_act": cfg.hidden_act,
         "layer_norm_eps": cfg.layer_norm_eps, "projection_dim": cfg.projection_dim or cfg.hidden_size}
    with open(os.path.join(folder, "config.json"), "w") as f:
        json.dump(d, f, indent=1)
    save_file({k: (v.half() if fp16 else v.float()).contiguous() for k, v in params.items()},
              os.path.join(folder, "model.fp16.safetensors" if fp16 else "model.safetensors"))


def load_state(unet_dir: str, controlnet_dir: str, vae_dir: str, lora_file: Optional[str] = None, lora_scale: float = 1.0) -> Dict:
    """The dict :func:`model_zoo.build_engine` consumes, from diffusers checkpoint folders (each with ``config.json`` + safetensors)."""
    ucfg_d, unet = load_model_dir(unet_dir)
    ccfg_d, cn = load_model_dir(controlnet_dir)
    vcfg_d, vae = load_model_dir(vae_dir)
    lora = None
    if lora_file:
        from safetensors.torch import load_file
        lora = lora_to_peft(load_file(lora_file), list(unet.keys()))
    return dict(unet_cfg=unet_config_from_json(ucfg_d, os.path.basename(os.path.normpath(unet_dir))), unet=unet,
                cn_cfg=controlnet_config_from_json(ccfg_d), cn=cn, vae_cfg=vae_config_from_json(vcfg_d), vae=vae, lora=lora, lora_scale=lora_scale,
                # real VAE checkpoints produce attention logits in the hundreds: keep them in fp32 between the passes (engine._VAEAttention)
                vae_scores_f32=True)


# ---- writing the same layout (used by the tests and to export synthetic models) ----
def unet_config_to_json(c: C.UNetConfig) -> Dict:
    return {"_class_name": "UNet2DConditionModel", "in_channels": c.in_channels, "out_channels": c.out_channels, "block_out_channels": list(c.block_out_channels),
            "layers_per_block": c.layers_per_block, "attention_head_dim": [ch // c.head_dim for ch in c.block_out_channels],
            "down_block_types": ["CrossAttnDownBlock2D" if len(d) else "DownBlock2D" for d in c.down_depths],
            "up_block_types": ["CrossAttnUpBlock2D" if len(d) else "UpBlock2D" for d in c.up_depths],
            "mid_block_type": "UNetMidBlock2DCrossAttn" if c.mid_depth is not None else "UNetMidBlock2D",
            "transformer_layers_per_block": [list(d) if len(d) else ([c.mid_depth or 1] * c.layers_per_block if i == len(c.down_depths) - 1 else 1)
                                             for i, d in enumerate(c.down_depths)],
            "reverse_transformer_layers_per_block": [list(d) if len(d) else 1 for d in c.up_depths] if len(c.up_depths) else None,
            "cross_attention_dim": c.cross_attention_dim, "norm_num_groups": c.norm_groups, "norm_eps": c.norm_eps,
            "addition_time_embed_dim": c.addition_time_embed_dim, "projection_class_embeddings_input_dim": c.projection_class_embeddings_input_dim}


def save_model_dir(folder: str, cfg_json: Dict, params: Dict[str, Tensor], fp16: bool = True):
    from safetensors.torch import save_file
    os.makedirs(folder, exist_ok=True)
    with open(os.path.join(folder, "config.json"), "w") as f:
        json.dump(cfg_json, f, indent=1)
    name = "diffusion_pytorch_model.fp16.safetensors" if fp16 else "diffusion_pytorch_model.safetensors"
    save_file({k: (v.half() if fp16 else v.float()).contiguous() for k, v in params.items()}, os.path.join(folder, name))
