"""CLIP text encoders on the fie_b200 kernels — SURVEY 8(f)-1, the stage next to the path: the two encoders the SDXL pipeline runs in
``encode_prompt`` before the denoising loop (loaded implicitly by the reference at ``src/pipeline.py:128-135,147-153``):
CLIP ViT-L/14 text (12 layers x 768, quick-GELU) and OpenCLIP bigG/14 text (32 layers x 1280, GELU, with ``text_projection``).
Parameter names are transformers' ``CLIPTextModel`` / ``CLIPTextModelWithProjection`` (``text_model.encoder.layers.N...``), so a real
checkpoint drops in; the tokenizer (CLIP BPE, vocabulary files unavailable offline) is out of scope — callers pass token ids.

Per layer: LayerNorm -> fused q/k/v GEMM (+bias) -> causal flash attention (head_dim 64) -> out-proj GEMM (+bias, +residual)
-> LayerNorm -> fc1 GEMM (+bias, activation in the epilogue) -> fc2 GEMM (+bias, +residual)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch

from . import ops
from .weights import LoraTarget

Tensor = torch.Tensor


@dataclass
class CLIPTextConfig:
    name: str = "clip-vit-l-text"
    vocab_size: int = 49408
    hidden_size: int = 768
    num_layers: int = 12
    num_heads: int = 12
    intermediate_size: int = 3072
    max_positions: int = 77
    hidden_act: str = "quick_gelu"            # "quick_gelu" (CLIP-L) or "gelu" (OpenCLIP bigG)
    layer_norm_eps: float = 1e-5
    projection_dim: Optional[int] = None      # set for CLIPTextModelWithProjection (bigG: 1280)
    seed: int = 31


def clip_l_config() -> CLIPTextConfig:        # openai/clip-vit-large-patch14 text tower (SDXL text_encoder)
    return CLIPTextConfig()


def openclip_bigg_config() -> CLIPTextConfig:  # laion/CLIP-ViT-bigG-14 text tower (SDXL text_encoder_2)
    return CLIPTextConfig(name="openclip-bigg-text", hidden_size=1280, num_layers=32, num_heads=20, intermediate_size=5120,
                          hidden_act="gelu", projection_dim=1280, seed=32)


def tiny_clip_config(proj: bool = False, act: str = "quick_gelu") -> CLIPTextConfig:
    return CLIPTextConfig(name="clip-tiny", vocab_size=1000, hidden_size=128, num_layers=3, num_heads=2, intermediate_size=256,
                          hidden_act=act, projection_dim=64 if proj else None, seed=33)


def make_clip_params(cfg: CLIPTextConfig) -> Dict[str, Tensor]:
    """Seeded random-init state dict with transformers' key names (fp32, CPU)."""
    g = torch.Generator("cpu").manual_seed(cfg.seed)
    c, p = cfg.hidden_size, {}
    rn = lambda *shape, std=0.02: torch.randn(shape, generator=g) * std
    p["text_model.embeddings.token_embedding.weight"] = rn(cfg.vocab_size, c)
    p["text_model.embeddings.position_embedding.weight"] = rn(cfg.max_positions, c, std=0.01)
    for i in range(cfg.num_layers):
        pre = f"text_model.encoder.layers.{i}."
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            p[pre + f"self_attn.{n}.weight"] = rn(c, c, std=c ** -0.5)
            p[pre + f"self_attn.{n}.bias"] = rn(c, std=0.02)
        for n in ("layer_norm1", "layer_norm2"):
            p[pre + n + ".weight"] = 1.0 + rn(c, std=0.05)
            p[pre + n + ".bias"] = rn(c, std=0.05)
        p[pre + "mlp.fc1.weight"] = rn(cfg.intermediate_size, c, std=c ** -0.5)
        p[pre + "mlp.fc1.bias"] = rn(cfg.intermediate_size, std=0.02)
        p[pre + "mlp.fc2.weight"] = rn(c, cfg.intermediate_size, std=cfg.intermediate_size ** -0.5)
        p[pre + "mlp.fc2.bias"] = rn(c, std=0.02)
    p["text_model.final_layer_norm.weight"] = 1.0 + rn(c, std=0.05)
    p["text_model.final_layer_norm.bias"] = rn(c, std=0.05)
    if cfg.projection_dim:
        p["text_projection.weight"] = rn(cfg.projection_dim, c, std=c ** -0.5)
    return p


class CLIPTextEncoder:
    """One CLIP text tower on one GPU.  ``forward(ids)`` -> (penultimate hidden states [B,T,C], last hidden state after the final
    LayerNorm at the EOS token [B,C], text_embeds [B,proj] or None) — what ``encode_prompt`` takes from transformers' outputs
    (``hidden_states[-2]``, ``pooler_output``, ``text_embeds``)."""

    def __init__(self, params: Dict[str, Tensor], cfg: CLIPTextConfig, device):
        if cfg.hidden_size % 64 or cfg.hidden_size // cfg.num_heads != 64:
            raise ValueError("CLIPTextEncoder: head_dim must be 64")
        self.cfg, self.dev = cfg, torch.device(device)
        self.param_names = list(params)
        h16 = lambda k: params[k].to(self.dev, torch.float16).contiguous()
        f32 = lambda k: params[k].to(self.dev, torch.float32).contiguous()
        self.tok, self.pos = h16("text_model.embeddings.token_embedding.weight"), h16("text_model.embeddings.position_embedding.weight")
        self.layers: List[dict] = []
        for i in range(cfg.num_layers):
            pre = f"text_model.encoder.layers.{i}."
            self.layers.append(dict(
                ln1=(f32(pre + "layer_norm1.weight"), f32(pre + "layer_norm1.bias")), ln2=(f32(pre + "layer_norm2.weight"), f32(pre + "layer_norm2.bias")),
                wqkv=torch.cat([h16(pre + f"self_attn.{n}.weight") for n in ("q_proj", "k_proj", "v_proj")], 0).contiguous(),
                bqkv=torch.cat([f32(pre + f"self_attn.{n}.bias") for n in ("q_proj", "k_proj", "v_proj")], 0).contiguous(),
                wo=h16(pre + "self_attn.out_proj.weight"), bo=f32(pre + "self_attn.out_proj.bias"),
                w1=h16(pre + "mlp.fc1.weight"), b1=f32(pre + "mlp.fc1.bias"), w2=h16(pre + "mlp.fc2.weight"), b2=f32(pre + "mlp.fc2.bias")))
        self.lnf = (f32("text_model.final_layer_norm.weight"), f32("text_model.final_layer_norm.bias"))
        self.proj = h16("text_projection.weight") if cfg.projection_dim else None
        self.act = ops.ACT_QUICKGELU if cfg.hidden_act == "quick_gelu" else ops.ACT_GELU

    def lora_targets(self) -> Dict[str, LoraTarget]:
        """{transformers module name: :class:`weights.LoraTarget`} of the projections a text-encoder LoRA adapts (plain rows; q/k/v fused)."""
        c, out = self.cfg.hidden_size, {}
        for i, L in enumerate(self.layers):
            pre = f"text_model.encoder.layers.{i}."
            for j, n in enumerate(("q_proj", "k_proj", "v_proj")):
                out[pre + "self_attn." + n] = LoraTarget("rows", L["wqkv"], c, c, row0=j * c)
            out[pre + "self_attn.out_proj"] = LoraTarget("rows", L["wo"], c, c)
            out[pre + "mlp.fc1"] = LoraTarget("rows", L["w1"], self.cfg.intermediate_size, c)
            out[pre + "mlp.fc2"] = LoraTarget("rows", L["w2"], c, self.cfg.intermediate_size)
        if self.proj is not None:
            out["text_projection"] = LoraTarget("rows", self.proj, self.cfg.projection_dim, c)
        return out

    @torch.no_grad()
    def forward(self, ids: Tensor) -> Tuple[Tensor, Tensor, Optional[Tensor]]:
        cfg = self.cfg
        b, t = ids.shape
        c, heads = cfg.hidden_size, cfg.num_heads
        if not ids.is_cuda:
            # through PyTorch's pinned-host cache, asynchronously: a pageable H2D copy would make the host wait for everything already
            # queued on the stream (the previous micro-batch's whole edit) and serialise FastEditor.edit_many's pipeline
            ids = ids.to(torch.int32).pin_memory().to(self.dev, non_blocking=True)
        ids = ids.to(self.dev)
        h = ops.embed_tokens(ids.to(torch.int32).contiguous(), self.tok, self.pos)          # [b*t, c]
        penultimate = h
        for i, L in enumerate(self.layers):
            if i == cfg.num_layers - 1:
                penultimate = h                                                            # hidden_states[-2]
            n1 = ops.layernorm(h, *L["ln1"], eps=cfg.layer_norm_eps)
            qkv = ops.gemm(n1, L["wqkv"], col_bias=L["bqkv"])
            a = ops.attention_d64(qkv[:, :c], qkv[:, c:2 * c], qkv[:, 2 * c:], b, heads, t, t, causal=True)
            h = ops.gemm(a, L["wo"], col_bias=L["bo"], residual=h)
            n2 = ops.layernorm(h, *L["ln2"], eps=cfg.layer_norm_eps)
            m = ops.gemm(n2, L["w1"], col_bias=L["b1"], act=self.act)
            h = ops.gemm(m, L["w2"], col_bias=L["b2"], residual=h)
        # pooled output: final LayerNorm of the EOS token (the highest id of each sequence, as transformers' CLIPTextTransformer)
        eos = ids.to(torch.int64).argmax(dim=-1) + torch.arange(b, device=self.dev) * t
        pooled = ops.layernorm(h.index_select(0, eos).contiguous(), *self.lnf, eps=cfg.layer_norm_eps)
        embeds = ops.gemm(pooled, self.proj) if self.proj is not None else None
        return penultimate.view(b, t, c), pooled, embeds


class SDXLTextEncoders:
    """``encode_prompt`` of the SDXL pipelines on token ids: prompt_embeds = cat(hidden_states[-2] of both towers) [B,77,2048],
    pooled = text_embeds of the second tower [B,1280]."""

    def __init__(self, params1, cfg1: CLIPTextConfig, params2, cfg2: CLIPTextConfig, device):
        assert cfg2.projection_dim, "the second tower is a CLIPTextModelWithProjection"
        self.enc1, self.enc2 = CLIPTextEncoder(params1, cfg1, device), CLIPTextEncoder(params2, cfg2, device)

    @torch.no_grad()
    def encode(self, ids1: Tensor, ids2: Tensor) -> Tuple[Tensor, Tensor]:
        h1, _, _ = self.enc1.forward(ids1)
        h2, _, e2 = self.enc2.forward(ids2)
        return torch.cat([h1, h2], dim=-1).contiguous(), e2


def pseudo_token_ids(text: str, vocab_size: int = 49408, length: int = 77) -> Tensor:
    """Deterministic stand-in for the CLIP BPE tokenizer (its vocabulary files are not available offline): one id per whitespace
    word by CRC32, BOS = vocab-2, EOS = vocab-1 (the highest id, as in CLIP), padded with EOS."""
    import zlib
    words = text.lower().split()[: length - 2]
    ids = [vocab_size - 2] + [1 + zlib.crc32(w.encode("utf-8")) % (vocab_size - 3) for w in words] + [vocab_size - 1]
    ids += [vocab_size - 1] * (length - len(ids))
    return torch.tensor(ids, dtype=torch.int64)
