"""Executors for the UNet, ControlNet and VAE of the edit path on the fie_b200 kernels.

These classes mirror the diffusers modules the reference instantiates (``UNet2DConditionModel``
``src/pipeline.py:115-124,147-153``; ``ControlNetModel`` ``:82-92``; ``AutoencoderKL`` ``:94-105``) but run
NHWC fp16 activations through the hand-written kernels in ``csrc/``.  Weights arrive as a diffusers-style state dict
(fp32, any device) plus the config dataclasses of :mod:`.configs`, and are packed once at load time:

* conv3x3 weights -> ``[Cout][kh][kw][Cin]`` fp16 (implicit-GEMM B operand), 1x1 convs / linears -> ``[out][in]``
* q/k/v of self-attention fused into one ``[3C, C]`` projection; every cross-attention k/v projection of the model
  concatenated into ONE ``[sum 2C, ctx]`` matrix (prompt-only, hoisted out of the step loop)
* GEGLU rows interleaved per accumulator tile; all ``time_emb_proj`` of a model concatenated into one matrix with
  ``conv1.bias`` folded in (one GEMM per model per step produces every resnet's time-embedding row bias)
* LCM-LoRA fused: ``W' = W + (alpha/r) B A`` (the reference leaves it unfused, ``src/pipeline.py:154``)
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import ops
from .configs import ControlNetConfig, UNetConfig, VAEConfig, skip_channels
from .weights import LoraTarget, cast_f16, geglu_rows, fold_layernorm, fuse_lora, pack_conv3x3, pack_conv3x3_c8, pack_conv_up2x, pack_geglu

Tensor = torch.Tensor
Params = Dict[str, Tensor]


def _pad32(n: int) -> int:
    return (n + 31) // 32 * 32


def _pad64(n: int) -> int:
    return (n + 63) // 64 * 64


class _Packer:
    """Pulls tensors out of a diffusers-style state dict, applies the LoRA fuse, moves them to the device."""

    def __init__(self, params: Params, device, lora: Optional[Params] = None, lora_scale: float = 1.0, prefix: str = "", dtype=torch.float16):
        self.p, self.dev, self.lora, self.ls, self.prefix = params, device, lora, lora_scale, prefix
        self.dtype = dtype        # element type of the packed GEMM / convolution weights (fp16, or bf16 for the bf16 VAE)

    def w(self, name: str) -> Tensor:
        """fp32 weight on the device with the LoRA delta (if any) fused."""
        w = self.p[self.prefix + name + ".weight"].to(self.dev, torch.float32)
        if self.lora is not None and (name + ".lora_A.weight") in self.lora:
            w = fuse_lora(w, self.lora[name + ".lora_A.weight"].to(self.dev), self.lora[name + ".lora_B.weight"].to(self.dev), self.ls)
        return w

    def b(self, name: str) -> Optional[Tensor]:
        k = self.prefix + name + ".bias"
        return self.p[k].to(self.dev, torch.float32).contiguous() if k in self.p else None

    def has(self, name: str) -> bool:
        return (self.prefix + name + ".weight") in self.p

    def linear(self, name: str) -> Tuple[Tensor, Optional[Tensor]]:
        return cast_f16(self.w(name), self.dtype), self.b(name)

    def conv3(self, name: str, pad_cout_to=None, pad_cin_to=None) -> Tuple[Tensor, Optional[Tensor]]:
        w = pack_conv3x3(self.w(name), pad_cout_to, pad_cin_to, self.dtype)
        b = self.b(name)
        if b is not None and pad_cout_to and pad_cout_to > b.numel():
            bp = torch.zeros(pad_cout_to, dtype=torch.float32, device=self.dev)
            bp[: b.numel()] = b
            b = bp
        return w, b

    def conv_up(self, name: str) -> Tuple[Tensor, Optional[Tensor]]:
        """Upsample2D conv: phase-decomposed weights for the fused nearest-2x upsample + conv3x3 kernel."""
        return pack_conv_up2x(self.w(name), self.dtype), self.b(name)

    def conv1(self, name: str) -> Tuple[Tensor, Optional[Tensor]]:
        w = self.w(name)
        return cast_f16(w.reshape(w.shape[0], w.shape[1]), self.dtype), self.b(name)

    def cin4(self, name: str) -> Tuple[Tensor, Optional[Tensor]]:
        """[Cout, Cin<=4, 3, 3] -> fp32 [Cout, 3, 3, 4] for the CUDA-core conv_in kernel."""
        w = self.w(name)
        out = torch.zeros((w.shape[0], 3, 3, 4), dtype=torch.float32, device=self.dev)
        out[..., : w.shape[1]] = w.permute(0, 2, 3, 1)
        return out.contiguous(), self.b(name)

    def c8(self, name: str, pad_cout_to=None) -> Tuple[Tensor, Optional[Tensor]]:
        """[Cout, Cin<=8, 3, 3] -> fp16 [Cout_p, 192] for the tensor-core conv_in on a zero-padded 8-channel image (fp16 also for the
        bf16 VAE: its inputs are bounded, only its output is bf16)."""
        w = pack_conv3x3_c8(self.w(name), pad_cout_to)
        b = self.b(name)
        if b is not None and pad_cout_to and pad_cout_to > b.numel():
            bp = torch.zeros(pad_cout_to, dtype=torch.float32, device=self.dev)
            bp[: b.numel()] = b
            b = bp
        return w, b

    def norm(self, name: str) -> Tuple[Tensor, Tensor]:
        return self.p[self.prefix + name + ".weight"].to(self.dev, torch.float32).contiguous(), self.b(name)


# ------------------------------------------------------------------------------------------------
# Building blocks
# ------------------------------------------------------------------------------------------------


class Resnet:
    """diffusers ResnetBlock2D: GN+SiLU -> conv3x3 (+time-embedding row bias) -> GN+SiLU -> conv3x3 (+shortcut)."""

    def __init__(self, pk: _Packer, pre: str, eps: float, groups: int, temb_slot: Optional[List] = None):
        self.eps, self.groups = eps, groups
        self.out_gn = 0       # > 0: conv2 also accumulates the GroupNorm statistics of the block output for its consumer
        self.n1 = pk.norm(pre + ".norm1")
        self.n2 = pk.norm(pre + ".norm2")
        self.w1, b1 = pk.conv3(pre + ".conv1")
        self.w2, self.b2 = pk.conv3(pre + ".conv2")
        self.cout = self.w1.shape[0]
        self.b1 = b1
        self.temb_off = None
        if pk.has(pre + ".time_emb_proj") and temb_slot is not None:
            tw, tb = pk.linear(pre + ".time_emb_proj")
            self.temb_off = sum(t[0].shape[0] for t in temb_slot)
            temb_slot.append((tw, tb + b1))       # conv1.bias folded into the time-embedding row bias
            self.b1 = None
        self.sc = pk.conv1(pre + ".conv_shortcut") if pk.has(pre + ".conv_shortcut") else None

    def lora_targets(self, pre: str, temb_w: Tensor, out: Dict[str, LoraTarget]):
        cin = self.w1.shape[1] // 9
        out[pre + ".conv1"] = LoraTarget("conv3", self.w1, self.cout, cin)
        out[pre + ".conv2"] = LoraTarget("conv3", self.w2, self.cout, self.cout)
        if self.sc is not None:
            out[pre + ".conv_shortcut"] = LoraTarget("rows", self.sc[0], self.cout, self.sc[0].shape[1])
        if self.temb_off is not None:
            out[pre + ".time_emb_proj"] = LoraTarget("rows", temb_w, self.cout, temb_w.shape[1], row0=self.temb_off)

    def __call__(self, x: Tensor, temb_all: Optional[Tensor] = None, skip: Optional[Tensor] = None) -> Tensor:
        n, h, w, _ = x.shape
        hcur = ops.groupnorm(x, self.n1[0], self.n1[1], self.eps, True, self.groups, skip)
        gn = self.groups if self.w1.dtype == torch.float16 else 0      # bf16: no producer-side GroupNorm statistics
        if self.temb_off is not None:
            rb = temb_all[:, self.temb_off:self.temb_off + self.cout]
            hcur = ops.conv3x3(hcur, self.w1, row_bias=rb, rows_per_group=h * w, gn_groups=gn)
        else:
            hcur = ops.conv3x3(hcur, self.w1, col_bias=self.b1, gn_groups=gn)
        hcur = ops.groupnorm(hcur, self.n2[0], self.n2[1], self.eps, True, self.groups)
        if self.sc is not None:
            res = ops.gemm(x, self.sc[0], a1=skip, col_bias=self.sc[1])
        else:
            assert skip is None
            res = x
        return ops.conv3x3(hcur, self.w2, col_bias=self.b2, residual=res, gn_groups=self.out_gn)


class TransformerBlock:
    """BasicTransformerBlock.  The three LayerNorms never run as kernels: the GEMM that produces each residual
    stream also accumulates its row statistics (ln_out), and the GEMM that consumes LN(x) runs on the raw rows with gamma, beta
    and the mean subtraction folded into its weights (weights.fold_layernorm) and scales by 1/sigma in its epilogue (ln_in)."""
    LN_EPS = 1e-5

    def __init__(self, pk: _Packer, pre: str, c: int, kv_slot: List):
        self.c = c
        ln1, ln2, ln3 = pk.norm(pre + ".norm1"), pk.norm(pre + ".norm2"), pk.norm(pre + ".norm3")
        self.ln = (ln1, ln2, ln3)          # kept for LoRA deltas of the folded projections (lora_targets)
        wqkv = torch.cat([pk.w(f"{pre}.attn1.{n}") for n in ("to_q", "to_k", "to_v")], 0)
        self.wo1 = pk.linear(pre + ".attn1.to_out.0")
        self.kv_off = sum(t.shape[0] for t in kv_slot)
        kv_slot.append(cast_f16(torch.cat([pk.w(pre + ".attn2.to_k"), pk.w(pre + ".attn2.to_v")], 0)))
        self.wo2 = pk.linear(pre + ".attn2.to_out.0")
        self.wf = pk.linear(pre + ".ff.net.2")
        self.wqkv, self.bqkv = fold_layernorm(wqkv, None, *ln1)
        self.wq2, self.bq2 = fold_layernorm(pk.w(pre + ".attn2.to_q"), pk.b(pre + ".attn2.to_q"), *ln2)
        self.wg, self.bg = pack_geglu(*fold_layernorm(pk.w(pre + ".ff.net.0.proj"), pk.b(pre + ".ff.net.0.proj"), *ln3))

    def lora_targets(self, pre: str, kv_w: Tensor, out: Dict[str, LoraTarget]):
        c = self.c
        for i, n in enumerate(("to_q", "to_k", "to_v")):
            out[f"{pre}.attn1.{n}"] = LoraTarget("rows", self.wqkv, c, c, row0=i * c, ln=self.ln[0], bias=self.bqkv)
        out[pre + ".attn1.to_out.0"] = LoraTarget("rows", self.wo1[0], c, c)
        out[pre + ".attn2.to_q"] = LoraTarget("rows", self.wq2, c, c, ln=self.ln[1], bias=self.bq2)
        out[pre + ".attn2.to_k"] = LoraTarget("rows", kv_w, c, kv_w.shape[1], row0=self.kv_off)
        out[pre + ".attn2.to_v"] = LoraTarget("rows", kv_w, c, kv_w.shape[1], row0=self.kv_off + c)
        out[pre + ".attn2.to_out.0"] = LoraTarget("rows", self.wo2[0], c, c)
        out[pre + ".ff.net.0.proj"] = LoraTarget("rows", self.wg, self.wg.shape[0], c, ln=self.ln[2], bias=self.bg,
                                                 perm=geglu_rows(self.wg.shape[0], self.wg.device))
        out[pre + ".ff.net.2"] = LoraTarget("rows", self.wf[0], c, self.wf[0].shape[1])

    def __call__(self, h: Tensor, b: int, ntok: int, ctx_kv: Tensor, nctx: int, st: Tensor, st_next: Optional[Tensor] = None) -> Tensor:
        """st: int64 [3, M, 2] row statistics (st[0] already holds those of h); st_next receives those of the result."""
        c, heads = self.c, self.c // 64
        k = ctx_kv[:, self.kv_off:self.kv_off + c]
        v = ctx_kv[:, self.kv_off + c:self.kv_off + 2 * c]
        eps = self.LN_EPS
        qkv = ops.gemm(h, self.wqkv, col_bias=self.bqkv, ln_in=(st[0], eps))
        a = ops.attention_d64(qkv[:, :c], qkv[:, c:2 * c], qkv[:, 2 * c:], b, heads, ntok, ntok)
        h = ops.gemm(a, self.wo1[0], col_bias=self.wo1[1], residual=h, ln_out=st[1])
        q = ops.gemm(h, self.wq2, col_bias=self.bq2, ln_in=(st[1], eps))
        a = ops.attention_d64(q, k, v, b, heads, ntok, nctx)
        h = ops.gemm(a, self.wo2[0], col_bias=self.wo2[1], residual=h, ln_out=st[2])
        g = ops.gemm(h, self.wg, col_bias=self.bg, act=ops.ACT_GEGLU, ln_in=(st[2], eps))
        return ops.gemm(g, self.wf[0], col_bias=self.wf[1], residual=h, ln_out=st_next)


class Transformer2D:
    def __init__(self, pk: _Packer, pre: str, c: int, depth: int, groups: int, kv_slot: List):
        self.c, self.groups = c, groups
        self.norm = pk.norm(pre + ".norm")
        self.pin = pk.linear(pre + ".proj_in")
        self.blocks = [TransformerBlock(pk, f"{pre}.transformer_blocks.{k}", c, kv_slot) for k in range(depth)]
        self.pout = pk.linear(pre + ".proj_out")

    def lora_targets(self, pre: str, kv_w: Tensor, out: Dict[str, LoraTarget]):
        out[pre + ".proj_in"] = LoraTarget("rows", self.pin[0], self.c, self.c)
        out[pre + ".proj_out"] = LoraTarget("rows", self.pout[0], self.c, self.c)
        for k, blk in enumerate(self.blocks):
            blk.lora_targets(f"{pre}.transformer_blocks.{k}", kv_w, out)

    def __call__(self, x: Tensor, ctx_kv: Tensor, nctx: int) -> Tensor:
        n, hh, ww, c = x.shape
        ntok = hh * ww
        h = ops.groupnorm(x, self.norm[0], self.norm[1], 1e-6, False, self.groups)
        fold = bool(self.blocks)
        # one zero-fill for the row statistics of all 3 x depth LayerNorm inputs of this transformer
        st = ops.zeros_i64((3 * len(self.blocks), n * ntok, 2), x.device) if fold else None
        h = ops.gemm(h.view(n * ntok, c), self.pin[0], col_bias=self.pin[1], ln_out=st[0] if fold else None)
        for i, blk in enumerate(self.blocks):
            h = blk(h, n, ntok, ctx_kv, nctx, st[3 * i:3 * i + 3], st[3 * i + 3] if i + 1 < len(self.blocks) else None)
        out = ops.gemm(h, self.pout[0], col_bias=self.pout[1], residual=x.view(n * ntok, c))
        return out.view(n, hh, ww, c)


class _EncoderPart:
    """conv_in, time/add embeddings, down blocks and mid block shared by the UNet and the ControlNet."""

    def __init__(self, pk: _Packer, cfg: UNetConfig):
        self.cfg = cfg
        g, eps = cfg.norm_groups, cfg.norm_eps
        ch = cfg.block_out_channels
        self.temb_slot: List = []
        self.kv_slot: List = []
        self.conv_in = pk.c8("conv_in")           # 4 latent channels -> block_out_channels[0] on the tensor cores (zero-padded 8-channel input)
        self.t1, self.t2 = pk.linear("time_embedding.linear_1"), pk.linear("time_embedding.linear_2")
        self.a1, self.a2 = pk.linear("add_embedding.linear_1"), pk.linear("add_embedding.linear_2")
        self.down: List[dict] = []
        for i in range(len(ch)):
            blk = dict(res=[], attn=[], down=None)
            for j in range(cfg.layers_per_block):
                blk["res"].append(Resnet(pk, f"down_blocks.{i}.resnets.{j}", eps, g, self.temb_slot))
                if len(cfg.down_depths[i]):
                    blk["attn"].append(Transformer2D(pk, f"down_blocks.{i}.attentions.{j}", ch[i], cfg.down_depths[i][j], g, self.kv_slot))
            if i < len(ch) - 1:
                blk["down"] = pk.conv3(f"down_blocks.{i}.downsamplers.0.conv")
            self.down.append(blk)
        self.mid_res0 = Resnet(pk, "mid_block.resnets.0", eps, g, self.temb_slot)
        self.mid_attn = self.mid_res1 = None
        if cfg.mid_depth is not None:
            self.mid_attn = Transformer2D(pk, "mid_block.attentions.0", ch[-1], cfg.mid_depth, g, self.kv_slot)
            self.mid_res1 = Resnet(pk, "mid_block.resnets.1", eps, g, self.temb_slot)

    def finalize(self, dev):
        """Concatenate the per-resnet time_emb_proj and per-block cross-attention k/v projections."""
        self.temb_w = torch.cat([t[0] for t in self.temb_slot], 0).contiguous()
        self.temb_b = torch.cat([t[1] for t in self.temb_slot], 0).contiguous()
        self.kv_w = torch.cat(self.kv_slot, 0).contiguous() if self.kv_slot else None
        self.temb_slot = self.kv_slot = None

    def lora_targets(self, out: Dict[str, LoraTarget]):
        """{diffusers module name: where its packed weight lives} for conv_in, the embeddings, down and mid blocks."""
        w = self.conv_in[0]
        out["conv_in"] = LoraTarget("c8", w, self.cfg.block_out_channels[0], self.cfg.in_channels)
        for name, lin in (("time_embedding.linear_1", self.t1), ("time_embedding.linear_2", self.t2), ("add_embedding.linear_1", self.a1),
                          ("add_embedding.linear_2", self.a2)):
            out[name] = LoraTarget("rows", lin[0], lin[0].shape[0], lin[0].shape[1])
        for i, blk in enumerate(self.down):
            for j, r in enumerate(blk["res"]):
                r.lora_targets(f"down_blocks.{i}.resnets.{j}", self.temb_w, out)
                if blk["attn"]:
                    blk["attn"][j].lora_targets(f"down_blocks.{i}.attentions.{j}", self.kv_w, out)
            if blk["down"] is not None:
                d = blk["down"][0]
                out[f"down_blocks.{i}.downsamplers.0.conv"] = LoraTarget("conv3", d, d.shape[0], d.shape[1] // 9)
        self.mid_res0.lora_targets("mid_block.resnets.0", self.temb_w, out)
        if self.mid_attn is not None:
            self.mid_attn.lora_targets("mid_block.attentions.0", self.kv_w, out)
            self.mid_res1.lora_targets("mid_block.resnets.1", self.temb_w, out)

    # ---- step-invariant (per prompt) work ----
    def prepare_prompt(self, ctx: Tensor, text_embeds: Tensor, time_ids: Sequence[float]):
        """ctx [B,77,D] fp16, text_embeds [B,P] fp16 -> (cross-attention K/V for every block, add-embedding aug)."""
        b = ctx.shape[0]
        cfg = self.cfg
        ctx_kv = ops.gemm(ctx.reshape(b * ctx.shape[1], ctx.shape[2]), self.kv_w) if self.kv_w is not None else None
        tid = ops.sincos_embedding(list(time_ids), cfg.addition_time_embed_dim, ctx.device).view(1, -1).expand(b, -1).contiguous()
        h = ops.gemm(text_embeds, self.a1[0], a1=tid, col_bias=self.a1[1], act=ops.ACT_SILU)
        aug = ops.gemm(h, self.a2[0], col_bias=self.a2[1])
        return ctx_kv, aug

    def time_rows(self, t: Tensor, aug: Tensor) -> Tensor:
        """Per-step: fp32 [B, sum Cout] row biases (time_emb_proj(SiLU(emb)) + conv1.bias) for every resnet.  ``t``: an fp32 CUDA
        tensor [B] with the timestep of each row (read on the device: the edit's parameter block)."""
        b = aug.shape[0]
        if t.numel() != b:
            raise ValueError(f"time_rows: {t.numel()} timesteps for {b} rows")
        te = ops.sincos_embedding(t, self.cfg.block_out_channels[0], aug.device)
        h = ops.gemm(te, self.t1[0], col_bias=self.t1[1], act=ops.ACT_SILU)
        emb = ops.gemm(h, self.t2[0], col_bias=self.t2[1], residual=aug)
        return ops.gemm(ops.silu(emb), self.temb_w, col_bias=self.temb_b, out_f32=True)

    def down_mid(self, h: Tensor, temb: Tensor, ctx_kv: Tensor, nctx: int):
        skips = [h]
        for blk in self.down:
            for j, r in enumerate(blk["res"]):
                h = r(h, temb)
                if blk["attn"]:
                    h = blk["attn"][j](h, ctx_kv, nctx)
                skips.append(h)
            if blk["down"] is not None:
                h = ops.conv3x3(h, blk["down"][0], stride=2, pad_mode=0, col_bias=blk["down"][1])
                skips.append(h)
        h = self.mid_res0(h, temb)
        if self.mid_attn is not None:
            h = self.mid_attn(h, ctx_kv, nctx)
            h = self.mid_res1(h, temb)
        return h, skips


class UNet:
    def __init__(self, params: Params, cfg: UNetConfig, device, lora: Optional[Params] = None, lora_scale: float = 1.0):
        pk = _Packer(params, device, lora, lora_scale)
        self.cfg, self.dev = cfg, device
        self.enc = _EncoderPart(pk, cfg)
        g, eps = cfg.norm_groups, cfg.norm_eps
        ch = cfg.block_out_channels
        rev = list(reversed(ch))
        self.up: List[dict] = []
        for i, cout in enumerate(rev):
            blk = dict(res=[], attn=[], up=None)
            for j in range(cfg.layers_per_block + 1):
                blk["res"].append(Resnet(pk, f"up_blocks.{i}.resnets.{j}", eps, g, self.enc.temb_slot))
                if len(cfg.up_depths[i]):
                    blk["attn"].append(Transformer2D(pk, f"up_blocks.{i}.attentions.{j}", cout, cfg.up_depths[i][j], g, self.enc.kv_slot))
            if i < len(rev) - 1:
                blk["up"] = pk.conv_up(f"up_blocks.{i}.upsamplers.0.conv")
            self.up.append(blk)
        self.norm_out = pk.norm("conv_norm_out")
        self.conv_out = pk.conv3("conv_out", pad_cout_to=32)
        self.enc.finalize(device)

    def prepare_prompt(self, ctx, text_embeds, time_ids):
        return self.enc.prepare_prompt(ctx, text_embeds, time_ids)

    def lora_targets(self) -> Dict[str, LoraTarget]:
        """{diffusers module name: :class:`weights.LoraTarget`} for every Linear / Conv2d of the UNet whose packed weight can take a LoRA
        delta in place (every one of them: the norms are the only parameters left out)."""
        out: Dict[str, LoraTarget] = {}
        self.enc.lora_targets(out)
        for i, blk in enumerate(self.up):
            for j, r in enumerate(blk["res"]):
                r.lora_targets(f"up_blocks.{i}.resnets.{j}", self.enc.temb_w, out)
                if blk["attn"]:
                    blk["attn"][j].lora_targets(f"up_blocks.{i}.attentions.{j}", self.enc.kv_w, out)
            if blk["up"] is not None:
                u = blk["up"][0]
                out[f"up_blocks.{i}.upsamplers.0.conv"] = LoraTarget("up2x", u, u.shape[1], u.shape[2] // 4)
        out["conv_out"] = LoraTarget("conv3", self.conv_out[0], self.cfg.out_channels, self.conv_out[0].shape[1] // 9)
        return out

    def forward(self, x: Tensor, t: Tensor, prompt_state, nctx: int = 77, merge=None) -> Tensor:
        """x [B,H,W,4] fp16, t fp32 CUDA [B] per-row timesteps -> eps [B,H,W,4] fp16 (UNet2DConditionModel.forward with ControlNet
        residuals).  The residuals come through ``merge(skips, h) -> (skips, h)`` (ControlNet.merge_into: the zero-convolution GEMMs
        add this UNet's skip tensors in their epilogue -- no add kernels)."""
        ctx_kv, aug = prompt_state
        cfg = self.cfg
        temb = self.enc.time_rows(t, aug)
        h = ops.conv3x3_c8(ops.pad8(x), self.enc.conv_in[0], col_bias=self.enc.conv_in[1])
        h, skips = self.enc.down_mid(h, temb, ctx_kv, nctx)
        if merge is not None:
            skips, h = merge(skips, h)
        for blk in self.up:
            for j, r in enumerate(blk["res"]):
                h = r(h, temb, skip=skips.pop())
                if blk["attn"]:
                    h = blk["attn"][j](h, ctx_kv, nctx)
            if blk["up"] is not None:
                h = ops.conv_up2x(h, blk["up"][0], col_bias=blk["up"][1])
        h = ops.groupnorm(h, self.norm_out[0], self.norm_out[1], cfg.norm_eps, True, cfg.norm_groups)
        return ops.conv3x3(h, self.conv_out[0], cout_valid=cfg.out_channels, col_bias=self.conv_out[1])


class ControlNet:
    def __init__(self, params: Params, cfg: ControlNetConfig, device):
        pk = _Packer(params, device)
        self.cfg, self.dev = cfg, device
        self.enc = _EncoderPart(pk, cfg.unet)
        cc = list(cfg.cond_channels)
        pads = [_pad64(c) for c in cc]
        self.cond_in = pk.c8("controlnet_cond_embedding.conv_in", pads[0])
        self.cond_blocks = []
        for i in range(len(cc) - 1):
            self.cond_blocks.append((pk.conv3(f"controlnet_cond_embedding.blocks.{2 * i}", pads[i], pads[i]), 1))
            self.cond_blocks.append((pk.conv3(f"controlnet_cond_embedding.blocks.{2 * i + 1}", pads[i + 1], pads[i]), 2))
        self.cond_out = pk.conv3("controlnet_cond_embedding.conv_out", None, pads[-1])
        self.cond_pad0 = pads[0]
        self.cond_c0 = cc[0]
        self.zero = [pk.conv1(f"controlnet_down_blocks.{i}") for i in range(len(skip_channels(cfg.unet)))]
        self.zero_mid = pk.conv1("controlnet_mid_block")
        self.enc.finalize(device)

    def prepare_prompt(self, ctx, text_embeds, time_ids):
        return self.enc.prepare_prompt(ctx, text_embeds, time_ids)

    def cond_embedding(self, cond_p8: Tensor) -> Tensor:
        """cond_p8: zero-padded [N,H+2,W+8,8] fp16 control image in {0,1} (ops.preprocess_pad8).  Step-invariant: once per image."""
        h = ops.conv3x3_c8(cond_p8, self.cond_in[0], col_bias=self.cond_in[1], act=ops.ACT_SILU)   # padded channels: silu(0) = 0
        for (w, b), stride in self.cond_blocks:
            h = ops.conv3x3(h, w, stride=stride, pad_mode=0, col_bias=b, act=ops.ACT_SILU)
        return ops.conv3x3(h, self.cond_out[0], col_bias=self.cond_out[1])

    def encode(self, x: Tensor, t: Tensor, prompt_state, cond_emb: Tensor, nctx: int = 77):
        """The ControlNet up to (not including) its zero convolutions -> (skip features, mid feature); see merge_into.
        t: fp32 CUDA [B] per-row timesteps."""
        ctx_kv, aug = prompt_state
        temb = self.enc.time_rows(t, aug)
        h = ops.conv3x3_c8(ops.pad8(x), self.enc.conv_in[0], col_bias=self.enc.conv_in[1], residual=cond_emb)     # conv_in(x) + conditioning embedding
        return self.enc.down_mid(h, temb, ctx_kv, nctx)

    def merge_into(self, feats, scale: Tensor):
        """-> merge(unet_skips, unet_h): every zero convolution writes scale * (W f + b) + <the UNet tensor it is added to> in one
        GEMM epilogue, i.e. `down_block_res_samples[i] + down_block_additional_residuals[i]` and the mid-block add of
        UNet2DConditionModel.forward without separate element-wise kernels (and with one rounding instead of two).
        ``scale``: an fp32 CUDA tensor with one conditioning scale per batch row (image and CFG half), read on the device as the
        GEMMs' group_scale."""
        cn_h, cn_skips = feats

        def zero_conv(f, w, b, res):
            n_, hh, ww, c_ = res.shape
            return ops.gemm(f.view(-1, f.shape[-1]), w, col_bias=b, residual=res.view(-1, c_), group_scale=scale,
                            rows_per_group=hh * ww).view(res.shape)

        def merge(skips, h):
            merged = [zero_conv(f, w, b, s) for f, (w, b), s in zip(cn_skips, self.zero, skips)]
            return merged, zero_conv(cn_h, self.zero_mid[0], self.zero_mid[1], h)
        return merge


class _VAEAttention:
    """AutoencoderKL mid-block attention: 1 head, d = C (512), N = H*W tokens.  Scores are materialised per row
    chunk in fp32 (GEMM -> row softmax -> GEMM on the tcgen05 GEMM kernel); V is produced transposed so that P V is a
    K-major GEMM."""

    def __init__(self, pk: _Packer, pre: str, groups: int, eps: float):
        self.groups, self.eps = groups, eps
        # fp16 scores by default (scaled in the GEMM epilogue, exp-only softmax in place, 1 / rowsum applied in fp32 by the P V
        # epilogue): half the score traffic, parity unchanged on the synthetic weights (1.5e-2).  fp32 scores, set by
        # VAE(..., attention_scores_f32=True), keep the logits in fp32 between the passes like diffusers' SDPA: the safe choice for
        # REAL checkpoints, whose VAE logits reach the hundreds.
        self.scores_f32 = False
        self.norm = pk.norm(pre + ".group_norm")
        self.q, self.k, self.v, self.o = (pk.linear(f"{pre}.{n}") for n in ("to_q", "to_k", "to_v", "to_out.0"))

    # chunk: query rows whose scores are materialised at a time (0 = the whole image: 512 MiB of fp16 scores at 1024^2).  Measured:
    # small L2-resident chunks lose more in the P V GEMM (M = 1024, N = 512 is 8 tiles on 74 CTA pairs) than they save in HBM traffic;
    # with a whole image per pass the P V product runs as 128 tiles.
    def __call__(self, x: Tensor, chunk: int = 0) -> Tensor:
        n, hh, ww, c = x.shape
        ntok = hh * ww
        hn = ops.groupnorm(x, self.norm[0], self.norm[1], self.eps, False, self.groups).view(n, ntok, c)
        xr = x.view(n, ntok, c)
        out = torch.empty_like(xr)
        scale = 1.0 / math.sqrt(c)
        f32 = self.scores_f32
        for i in range(n):
            q = ops.gemm(hn[i], self.q[0], col_bias=self.q[1])
            k = ops.gemm(hn[i], self.k[0], col_bias=self.k[1])
            vt = ops.gemm(self.v[0], hn[i], m_bias=self.v[1])                 # V^T [c, ntok]
            if ops.PROFILE is None and ntok % 8 == 0:
                o = ops.attention_vae(q, k, vt, scale, f32_scores=f32, chunk_rows=chunk)       # one C-ABI call: fie_attn_vae_d512_f16
            else:
                o = self._attention_unfused(q, k, vt, ntok, c, scale, chunk or ntok, f32)      # same passes, one profiled call each
            ops.gemm(o, self.o[0], col_bias=self.o[1], residual=xr[i], out=out[i])
        return out.view(n, hh, ww, c)       # (per-image GEMMs: the statistics of this output are left to the GroupNorm kernel)

    @staticmethod
    def _attention_unfused(q, k, vt, ntok, c, scale, chunk, f32):
        o = torch.empty((ntok, c), dtype=q.dtype, device=q.device)
        for r0 in range(0, ntok, chunk):
            r1 = min(r0 + chunk, ntok)
            if q.dtype == torch.bfloat16:                                  # bf16 VAE: fp32 logits, bf16 P for the P V GEMM
                s = ops.gemm(q[r0:r1], k, out_f32=True)
                ops.gemm(ops.softmax_rows(s, scale, out_dtype=torch.bfloat16), vt, out=o[r0:r1])
            elif not f32 and ntok % 4 == 0 and ntok <= 16384:
                s = ops.gemm(q[r0:r1], k, scale=scale)                     # [rows, ntok] fp16, already scaled
                p, inv = ops.softmax_rows_exp(s, 1.0, out=s)               # exp only, in place; 1 / rowsum on the side
                ops.gemm(p, vt, out=o[r0:r1], row_scale=inv)               # ... applied in fp32 by the P V epilogue
            elif not f32:
                s = ops.gemm(q[r0:r1], k, scale=scale)
                ops.gemm(ops.softmax_rows(s, 1.0, out=s), vt, out=o[r0:r1])
            else:
                s = ops.gemm(q[r0:r1], k, out_f32=True)                    # [rows, ntok] fp32
                ops.gemm(ops.softmax_rows(s, scale), vt, out=o[r0:r1])
        return o


class VAE:
    """AutoencoderKL.  ``dtype=torch.bfloat16`` (VAE checkpoints whose activations leave the fp16 range, DESIGN.md 3.11): bf16
    weights and stored activations, fp32 accumulation and fp32 attention logits, no producer-side GroupNorm statistics.  The interface
    does not depend on it: ``encode_moments`` returns fp16 moments and ``decode`` an fp16 image either way."""

    def __init__(self, params: Params, cfg: VAEConfig, device, attention_scores_f32: bool = False, dtype=torch.float16):
        if dtype not in (torch.float16, torch.bfloat16):
            raise ValueError(f"VAE dtype must be torch.float16 or torch.bfloat16, not {dtype}")
        pk = _Packer(params, device, dtype=dtype)
        self.cfg, self.dev, self.dtype = cfg, device, dtype
        g, eps = cfg.norm_groups, cfg.norm_eps
        ch = list(cfg.block_out_channels)
        L = cfg.latent_channels
        # ---- encoder ----
        self.e_in = pk.c8("encoder.conv_in")
        self.e_down = []
        for i in range(len(ch)):
            res = [Resnet(pk, f"encoder.down_blocks.{i}.resnets.{j}", eps, g) for j in range(cfg.layers_per_block)]
            ds = pk.conv3(f"encoder.down_blocks.{i}.downsamplers.0.conv") if i < len(ch) - 1 else None
            self.e_down.append((res, ds))
        self.e_mid = (Resnet(pk, "encoder.mid_block.resnets.0", eps, g), _VAEAttention(pk, "encoder.mid_block.attentions.0", g, eps),
                      Resnet(pk, "encoder.mid_block.resnets.1", eps, g))
        self.e_norm = pk.norm("encoder.conv_norm_out")
        self.e_out = pk.conv3("encoder.conv_out", pad_cout_to=32)
        self.quant = pk.conv1("quant_conv")
        # ---- decoder ----
        pq_w, pq_b = pk.w("post_quant_conv"), pk.b("post_quant_conv")
        w = torch.zeros((L, 3, 3, 4), dtype=torch.float32, device=device)
        w[:, 1, 1, :L] = pq_w.reshape(L, L) / cfg.scaling_factor          # 1x1 conv as centre tap; latents/scaling folded in
        self.pq = (w.contiguous(), pq_b)
        self.d_in = pk.c8("decoder.conv_in")
        self.d_mid = (Resnet(pk, "decoder.mid_block.resnets.0", eps, g), _VAEAttention(pk, "decoder.mid_block.attentions.0", g, eps),
                      Resnet(pk, "decoder.mid_block.resnets.1", eps, g))
        self.d_up = []
        for i in range(len(ch)):
            res = [Resnet(pk, f"decoder.up_blocks.{i}.resnets.{j}", eps, g) for j in range(cfg.layers_per_block + 1)]
            us = pk.conv_up(f"decoder.up_blocks.{i}.upsamplers.0.conv") if i < len(ch) - 1 else None
            self.d_up.append((res, us))
        self.d_norm = pk.norm("decoder.conv_norm_out")
        self.d_out = pk.conv3("decoder.conv_out", pad_cout_to=32)
        # every block output of the VAE is consumed by a GroupNorm: let the producing epilogue accumulate its statistics (fp16 only:
        # the bf16 GroupNorm computes range-safe statistics itself)
        bf = dtype == torch.bfloat16
        for res, _ in self.e_down + self.d_up:
            for r in res:
                r.out_gn = 0 if bf else g
        for blk in (self.e_mid, self.d_mid):
            blk[0].out_gn = blk[2].out_gn = 0 if bf else g
        self.gn_groups = 0 if bf else g
        self.e_mid[1].scores_f32 = self.d_mid[1].scores_f32 = bool(attention_scores_f32)

    def encode_moments(self, xp8: Tensor) -> Tensor:
        """xp8: zero-padded [N,H+2,W+8,8] fp16 image in [-1,1] (ops.preprocess_pad8) -> moments [N,H/8,W/8,2L] fp16."""
        cfg = self.cfg
        h = ops.conv3x3_c8(xp8, self.e_in[0], col_bias=self.e_in[1], gn_groups=self.gn_groups, out_dtype=self.dtype)
        for res, ds in self.e_down:
            for r in res:
                h = r(h)
            if ds is not None:
                h = ops.conv3x3(h, ds[0], stride=2, pad_mode=1, col_bias=ds[1], gn_groups=self.gn_groups)
        h = self.e_mid[0](h)
        h = self.e_mid[1](h)
        h = self.e_mid[2](h)
        h = ops.groupnorm(h, self.e_norm[0], self.e_norm[1], cfg.norm_eps, True, cfg.norm_groups)
        h = ops.conv3x3(h, self.e_out[0], cout_valid=2 * cfg.latent_channels, col_bias=self.e_out[1])
        n, hh, ww, c = h.shape
        return ops.gemm(h.view(n * hh * ww, c), self.quant[0], col_bias=self.quant[1], out_dtype=torch.float16).view(n, hh, ww, c)

    def decode(self, z: Tensor) -> Tensor:
        """z [N,h,w,4] fp16 latents (scaled) -> image [N,8h,8w,4] fp16 (3 valid channels) in ~[-1,1]."""
        cfg = self.cfg
        L = cfg.latent_channels
        h = ops.conv3x3_cin4(z, self.pq[0], self.pq[1], L, ld_out=4)
        h = ops.conv3x3_c8(ops.pad8(h), self.d_in[0], col_bias=self.d_in[1], gn_groups=self.gn_groups, out_dtype=self.dtype)
        h = self.d_mid[0](h)
        h = self.d_mid[1](h)
        h = self.d_mid[2](h)
        for res, us in self.d_up:
            for r in res:
                h = r(h)
            if us is not None:
                h = ops.conv_up2x(h, us[0], col_bias=us[1], gn_groups=self.gn_groups)
        h = ops.groupnorm(h, self.d_norm[0], self.d_norm[1], cfg.norm_eps, True, cfg.norm_groups)
        n, hh, ww, _ = h.shape
        out = torch.empty((n, hh, ww, 4), dtype=torch.float16, device=h.device)
        ops.conv3x3(h, self.d_out[0], cout_valid=3, out=out, col_bias=self.d_out[1])
        return out
