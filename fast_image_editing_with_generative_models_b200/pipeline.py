"""The guided img2img edit path on the B200 kernels: the work ``StableDiffusionXLControlNetImg2ImgPipeline.__call__``
does for the reference at ``src/pipeline.py:261-272`` (order per SURVEY Appendix A.1), batched over images."""
from __future__ import annotations

import os
from collections import OrderedDict
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import torch

from . import ops
from .configs import ControlNetConfig, UNetConfig, VAEConfig
from .engine import VAE, ControlNet, UNet
from .scheduler import LCMSchedule

Tensor = torch.Tensor


@dataclass
class EditOutput:
    """Results of one engine call.  With ``use_graph`` the tensors ALIAS the CUDA graph's static output buffers: they are valid
    until the next ``edit_batch`` call with the same (shapes, arguments) key, which overwrites them in stream order — copy them
    (``.cpu()``, ``.clone()``, an asynchronous D2H copy enqueued before the next call) if they must outlive it."""
    images: Tensor                      # uint8 [B,H,W,3] on the device
    edges: Tensor                       # uint8 [B,H,W,3] Canny control image
    latents: Optional[Tensor] = None    # fp32 [B,h,w,4] final latents (the scheduler state; the VAE decodes its fp16 copy)
    extras: Optional[Dict] = None


def sdxl_time_ids(height: int, width: int) -> List[float]:
    """SDXL micro-conditioning of an uncropped image edited at its own size: original size, crop corner (0, 0), target size, each as
    (height, width), as diffusers' ``_get_add_time_ids``."""
    return [float(height), float(width), 0.0, 0.0, float(height), float(width)]


def _move_to(obj, dev, seen=None):
    """Recursively moves every tensor reachable from ``obj`` (attributes, lists, tuples, dicts) to ``dev``; returns the moved object."""
    seen = set() if seen is None else seen
    if isinstance(obj, Tensor):
        return obj.to(dev)
    if isinstance(obj, torch.device):
        return dev
    if isinstance(obj, (list, tuple)):
        out = [_move_to(v, dev, seen) for v in obj]
        if isinstance(obj, list):
            obj[:] = out
            return obj
        return tuple(out)
    if isinstance(obj, dict):
        for k in list(obj):
            obj[k] = _move_to(obj[k], dev, seen)
        return obj
    if hasattr(obj, "__dict__") and not isinstance(obj, type) and type(obj).__module__.startswith(__name__.rsplit(".", 1)[0]) and id(obj) not in seen:
        seen.add(id(obj))
        for k, v in list(vars(obj).items()):
            setattr(obj, k, _move_to(v, dev, seen))
    return obj


class EditEngine:
    """Owns the packed weights of one (UNet, ControlNet, VAE) triple on one GPU and runs batched edits."""

    def __init__(self, unet_params, unet_cfg: UNetConfig, cn_params, cn_cfg: ControlNetConfig, vae_params, vae_cfg: VAEConfig,
                 device="cuda", lora=None, lora_scale: float = 1.0, pack_on_host: bool = False, vae_scores_f32: bool = False,
                 vae_dtype=torch.float16):
        """Load-time weight packing (layout transforms, LoRA fuse, LayerNorm fold; cold path, reference ``src/pipeline.py:45-181``)
        uses plain torch tensor ops: by default on the GPU (ATen / cuBLAS kernels, seconds for SDXL), with ``pack_on_host`` on the
        CPU followed by plain H2D copies — then no library kernel is ever launched on the device, only ours (``smoke()``).
        ``vae_dtype=torch.bfloat16`` runs the VAE with bf16 weights and activations (engine.VAE); its interface stays fp16."""
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise RuntimeError("EditEngine runs on CUDA (sm_100a) only; there is no CPU path")
        with torch.cuda.device(self.dev):
            pdev = torch.device("cpu") if pack_on_host else self.dev
            self.unet = UNet(unet_params, unet_cfg, pdev, lora, lora_scale)
            self.cn = ControlNet(cn_params, cn_cfg, pdev)
            self.vae = VAE(vae_params, vae_cfg, pdev, attention_scores_f32=vae_scores_f32, dtype=vae_dtype)   # fp32 VAE attention logits: real checkpoints
            if pack_on_host:
                for m in (self.unet, self.cn, self.vae):
                    _move_to(m, self.dev)
        self.sched = LCMSchedule()
        self.use_graphs = False           # opt-in: replay each edit as one CUDA graph (see edit_batch)
        # captured graphs, least recently used first.  Every distinct (shapes, strength, guidance, thresholds, ...) key owns a
        # private multi-GB memory pool, so the cache is a small LRU (FIE_GRAPH_CACHE, default 4) and clear_memory() trims it.
        self._graphs: "OrderedDict" = OrderedDict()
        self.max_graphs = max(int(os.environ.get("FIE_GRAPH_CACHE", "4")), 1)

    def release_graphs(self, keep: int = 0):
        """Drop captured CUDA graphs (and their private memory pools), keeping the ``keep`` most recently used."""
        while len(self._graphs) > max(keep, 0):
            _, g = self._graphs.popitem(last=False)
            g.clear()

    @torch.no_grad()
    def edit_batch(self, images_u8: Tensor, prompt_embeds: Tensor, pooled: Tensor, noises: Sequence[Tensor], strength: float = 0.5,
                   num_inference_steps: int = 4, guidance_scale: float = 1.5, controlnet_conditioning_scale: float = 0.5,
                   canny_low: int = 100, canny_high: int = 200, return_latents: bool = False, return_extras: bool = False,
                   use_graph: Optional[bool] = None, canny_blur: bool = False) -> EditOutput:
        """images_u8: uint8 [B,H,W,3] (CUDA, H and W multiples of 8; 1024 for the reference path).
        prompt_embeds [2,77,D] / pooled [2,P] (row 0 negative, row 1 positive; shared by the batch) or per image
        [B,2,77,D] / [B,2,P].  noises: [xi, n, z1, ...] each [B,4,h,w] (reference RNG order).

        ``use_graph`` (default: ``self.use_graphs``): replay the whole edit — ~2500 kernel launches — as ONE CUDA graph
        captured on first use for this (shapes, schedule) key; inputs are copied into the graph's static buffers and the
        returned tensors are the graph's static outputs (valid until the next call with the same key)."""
        with torch.cuda.device(self.dev):           # kernels launch on the CURRENT device's stream: make that this engine's device
            return self._edit_batch(images_u8, prompt_embeds, pooled, noises, strength, num_inference_steps, guidance_scale,
                                    controlnet_conditioning_scale, canny_low, canny_high, return_latents, return_extras, use_graph, canny_blur)

    def _edit_batch(self, images_u8, prompt_embeds, pooled, noises, strength, num_inference_steps, guidance_scale, controlnet_conditioning_scale,
                    canny_low, canny_high, return_latents, return_extras, use_graph, canny_blur) -> EditOutput:
        dev = self.dev
        if strength < 0 or strength > 1:
            raise ValueError(f"The value of strength should in [0.0, 1.0] but is {strength}")
        if min(int(num_inference_steps * strength), num_inference_steps) < 1:       # diffusers: get_timesteps leaves no step to run
            raise ValueError(f"After adjusting the num_inference_steps by strength parameter: {strength}, the number of pipeline steps is 0 "
                             "which is < 1 and not appropriate for this pipeline.")
        nz = [n.to(dev, torch.float16).permute(0, 2, 3, 1).contiguous() for n in noises]
        pe = prompt_embeds.to(dev, torch.float16)
        pl = pooled.to(dev, torch.float16)
        images_u8 = images_u8.to(dev)
        args = dict(strength=strength, num_inference_steps=num_inference_steps, guidance_scale=guidance_scale,
                    controlnet_conditioning_scale=controlnet_conditioning_scale, canny_low=canny_low, canny_high=canny_high, canny_blur=bool(canny_blur))
        graph = self.use_graphs if use_graph is None else use_graph
        if not graph or return_extras or ops.PROFILE is not None:
            return self._edit_core(images_u8, pe, pl, nz, return_latents=return_latents, return_extras=return_extras, **args)
        key = (tuple(images_u8.shape), tuple(pe.shape), tuple(pl.shape), len(nz), tuple(sorted(args.items())))
        g = self._graphs.get(key)
        if g is None:
            self.release_graphs(keep=self.max_graphs - 1)
            g = self._capture(key, images_u8, pe, pl, nz, args)
        else:
            self._graphs.move_to_end(key)
        g["img"].copy_(images_u8); g["pe"].copy_(pe); g["pl"].copy_(pl)
        for d, s_ in zip(g["nz"], nz):
            d.copy_(s_)
        g["graph"].replay()
        ops.LAUNCHES += g["launches"]
        out = g["out"]
        return EditOutput(images=out.images, edges=out.edges, latents=out.latents if return_latents else None)

    def _capture(self, key, images_u8, pe, pl, nz, args):
        """Warm up eagerly (first-use attribute setup, allocator pools), then record one edit into a CUDA graph."""
        st = dict(img=images_u8.clone(), pe=pe.clone(), pl=pl.clone(), nz=[n.clone() for n in nz])
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            self._edit_core(st["img"], st["pe"], st["pl"], st["nz"], return_latents=True, **args)
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        graph = torch.cuda.CUDAGraph()
        l0 = ops.LAUNCHES
        # an explicit capture stream on THIS engine's device: torch.cuda.graph's default capture stream is a process-wide singleton that
        # lives on the device of the first capture, which would silently move a cuda:1 engine's capture (and its launches) to cuda:0
        if getattr(self, "_capture_stream", None) is None:
            self._capture_stream = torch.cuda.Stream(device=self.dev)
        with torch.cuda.graph(graph, stream=self._capture_stream):
            out = self._edit_core(st["img"], st["pe"], st["pl"], st["nz"], return_latents=True, **args)
        st.update(graph=graph, out=out, launches=ops.LAUNCHES - l0)
        ops.LAUNCHES = l0                         # capture records launches, it does not execute them
        self._graphs[key] = st
        return st

    def _edit_core(self, images_u8: Tensor, pe: Tensor, pl: Tensor, nz: List[Tensor], strength: float = 0.5,
                   num_inference_steps: int = 4, guidance_scale: float = 1.5, controlnet_conditioning_scale: float = 0.5,
                   canny_low: int = 100, canny_high: int = 200, canny_blur: bool = False, return_latents: bool = False,
                   return_extras: bool = False) -> EditOutput:
        """The edit itself; every tensor is already on the device (fp16, noises NHWC) — nothing here touches the host."""
        B, H, W, _ = images_u8.shape
        sched = self.sched
        timesteps, begin = sched.img2img_timesteps(num_inference_steps, strength)
        do_cfg = guidance_scale > 1
        nrow = 2 if do_cfg else 1
        # ---- Canny control image + conditioning embedding (step-invariant) ----
        ops.stage("canny+cond_embedding")
        edges3 = ops.canny(images_u8, canny_low, canny_high, out_channels=3, gaussian_blur=canny_blur)     # blur: opt-in, the reference has none
        cond_emb = self.cn.cond_embedding(ops.preprocess_pad8(edges3, normalize=False))
        if do_cfg:
            cond_emb = torch.cat([cond_emb, cond_emb], 0)
        # ---- VAE encode -> posterior sample -> scale -> add_noise ----
        ops.stage("vae_encode")
        moments = self.vae.encode_moments(ops.preprocess_pad8(images_u8, normalize=True))
        sa, s1 = sched.add_noise_coeffs(timesteps[0])
        x32, x = ops.vae_sample_add_noise(moments, nz[0], nz[1], self.vae.cfg.scaling_factor, sa, s1)    # fp32 state, fp16 copy
        # ---- prompt conditioning (step-invariant): rows [neg]*B + [pos]*B as diffusers ----
        ops.stage("prompt_kv")
        if pe.dim() == 3:
            pe, pl = pe[None].expand(B, -1, -1, -1), pl[None].expand(B, -1, -1)
        rows = [0, 1] if do_cfg else [1]
        ctx = torch.cat([pe[:, r] for r in rows], 0).contiguous()
        te = torch.cat([pl[:, r] for r in rows], 0).contiguous()
        time_ids = sdxl_time_ids(H, W)
        nctx = ctx.shape[1]
        ps_cn = self.cn.prepare_prompt(ctx, te, time_ids)
        ps_un = self.unet.prepare_prompt(ctx, te, time_ids)
        # ---- denoising loop ----
        zi = 2
        eps_list = []
        for k, t in enumerate(timesteps):
            ops.stage("controlnet_step")
            x2 = torch.cat([x] * nrow, 0) if do_cfg else x
            feats = self.cn.encode(x2, float(t), ps_cn, cond_emb, nctx)
            ops.stage("unet_step")
            eps = self.unet.forward(x2, float(t), ps_un, nctx=nctx, merge=self.cn.merge_into(feats, controlnet_conditioning_scale))
            c = sched.step_coeffs(begin + k)
            z = None
            if not c["last"]:
                z = nz[zi]
                zi += 1
            eu, ec = (eps[:B], eps[B:]) if do_cfg else (eps, eps)
            if return_extras:
                eps_list.append(eps)
            x32, x = ops.cfg_lcm_step(eu, ec, x32, z, guidance_scale if do_cfg else 1.0, c)
        # ---- VAE decode (latents / scaling folded into post_quant_conv) + postprocess ----
        ops.stage("vae_decode")
        decoded = self.vae.decode(x)
        images = ops.postprocess(decoded)
        ops.stage("end")
        extras = dict(moments=moments, eps=eps_list, decoded=decoded) if return_extras else None
        return EditOutput(images=images, edges=edges3, latents=x32 if (return_latents or return_extras) else None, extras=extras)
