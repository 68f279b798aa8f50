"""The guided img2img edit path on the B200 kernels: the work ``StableDiffusionXLControlNetImg2ImgPipeline.__call__``
does for the reference at ``src/pipeline.py:261-272`` (order per SURVEY Appendix A.1), batched over images."""
from __future__ import annotations

import math
import numbers
import os
from collections import OrderedDict
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import ops
from .configs import ControlNetConfig, UNetConfig, VAEConfig
from .engine import VAE, ControlNet, UNet
from .scheduler import LCMSchedule

Tensor = torch.Tensor


@dataclass
class EditOutput:
    """Results of one engine call.  With ``use_graph`` the tensors ALIAS the CUDA graph's static output buffers: they are valid
    until the next ``edit_batch`` call with the same graph key (shapes, executed step count, CFG on/off, blur; see ``graph_key``),
    whatever its guidance, scales, thresholds or strengths, which overwrites them in stream order — copy them (``.cpu()``,
    ``.clone()``, an asynchronous D2H copy enqueued before the next call) if they must outlive it."""
    images: Tensor                      # uint8 [B,H,W,3] on the device
    edges: Tensor                       # uint8 [B,H,W,3] Canny control image
    latents: Optional[Tensor] = None    # fp32 [B,h,w,4] final latents (the scheduler state; the VAE decodes its fp16 copy)
    extras: Optional[Dict] = None


def per_image(name: str, value, n: int) -> list:
    """A scalar (broadcast) or a length-``n`` sequence of finite numbers -> list of ``n`` values; ValueError otherwise."""
    if isinstance(value, (str, bytes)):
        raise ValueError(f"{name} must be a number or a sequence of {n} numbers, not {value!r}")
    if isinstance(value, (Sequence, np.ndarray, Tensor)):
        vals = [v.item() if hasattr(v, "item") else v for v in value]
        if len(vals) != n:
            raise ValueError(f"{name}: {len(vals)} values for {n} images")
    else:
        vals = [value] * n
    for i, v in enumerate(vals):
        if isinstance(v, bool) or not isinstance(v, numbers.Real) or not math.isfinite(v):
            raise ValueError(f"{name} of image {i} must be a finite number, not {v!r}")
    return vals


def executed_steps(strength, num_inference_steps) -> int:
    """diffusers img2img ``check_inputs`` + ``get_timesteps``: the number of denoising steps an image executes (ValueError if none)."""
    if strength < 0 or strength > 1:
        raise ValueError(f"The value of strength should in [0.0, 1.0] but is {strength}")
    if not isinstance(num_inference_steps, int) or num_inference_steps <= 0:
        raise ValueError(f"`num_inference_steps` has to be a positive integer but is {num_inference_steps}")
    n_exec = min(int(num_inference_steps * strength), num_inference_steps)
    if n_exec < 1:                   # diffusers: get_timesteps leaves no step to run
        raise ValueError(f"After adjusting the num_inference_steps by strength parameter: {strength}, the number of pipeline steps is "
                         f"{n_exec} which is < 1 and not appropriate for this pipeline.")
    return n_exec


def per_image_settings(n: int, strength, num_inference_steps, guidance_scale, controlnet_conditioning_scale, canny_low_threshold,
                       canny_high_threshold) -> Dict[str, list]:
    """The numeric settings of an edit, each a scalar (every image) or a sequence with one value per image -> {name: list of ``n``
    values} plus "n_exec", the denoising steps each image executes.  ValueError (naming the image) for a wrong length, a non-finite
    value or an invalid strength / step count."""
    st = dict(strength=strength, num_inference_steps=num_inference_steps, guidance_scale=guidance_scale,
              controlnet_conditioning_scale=controlnet_conditioning_scale, canny_low_threshold=canny_low_threshold,
              canny_high_threshold=canny_high_threshold)
    st = {name: per_image(name, v, n) for name, v in st.items()}
    st["n_exec"] = []
    for i in range(n):
        try:
            st["n_exec"].append(executed_steps(st["strength"][i], st["num_inference_steps"][i]))
        except ValueError as err:
            raise ValueError(f"image {i}: {err}") from None
    return st


@dataclass
class EditParams:
    """The numeric settings of one engine call, per image, packed on the host into the parameter block the kernels read on the
    device (a static input of the CUDA graph, like the images).  Layout of ``block`` (fp32 words, B images, R = 2B rows with CFG, else
    B, n = n_exec):  [0, 2B) Canny (low, high) int32 pairs | [2B, 4B) add-noise (sqrt_a, sqrt_1ma) | [4B, 4B+R) ControlNet scale per
    UNet row (row r: image r mod B) | n x R timesteps per row | n x B x 7 step table (LCMSchedule.STEP_COLUMNS)."""
    n_images: int
    n_exec: int
    cfg: bool
    block: np.ndarray

    @staticmethod
    def pack(sched: LCMSchedule, n_images: int, strength=0.5, num_inference_steps=4, guidance_scale=1.5, controlnet_conditioning_scale=0.5,
             canny_low=100, canny_high=200) -> "EditParams":
        """Each setting a scalar (the whole batch) or a sequence with one value per image.  All images must execute the same number of
        steps and agree on CFG (guidance > 1 for all, or for none: diffusers runs the positive rows only at guidance <= 1)."""
        B = n_images
        st = per_image_settings(B, strength, num_inference_steps, guidance_scale, controlnet_conditioning_scale, canny_low, canny_high)
        n_exec = st["n_exec"][0]
        for i, e in enumerate(st["n_exec"]):
            if e != n_exec:
                raise ValueError(f"image {i} executes {e} denoising steps, image 0 executes {n_exec}: the images of one batch must execute "
                                 "the same number of steps")
        guidance = st["guidance_scale"]
        cfg = guidance[0] > 1
        if any((g > 1) != cfg for g in guidance):
            raise ValueError("guidance_scale: the images of one batch must all be > 1 (classifier-free guidance) or all <= 1")
        ts, add, table = sched.batch_tables(st["num_inference_steps"], st["strength"], [g if cfg else 1.0 for g in guidance])
        nrow = 2 if cfg else 1
        thr = np.array([ops.canny_thresholds(lo, hi) for lo, hi in zip(st["canny_low_threshold"], st["canny_high_threshold"])],
                       dtype=np.int32).reshape(B, 2)
        tsr = np.array(ts, dtype=np.float32).T                               # [n_exec, B]
        scale = st["controlnet_conditioning_scale"]
        block = np.concatenate([thr.view(np.float32).ravel(), add.ravel(), np.tile(np.asarray(scale, np.float32), nrow),
                                np.tile(tsr, (1, nrow)).ravel(), table.ravel()])
        return EditParams(B, n_exec, cfg, np.ascontiguousarray(block, dtype=np.float32))

    def views(self, dev_block: Tensor) -> Dict[str, Tensor]:
        """Device block -> named views: thr int32 [B,2], add [B,2], scale [R], t [n,R], step [n,B,7]."""
        B, n, R = self.n_images, self.n_exec, (2 if self.cfg else 1) * self.n_images
        o = [0, 2 * B, 4 * B, 4 * B + R, 4 * B + R + n * R, 4 * B + R + n * R + 7 * n * B]
        return dict(thr=dev_block[o[0]:o[1]].view(torch.int32).view(B, 2), add=dev_block[o[1]:o[2]].view(B, 2), scale=dev_block[o[2]:o[3]],
                    t=dev_block[o[3]:o[4]].view(n, R), step=dev_block[o[4]:o[5]].view(n, B, 7))


def graph_key(images_shape, pe_shape, pl_shape, n_noises: int, params: EditParams, canny_blur: bool) -> tuple:
    """The CUDA-graph cache key of an edit: what changes its launch sequence (shapes, executed step count, CFG on/off, Canny blur).
    Guidance, ControlNet scale, thresholds and strengths are device data (``EditParams``) and stay out of it."""
    return (tuple(images_shape), tuple(pe_shape), tuple(pl_shape), int(n_noises), params.n_exec, params.cfg, bool(canny_blur))


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
        # captured graphs, least recently used first.  Every distinct graph_key (shapes, executed steps, CFG, blur) owns a private
        # multi-GB memory pool, so the cache is a small LRU (FIE_GRAPH_CACHE, default 4) and clear_memory() trims it.
        self._graphs: "OrderedDict" = OrderedDict()
        self.max_graphs = max(int(os.environ.get("FIE_GRAPH_CACHE", "4")), 1)
        self._staging: Dict[int, List] = {}   # parameter-block size -> ring of [pinned host block, event after its H2D copy]
        self._staging_next = 0

    def release_graphs(self, keep: int = 0):
        """Drop captured CUDA graphs (and their private memory pools), keeping the ``keep`` most recently used."""
        while len(self._graphs) > max(keep, 0):
            _, g = self._graphs.popitem(last=False)
            g.clear()

    @torch.no_grad()
    def edit_batch(self, images_u8: Tensor, prompt_embeds: Tensor, pooled: Tensor, noises: Sequence[Tensor], strength=0.5,
                   num_inference_steps=4, guidance_scale=1.5, controlnet_conditioning_scale=0.5,
                   canny_low=100, canny_high=200, return_latents: bool = False, return_extras: bool = False,
                   use_graph: Optional[bool] = None, canny_blur: bool = False) -> EditOutput:
        """images_u8: uint8 [B,H,W,3] (CUDA, H and W multiples of 8; 1024 for the reference path).
        prompt_embeds [2,77,D] / pooled [2,P] (row 0 negative, row 1 positive; shared by the batch) or per image
        [B,2,77,D] / [B,2,P].  noises: [xi, n, z1, ...] each [B,4,h,w] (reference RNG order).

        ``strength``, ``num_inference_steps``, ``guidance_scale``, ``controlnet_conditioning_scale``, ``canny_low`` and ``canny_high``
        each take a scalar (the whole batch) or a sequence with one value per image (see ``EditParams.pack``: every image must execute
        the same number of steps, and guidance must be > 1 for all images or for none).  They reach the kernels as device data.

        ``use_graph`` (default: ``self.use_graphs``): replay the whole edit — ~2500 kernel launches — as ONE CUDA graph
        captured on first use for its ``graph_key``; inputs and settings are copied into the graph's static buffers and the
        returned tensors are the graph's static outputs (valid until the next call with the same key)."""
        with torch.cuda.device(self.dev):           # kernels launch on the CURRENT device's stream: make that this engine's device
            params = EditParams.pack(self.sched, images_u8.shape[0], strength, num_inference_steps, guidance_scale, controlnet_conditioning_scale,
                                     canny_low, canny_high)
            return self._edit_batch(images_u8, prompt_embeds, pooled, noises, params, return_latents, return_extras, use_graph, canny_blur)

    def _upload_params(self, params: EditParams, out: Optional[Tensor] = None) -> Tensor:
        """Host parameter block -> device (into ``out``, a graph's static buffer, or a new tensor) by an asynchronous copy from a pinned
        buffer.  The buffers form a ring of two per block size; a buffer is rewritten only after its previous copy has run."""
        ring = self._staging.get(params.block.size)
        if ring is None:
            ring = self._staging[params.block.size] = [[torch.empty(params.block.size, dtype=torch.float32).pin_memory(), None] for _ in range(2)]
        slot = ring[self._staging_next % 2]
        self._staging_next += 1
        if slot[1] is not None:
            slot[1].synchronize()
        slot[0].numpy()[:] = params.block
        if out is None:
            out = torch.empty(params.block.size, dtype=torch.float32, device=self.dev)
        out.copy_(slot[0], non_blocking=True)
        slot[1] = torch.cuda.Event()
        slot[1].record(torch.cuda.current_stream(self.dev))
        return out

    def _edit_batch(self, images_u8, prompt_embeds, pooled, noises, params: EditParams, return_latents, return_extras, use_graph,
                    canny_blur) -> EditOutput:
        dev = self.dev
        nz = [n.to(dev, torch.float16).permute(0, 2, 3, 1).contiguous() for n in noises]
        pe = prompt_embeds.to(dev, torch.float16)
        pl = pooled.to(dev, torch.float16)
        images_u8 = images_u8.to(dev)
        graph = self.use_graphs if use_graph is None else use_graph
        if not graph or return_extras or ops.PROFILE is not None:
            return self._edit_core(images_u8, pe, pl, nz, self._upload_params(params), params, canny_blur=bool(canny_blur),
                                   return_latents=return_latents, return_extras=return_extras)
        key = graph_key(images_u8.shape, pe.shape, pl.shape, len(nz), params, canny_blur)
        g = self._graphs.get(key)
        if g is None:
            self.release_graphs(keep=self.max_graphs - 1)
            g = self._capture(key, images_u8, pe, pl, nz, params, bool(canny_blur))
        else:
            self._graphs.move_to_end(key)
        g["img"].copy_(images_u8); g["pe"].copy_(pe); g["pl"].copy_(pl)
        for d, s_ in zip(g["nz"], nz):
            d.copy_(s_)
        self._upload_params(params, out=g["prm"])
        g["graph"].replay()
        ops.LAUNCHES += g["launches"]
        out = g["out"]
        return EditOutput(images=out.images, edges=out.edges, latents=out.latents if return_latents else None)

    def _capture(self, key, images_u8, pe, pl, nz, params: EditParams, canny_blur: bool):
        """Warm up eagerly (first-use attribute setup, allocator pools), then record one edit into a CUDA graph."""
        st = dict(img=images_u8.clone(), pe=pe.clone(), pl=pl.clone(), nz=[n.clone() for n in nz], prm=self._upload_params(params))
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            self._edit_core(st["img"], st["pe"], st["pl"], st["nz"], st["prm"], params, canny_blur=canny_blur, return_latents=True)
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        graph = torch.cuda.CUDAGraph()
        l0 = ops.LAUNCHES
        # an explicit capture stream on THIS engine's device: torch.cuda.graph's default capture stream is a process-wide singleton that
        # lives on the device of the first capture, which would silently move a cuda:1 engine's capture (and its launches) to cuda:0
        if getattr(self, "_capture_stream", None) is None:
            self._capture_stream = torch.cuda.Stream(device=self.dev)
        with torch.cuda.graph(graph, stream=self._capture_stream):
            out = self._edit_core(st["img"], st["pe"], st["pl"], st["nz"], st["prm"], params, canny_blur=canny_blur, return_latents=True)
        st.update(graph=graph, out=out, launches=ops.LAUNCHES - l0)
        ops.LAUNCHES = l0                         # capture records launches, it does not execute them
        self._graphs[key] = st
        return st

    def _edit_core(self, images_u8: Tensor, pe: Tensor, pl: Tensor, nz: List[Tensor], prm: Tensor, params: EditParams, canny_blur: bool = False,
                   return_latents: bool = False, return_extras: bool = False) -> EditOutput:
        """The edit itself; every tensor is already on the device (fp16, noises NHWC; ``prm`` the parameter block of ``params``, whose
        values are read by the kernels only) — nothing here touches the host."""
        B, H, W, _ = images_u8.shape
        v = params.views(prm)
        do_cfg = params.cfg
        nrow = 2 if do_cfg else 1
        # ---- Canny control image + conditioning embedding (step-invariant) ----
        ops.stage("canny+cond_embedding")
        edges3 = ops.canny(images_u8, out_channels=3, gaussian_blur=canny_blur, thresholds=v["thr"])     # blur: opt-in, the reference has none
        cond_emb = self.cn.cond_embedding(ops.preprocess_pad8(edges3, normalize=False))
        if do_cfg:
            cond_emb = torch.cat([cond_emb, cond_emb], 0)
        # ---- VAE encode -> posterior sample -> scale -> add_noise ----
        ops.stage("vae_encode")
        moments = self.vae.encode_moments(ops.preprocess_pad8(images_u8, normalize=True))
        x32, x = ops.vae_sample_add_noise(moments, nz[0], nz[1], self.vae.cfg.scaling_factor, v["add"])    # fp32 state, fp16 copy
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
        for k in range(params.n_exec):
            ops.stage("controlnet_step")
            x2 = torch.cat([x] * nrow, 0) if do_cfg else x
            feats = self.cn.encode(x2, v["t"][k], ps_cn, cond_emb, nctx)
            ops.stage("unet_step")
            eps = self.unet.forward(x2, v["t"][k], ps_un, nctx=nctx, merge=self.cn.merge_into(feats, v["scale"]))
            last = k == params.n_exec - 1
            z = None
            if not last:
                z = nz[zi]
                zi += 1
            eu, ec = (eps[:B], eps[B:]) if do_cfg else (eps, eps)
            if return_extras:
                eps_list.append(eps)
            x32, x = ops.cfg_lcm_step(eu, ec, x32, z, v["step"][k], last)
        # ---- VAE decode (latents / scaling folded into post_quant_conv) + postprocess ----
        ops.stage("vae_decode")
        decoded = self.vae.decode(x)
        images = ops.postprocess(decoded)
        ops.stage("end")
        extras = dict(moments=moments, eps=eps_list, decoded=decoded) if return_extras else None
        return EditOutput(images=images, edges=edges3, latents=x32 if (return_latents or return_extras) else None, extras=extras)
