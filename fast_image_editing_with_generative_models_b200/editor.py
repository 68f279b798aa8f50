"""``FastEditor`` — drop-in mirror of the reference class (``src/pipeline.py:17-293``) on the B200 engine.

Same constructor, ``edit`` / ``preprocess_image`` / ``clear_memory`` / ``get_memory_usage`` signatures, attributes
(``model_name, device, dtype, config, controlnet, pipe``) and error behaviour (``ValueError`` for an unknown model and for
an invalid ``strength``, Python exceptions per image, usable after a failed call) as the reference; the arithmetic runs in
the hand-written CUDA kernels behind ``include/fie_b200.h``.  One addition: :meth:`FastEditor.edit_many`, the batched form
of ``edit`` (micro-batches of 8 images per GPU, SURVEY 8(e)) that ``run_batch.py`` uses.  ``edit``, ``edit_many`` and ``warm_up`` take a
keyword-only ``size``: ``None`` (the reference's 1024 x 1024), a ``(width, height)`` or ``"auto"`` (the SDXL aspect-ratio bucket
closest to the input's shape, ``FastEditor.SDXL_BUCKETS``).

Differences, all forced by the environment and stated in DESIGN.md:

* weights: ``checkpoints={...}`` (or the ``FIE_CHECKPOINTS`` / ``FIE_CONTROLNET`` / ``FIE_VAE`` / ``FIE_LCM_LORA`` environment
  variables, or the CLIs' ``--checkpoints`` flags) loads diffusers folders incl. the two CLIP text encoders and tokenizers;
  without them seeded synthetic tensors of the named architectures are generated and a loud warning is printed (there are
  no checkpoints and no network in the build environment);
* compute is fp16 with fp32 accumulation on the GPU.  ``use_full_precision=True`` is accepted and ``.dtype`` reports
  ``torch.float32`` like the reference (callers only use it for naming), but the kernels stay fp16 and a warning says so;
  ``.compute_dtype`` is always ``torch.float16``.  ``enable_cpu_offload`` is a no-op on a 180 GB part.
  The VAE alone may run in bf16 (``vae_dtype``, ``.vae_dtype``): by default whenever its ``config.json`` says ``"force_upcast": true``.
"""
from __future__ import annotations

import os
import warnings
import zlib
from collections import OrderedDict
from typing import Callable, Dict, List, Optional, Sequence, Union

import numpy as np
import torch
from PIL import Image

from . import model_zoo, ops
from . import synthetic as S
from .lora import LoraAdapters
from .pipeline import executed_steps, per_image_settings

_ENV_KEYS = {"root": "FIE_CHECKPOINTS", "controlnet": "FIE_CONTROLNET", "vae": "FIE_VAE", "lora": "FIE_LCM_LORA"}


def checkpoints_from_env() -> Optional[Dict[str, str]]:
    """``FIE_CHECKPOINTS`` = a diffusers SDXL pipeline folder (``unet/ vae/ text_encoder/ text_encoder_2/ tokenizer/ tokenizer_2/``),
    ``FIE_CONTROLNET`` = the ControlNet folder, optional ``FIE_VAE`` (fp16-fix VAE folder) and ``FIE_LCM_LORA`` (safetensors file)."""
    root = os.environ.get(_ENV_KEYS["root"])
    if not root:
        return None
    return expand_checkpoints(root, os.environ.get(_ENV_KEYS["controlnet"]), os.environ.get(_ENV_KEYS["vae"]), os.environ.get(_ENV_KEYS["lora"]))


def expand_checkpoints(root: str, controlnet: Optional[str], vae: Optional[str] = None, lora: Optional[str] = None, unet: Optional[str] = None) -> Dict[str, str]:
    """Pipeline folder + ControlNet folder -> the ``checkpoints`` dict of :class:`FastEditor`.  ``unet`` overrides ``root/unet``
    (SSD-1B: the ``latent-consistency/lcm-ssd-1b`` UNet replaces the base one, reference ``src/pipeline.py:115-124``)."""
    if not controlnet:
        raise ValueError("a ControlNet checkpoint folder is required (FIE_CONTROLNET / --controlnet_dir)")
    ck = {"unet": unet or os.path.join(root, "unet"), "controlnet": controlnet, "vae": vae or os.path.join(root, "vae")}
    if lora:
        ck["lora"] = lora
    for k in ("text_encoder", "text_encoder_2", "tokenizer", "tokenizer_2"):
        if os.path.isdir(os.path.join(root, k)):
            ck[k] = os.path.join(root, k)
    return ck


def resolve_vae_dtype(vae_dtype: Optional[torch.dtype], force_upcast: Optional[bool]) -> torch.dtype:
    """``FastEditor(vae_dtype=...)``: None -> bf16 when the VAE config says ``force_upcast: true`` (activations beyond the fp16 range),
    else fp16; ``torch.float16`` / ``torch.bfloat16`` force the choice."""
    if vae_dtype is None:
        return torch.bfloat16 if force_upcast else torch.float16
    if vae_dtype not in (torch.float16, torch.bfloat16):
        raise ValueError(f"vae_dtype must be None, torch.float16 or torch.bfloat16, not {vae_dtype}")
    return vae_dtype


def vae_fp16_warning(real_weights: bool, vae_dtype: torch.dtype, force_upcast: Optional[bool]) -> Optional[str]:
    """The RuntimeWarning text when a loaded VAE checkpoint runs in fp16 without its config stating ``force_upcast: false`` (diffusers
    treats a missing key as true and upcasts), else None."""
    if not real_weights or vae_dtype != torch.float16 or force_upcast is False:
        return None
    return ("FastEditor: the VAE runs in fp16, but its config.json does not state \"force_upcast\": false; a VAE whose activations exceed "
            "the fp16 range (e.g. stabilityai/sdxl-vae) gives inf/NaN images in fp16.  Use the fp16-fix VAE (madebyollin/sdxl-vae-fp16-fix, "
            "--vae_dir) or FastEditor(vae_dtype=torch.bfloat16) (--vae_dtype bf16).")


MAX_PIXELS = 1024 * 1024        # VAE mid-block attention: at most 16384 latent tokens (fie_softmax_rows_exp_f16)


def resolve_size(size, image_size) -> tuple:
    """``size`` argument -> (width, height) of the edit for an input of PIL size ``image_size`` = (width, height).

    ``None``: 1024 x 1024.  ``(width, height)``: each side a multiple of 64 in [256, 2048] and width * height <= 1024^2.
    ``"auto"``: the entry of :data:`FastEditor.SDXL_BUCKETS` whose aspect ratio is closest to the input's in log space (ties: the
    earlier one)."""
    if size is None:
        return (FastEditor.OUT_SIZE, FastEditor.OUT_SIZE)
    if isinstance(size, str):
        if size != "auto":
            raise ValueError(f"size must be None, (width, height) or 'auto', not {size!r}")
        iw, ih = image_size
        if iw <= 0 or ih <= 0:
            raise ValueError(f"size='auto' needs a non-empty image, got {image_size}")
        r = np.log(iw) - np.log(ih)
        # log w - log h: exactly antisymmetric, so transposed buckets are exactly equidistant from a square input; min keeps the first
        return min(FastEditor.SDXL_BUCKETS, key=lambda b: abs(np.log(b[0]) - np.log(b[1]) - r))
    try:
        w, h = size
    except (TypeError, ValueError):
        raise ValueError(f"size must be None, (width, height) or 'auto', not {size!r}") from None
    if not all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in (w, h)):
        raise ValueError(f"size sides must be integers, got {size!r}")
    w, h = int(w), int(h)
    if w % 64 or h % 64 or not (256 <= w <= 2048 and 256 <= h <= 2048):
        raise ValueError(f"size {w}x{h}: each side must be a multiple of 64 in [256, 2048]")
    if w * h > MAX_PIXELS:
        raise ValueError(f"size {w}x{h}: at most {MAX_PIXELS} pixels (1024 x 1024)")
    return (w, h)


def micro_batches(sizes: Sequence[tuple], n_exec: Sequence[int], guidance: Sequence[float], mb: int) -> List[tuple]:
    """edit_many's plan: the image indices grouped by (size, executed step count, guidance > 1) -- the images of one engine call share
    its launch sequence -- each group cut into micro-batches of at most ``mb`` images in input order -> [((size, n_exec, cfg), [index,
    ...]), ...]."""
    groups: Dict[tuple, List[int]] = {}
    for i, wh in enumerate(sizes):
        groups.setdefault((tuple(wh), int(n_exec[i]), guidance[i] > 1), []).append(i)
    return [(key, idx[b0:b0 + mb]) for key, idx in groups.items() for b0 in range(0, len(idx), mb)]


class _PipeShim:
    """What callers touch on ``editor.pipe``: ``run_batch.py:157-158`` calls ``set_progress_bar_config(disable=True)``, and users of
    diffusers' pipeline add style LoRAs with ``load_lora_weights`` / ``set_adapters`` (as the reference adds its LCM-LoRA,
    ``src/pipeline.py:154``).  The adapters are fused into the packed weights in place (:mod:`.lora`): every edit after a change uses
    them, captured CUDA graphs included.  An adapter is active at weight 1.0 once loaded; with SDXL the load-time LCM-LoRA is adapter
    ``"default_0"``."""

    def __init__(self, engine, adapters: Optional[LoraAdapters] = None):
        self.engine = engine
        self.progress_bar_config: Dict = {}
        self.adapters = adapters or LoraAdapters(engine)

    def set_progress_bar_config(self, **kwargs):
        self.progress_bar_config.update(kwargs)

    def load_lora_weights(self, pretrained_model_name_or_path_or_dict, adapter_name: Optional[str] = None, weight_name: Optional[str] = None):
        """A local ``.safetensors`` file, a folder holding ``pytorch_lora_weights.safetensors`` (or ``weight_name``), or a state dict (kohya
        or peft / diffusers keys) -> adapter ``adapter_name`` (default: the next ``default_<i>``), active at 1.0 next to the active ones."""
        self.adapters.load_lora_weights(pretrained_model_name_or_path_or_dict, adapter_name, weight_name)

    def set_adapters(self, adapter_names, adapter_weights=None):
        """Make exactly these adapters active, with these weights (default 1.0; one number for all, or one per adapter)."""
        self.adapters.set_adapters(adapter_names, adapter_weights)

    def get_active_adapters(self) -> List[str]:
        return self.adapters.get_active_adapters()

    def get_list_adapters(self) -> Dict[str, List[str]]:
        return self.adapters.get_list_adapters()

    def delete_adapters(self, adapter_names):
        self.adapters.delete_adapters(adapter_names)

    def unload_lora_weights(self):
        """Remove every adapter loaded after the editor was built: the weights are again, byte for byte, the ones it was built with."""
        self.adapters.unload_lora_weights()


class FastEditor:
    """Fast image editor: SDXL / SSD-1B + ControlNet (Canny) + LCM, 4-step img2img with structure preservation."""

    MODEL_CONFIGS = {
        "sdxl": {
            "base_model": "stabilityai/stable-diffusion-xl-base-1.0",
            "lcm_lora": "latent-consistency/lcm-lora-sdxl",
            "use_full_lcm": False,
            "description": "Full SDXL (highest quality, ~6GB VRAM)",
        },
        "ssd-1b": {
            "base_model": "segmind/SSD-1B",
            "lcm_model": "latent-consistency/lcm-ssd-1b",
            "use_full_lcm": True,
            "description": "SSD-1B distilled (50% smaller, 60% faster, ~4GB VRAM)",
        },
    }
    MICRO_BATCH = 8            # images per GPU per engine call in edit_many (SURVEY 8(e))
    OUT_SIZE = 1024            # the reference resizes every input to 1024 x 1024 (src/pipeline.py:251); the default of ``size``
    # size="auto": SDXL / SSD-1B training resolutions of about one megapixel, (width, height)
    SDXL_BUCKETS = ((1024, 1024), (1152, 896), (896, 1152), (1216, 832), (832, 1216), (1344, 768), (768, 1344), (1536, 640), (640, 1536))

    def __init__(self, model_name="sdxl", device="cuda", dtype=torch.float16, enable_cpu_offload=True, use_full_precision=False,
                 use_full_controlnet=False, *, state: Optional[Dict] = None, prompt_encoder: Optional[Callable] = None, tiny: bool = False,
                 text_encoders: bool = False, checkpoints: Optional[Dict[str, str]] = None, tokenizers: Optional[Sequence[str]] = None,
                 verbose: bool = True, vae_dtype: Optional[torch.dtype] = None):
        if model_name not in self.MODEL_CONFIGS:
            raise ValueError(f"Unknown model: {model_name}. Choose from {list(self.MODEL_CONFIGS.keys())}")
        self.model_name = model_name
        self.device = device
        self.dtype = torch.float32 if use_full_precision else dtype
        self.compute_dtype = torch.float16
        self.enable_cpu_offload = enable_cpu_offload
        self.use_full_controlnet = use_full_controlnet
        self.config = self.MODEL_CONFIGS[model_name]
        self._say = print if verbose else (lambda *a, **k: None)
        self._say(f"[FastEditor] Initializing with {model_name.upper()} (B200-native engine)")
        self._say(f"[FastEditor] {self.config['description']}")
        self._say(f"[FastEditor] Device: {device}, Dtype: {self.dtype} (kernels compute fp16 with fp32 accumulation)")
        if not str(device).startswith("cuda"):
            raise RuntimeError("FastEditor (B200-native) needs a CUDA device; there is no CPU path")
        if not torch.cuda.is_available():
            raise RuntimeError("FastEditor (B200-native): no CUDA device available")
        self._dev = torch.device(device)
        if self._dev.index is None:
            self._dev = torch.device("cuda", torch.cuda.current_device())
        if use_full_precision:
            warnings.warn("FastEditor(use_full_precision=True): the B200 kernels compute fp16 operands with fp32 accumulation; the "
                          "reference's fp32 'quality mode' (src/pipeline.py:67-71) is NOT executed in fp32 here", RuntimeWarning, stacklevel=2)
        tiny = tiny or os.environ.get("FIE_TINY") == "1"     # small same-topology models: CLI smoke tests
        if state is None and checkpoints is None:
            checkpoints = checkpoints_from_env()
        self.synthetic_weights = state is None and not checkpoints
        if state is None and checkpoints:
            # real weights (SURVEY 8(f)-3): diffusers folders {unet, controlnet, vae} (+ optional LCM-LoRA file), see checkpoints.py
            from . import checkpoints as K
            self._say("[FastEditor] Loading checkpoints...")
            state = K.load_state(checkpoints["unet"], checkpoints["controlnet"], checkpoints["vae"], checkpoints.get("lora"))
        if state is None:
            warnings.warn("FastEditor: NO CHECKPOINTS given (checkpoints= / FIE_CHECKPOINTS): running on seeded SYNTHETIC random-init weights of "
                          f"the {model_name} architecture — outputs are not meaningful edits", RuntimeWarning, stacklevel=2)
            self._say("[FastEditor] WARNING: generating seeded synthetic weights (no checkpoints given) — outputs are NOT meaningful edits")
            state = model_zoo.synthetic_state(model_name, use_full_controlnet, tiny)
        if use_full_precision:
            # the one fp32 lever the engine has: VAE mid-block attention logits kept in fp32 between the passes (engine._VAEAttention)
            state = dict(state, vae_scores_f32=True)
        force_upcast = getattr(state["vae_cfg"], "force_upcast", None)
        self.vae_dtype = resolve_vae_dtype(vae_dtype, force_upcast)
        msg = vae_fp16_warning(bool(checkpoints) and not self.synthetic_weights, self.vae_dtype, force_upcast)
        if msg:
            warnings.warn(msg, RuntimeWarning, stacklevel=2)
        state = dict(state, vae_dtype=self.vae_dtype)
        self._say(f"[FastEditor] VAE dtype: {self.vae_dtype}")
        with torch.cuda.device(self._dev):
            self._engine = model_zoo.build_engine(state, self._dev)
        self._engine.use_graphs = True      # every edit has the same shapes: replay it as one CUDA graph after the first call
        self.controlnet = self._engine.cn
        # the LoRA fused at build time is adapter "default_0" (diffusers' name for an unnamed first adapter): its factors (no copy; B is
        # scaled as it was fused only when they move to the device at the first change) are what re-weighting or deleting it subtracts
        base = {"default_0": (state["lora"], float(state.get("lora_scale", 1.0)))} if state.get("lora") else None
        self.pipe = _PipeShim(self._engine, LoraAdapters(self._engine, base, text=lambda: self._text, on_change=self._prompt_cache_clear))
        self._prompt_encoder = prompt_encoder
        self._prompt_cache: "OrderedDict" = OrderedDict()
        self._text = None
        self._tokenizers = None
        ck_text = bool(checkpoints and "text_encoder" in checkpoints and "text_encoder_2" in checkpoints)
        if (text_encoders or ck_text) and prompt_encoder is None:
            # SURVEY 8(f)-1: the two CLIP text towers of encode_prompt on the same kernels
            from . import text_encoder as T
            ucfg = self._engine.unet.cfg
            if ck_text:
                from . import checkpoints as K
                self._say("[FastEditor] Loading the CLIP text encoders...")
                c1, p1 = K.load_clip_dir(checkpoints["text_encoder"])
                c2, p2 = K.load_clip_dir(checkpoints["text_encoder_2"])
                tokenizers = tokenizers or ((checkpoints["tokenizer"], checkpoints["tokenizer_2"]) if "tokenizer" in checkpoints and "tokenizer_2" in checkpoints else None)
            else:
                c1, c2 = (T.tiny_clip_config(False, "quick_gelu"), T.tiny_clip_config(True, "gelu")) if tiny else (T.clip_l_config(), T.openclip_bigg_config())
                self._say("[FastEditor] Building the CLIP text encoders (synthetic weights)...")
                p1, p2 = T.make_clip_params(c1), T.make_clip_params(c2)
            pooled_dim = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
            if c1.hidden_size + c2.hidden_size != ucfg.cross_attention_dim or c2.projection_dim != pooled_dim:
                raise ValueError("text encoder widths do not match the UNet's cross_attention_dim / pooled embedding size")
            with torch.cuda.device(self._dev):
                self._text = T.SDXLTextEncoders(p1, c1, p2, c2, self._dev)
            self._text_vocab = c1.vocab_size
            if tokenizers:
                # (tokenizer, tokenizer_2) folders with vocab.json + merges.txt: the real CLIP BPE (tokenizer.py)
                from .tokenizer import CLIPBPETokenizer
                self._tokenizers = (CLIPBPETokenizer.from_files(tokenizers[0]), CLIPBPETokenizer.from_files(tokenizers[1], pad_token="!"))
            elif ck_text:
                warnings.warn("FastEditor: text encoder checkpoints given without tokenizer folders; prompts are mapped to pseudo token ids", RuntimeWarning)
        elif checkpoints and prompt_encoder is None:
            warnings.warn("FastEditor: checkpoints without text_encoder / text_encoder_2 folders — prompts are mapped to seeded RANDOM "
                          "embeddings (pass prompt_encoder= or add the CLIP folders)", RuntimeWarning, stacklevel=2)
        self._say("[FastEditor] Initialization complete!")

    # ---- LoRA adapters (diffusers' names; see _PipeShim) ----
    def load_lora_weights(self, pretrained_model_name_or_path_or_dict, adapter_name: Optional[str] = None, weight_name: Optional[str] = None):
        self.pipe.load_lora_weights(pretrained_model_name_or_path_or_dict, adapter_name, weight_name)

    def set_adapters(self, adapter_names, adapter_weights=None):
        self.pipe.set_adapters(adapter_names, adapter_weights)

    def get_active_adapters(self) -> List[str]:
        return self.pipe.get_active_adapters()

    def get_list_adapters(self) -> Dict[str, List[str]]:
        return self.pipe.get_list_adapters()

    def delete_adapters(self, adapter_names):
        self.pipe.delete_adapters(adapter_names)

    def unload_lora_weights(self):
        self.pipe.unload_lora_weights()

    def _prompt_cache_clear(self):
        """Adapters changed: cached prompt embeddings may come from the old text-encoder weights."""
        self._prompt_cache.clear()

    # ---- prompt -> embeddings ----
    def _encode_prompt(self, prompt: str, negative_prompt: str):
        """-> (prompt_embeds [2,77,D], pooled [2,P]) with row 0 = negative, row 1 = positive (the empty negative prompt is ENCODED,
        as in the reference: it is passed explicitly, src/pipeline.py:263)."""
        pe, pl = self._encode_prompts([prompt], [negative_prompt])
        return pe[0], pl[0]

    def _encode_prompts(self, prompts: Sequence[str], negs: Sequence[str]):
        """Batched ``encode_prompt``: -> (prompt_embeds [B,2,77,D], pooled [B,2,P]) on the device.  Every distinct text runs through the
        two CLIP towers ONCE per call (all texts of the micro-batch in one pass; a tower treats sequences independently), and a small
        LRU keeps recent texts — the negative prompt is the same string for a whole sweep."""
        dev = self._dev
        if self._prompt_encoder is not None:                      # user hook: (prompt, negative) -> ([2,77,D], [2,P])
            enc = [self._prompt_encoder(p, n) for p, n in zip(prompts, negs)]
            return (torch.stack([e[0].to(dev, torch.float16) for e in enc]), torch.stack([e[1].to(dev, torch.float16) for e in enc]))
        cache = self._prompt_cache
        todo = [t for t in dict.fromkeys(list(negs) + list(prompts)) if t not in cache]
        if todo:
            if self._text is not None:
                if self._tokenizers is not None:
                    ids1, ids2 = (torch.tensor(t(todo), dtype=torch.int64) for t in self._tokenizers)
                else:
                    from .text_encoder import pseudo_token_ids
                    ids1 = ids2 = torch.stack([pseudo_token_ids(t, self._text_vocab) for t in todo])
                hid, pooled = self._text.encode(ids1, ids2)          # [T,77,2048], [T,1280]
                for i, t in enumerate(todo):
                    cache[t] = (hid[i], pooled[i])
            else:
                ucfg = self._engine.unet.cfg
                pooled_dim = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
                for t in todo:                                       # no text encoder: deterministic embeddings seeded by the text
                    e = S.synthetic_prompt(zlib.crc32(t.encode("utf-8")) % (1 << 30), ucfg.cross_attention_dim, pooled_dim)
                    cache[t] = tuple(v.to(torch.float16).pin_memory().to(dev, non_blocking=True) for v in (e[0][1], e[1][1]))   # (async: see text_encoder.forward)
        pe = torch.stack([torch.stack([cache[n][0], cache[p][0]]) for p, n in zip(prompts, negs)])
        pl = torch.stack([torch.stack([cache[n][1], cache[p][1]]) for p, n in zip(prompts, negs)])
        for t in list(negs) + list(prompts):
            cache.move_to_end(t)
        while len(cache) > 64:
            cache.popitem(last=False)
        return pe, pl

    def preprocess_image(self, image, low_threshold=100, high_threshold=200, *, gaussian_blur=False):
        """PIL image (RGB, or 2-D gray array) -> PIL RGB Canny edge map (reference ``src/pipeline.py:183-210``).
        ``gaussian_blur`` (extension, default off as in the reference): cv2.GaussianBlur(gray, (5, 5), 0) before cv2.Canny."""
        image_np = np.ascontiguousarray(np.array(image))
        if image_np.dtype != np.uint8 or image_np.ndim not in (2, 3):
            raise ValueError("preprocess_image expects an 8-bit RGB or gray image")
        if image_np.ndim == 3 and image_np.shape[2] != 3:
            image_np = np.ascontiguousarray(image_np[..., :3])
        with torch.cuda.device(self._dev):
            d = torch.from_numpy(image_np[None]).to(self._dev)
            edges = ops.canny(d, int(np.floor(low_threshold)), int(np.floor(high_threshold)), out_channels=3, gaussian_blur=gaussian_blur)
            return Image.fromarray(edges[0].cpu().numpy())

    def _draw_noises(self, seed, n_exec: int, size=(OUT_SIZE, OUT_SIZE)) -> List[torch.Tensor]:
        """Reference RNG order for one image of ``size`` = (width, height): posterior sample, init noise, then one draw per non-final
        executed step, each [1, 4, height/8, width/8]."""
        gen = torch.Generator(device=self._dev)
        if seed is not None:
            gen.manual_seed(int(seed))
        else:
            gen.seed()
        shape = (1, 4, size[1] // 8, size[0] // 8)
        return [torch.randn(shape, generator=gen, device=self._dev, dtype=torch.float16) for _ in range(2 + max(n_exec - 1, 0))]

    def _to_device(self, image, size=(OUT_SIZE, OUT_SIZE)) -> torch.Tensor:
        """PIL image of any size -> uint8 [1,height,width,3] on the GPU; ``image.resize(size, Image.LANCZOS)`` of the reference
        (src/pipeline.py:251, there with size = (1024, 1024)) runs on the GPU, bit-identical to Pillow."""
        arr = np.ascontiguousarray(np.array(image.convert("RGB")))
        img = torch.from_numpy(arr[None]).pin_memory().to(self._dev, non_blocking=True)      # pinned staging: the copy does not block the host
        w, h = size
        if img.shape[1] != h or img.shape[2] != w:
            img = ops.resize_lanczos(img, h, w)
        return img

    def edit(self, image, prompt, negative_prompt="", strength=0.80, num_inference_steps=4, guidance_scale=1.5,
             controlnet_conditioning_scale=0.5, canny_low_threshold=100, canny_high_threshold=200, seed=None, *, canny_gaussian_blur=False,
             size=None):
        """Edit an image with a text prompt, preserving structure via Canny conditioning -> PIL RGB image of ``size`` (default
        1024x1024; see :func:`resolve_size`).  One image through :meth:`edit_many`: warm_up(micro_batch=1) captures the graph it
        replays."""
        executed_steps(strength, num_inference_steps)         # diffusers' check_inputs / get_timesteps messages, naming no image
        return self.edit_many([image], [prompt], [negative_prompt], strength, num_inference_steps, guidance_scale, controlnet_conditioning_scale,
                              canny_low_threshold, canny_high_threshold, seeds=[seed], micro_batch=1, canny_gaussian_blur=canny_gaussian_blur,
                              size=size)[0]

    def edit_many(self, images: Sequence, prompts: Union[str, Sequence[str]], negative_prompt: Union[str, Sequence[str]] = "", strength=0.80,
                  num_inference_steps=4, guidance_scale=1.5, controlnet_conditioning_scale=0.5, canny_low_threshold=100, canny_high_threshold=200,
                  seed=None, seeds: Optional[Sequence[Optional[int]]] = None, micro_batch: Optional[int] = None,
                  canny_gaussian_blur: bool = False, output: str = "pil", jpeg_quality: int = 75, *, size=None) -> List:
        """Batched ``edit``: ``[edit(images[i], prompts[i], ..., seed=seeds[i]) for i]`` — same per-image semantics (each image gets its
        own generator seeded with ``seeds[i]``, or ``seed`` for all, drawing in the reference's order; the results are the ones the
        per-image calls give) but run in micro-batches of ``micro_batch`` (default 8) images per engine call.

        ``output="jpeg"``: returns the edited images as JPEG files (``bytes``, what ``image.save("x.jpg")`` would write — byte-identical
        to Pillow's encoder at ``jpeg_quality``), encoded on the GPU: ~0.1-0.3 MB instead of 3 MB per image cross PCIe and the host
        does no pixel work at all.

        ``strength``, ``num_inference_steps``, ``guidance_scale``, ``controlnet_conditioning_scale``, ``canny_low_threshold`` and
        ``canny_high_threshold`` each take a scalar (every image) or a sequence with one value per image.  The values are device data of
        the edit, so images with different settings share a micro-batch and its CUDA graph.

        ``size`` as in :meth:`edit`.  The images are grouped by (size, executed step count, guidance > 1): the images of one micro-batch
        run the same launch sequence (with ``guidance_scale <= 1`` only the positive prompt rows run, as in diffusers).  Each group runs
        in its own micro-batches and the results come back in input order.

        The host side is pipelined: while the GPU runs micro-batch *i* (one CUDA-graph replay), the host converts the outputs of
        micro-batch *i-1* to PIL images and stages the inputs of *i+1* (pinned buffers, asynchronous copies)."""
        n = len(images)
        if isinstance(prompts, str):
            prompts = [prompts] * n
        negs = [negative_prompt] * n if isinstance(negative_prompt, str) else list(negative_prompt)
        if len(prompts) != n or len(negs) != n:
            raise ValueError("edit_many: images, prompts (and negative prompts) must have the same length")
        if seeds is None:
            seeds = [seed] * n
        if len(seeds) != n:
            raise ValueError("edit_many: seeds must have one entry per image")
        if output not in ("pil", "jpeg"):
            raise ValueError("edit_many: output must be 'pil' or 'jpeg'")
        st = per_image_settings(n, strength, num_inference_steps, guidance_scale, controlnet_conditioning_scale, canny_low_threshold,
                                canny_high_threshold)
        mb = int(micro_batch or self.MICRO_BATCH)
        sizes = [resolve_size(size, im.size) for im in images]
        chunks = micro_batches(sizes, st["n_exec"], st["guidance_scale"], mb)
        results: List[Optional[Image.Image]] = [None] * n
        pending = None                                   # (index list, pinned output buffer, event) of the micro-batch in flight
        with torch.cuda.device(self._dev):
            stream = torch.cuda.current_stream(self._dev)

            def finalize(p):
                idx, host_out, ev = p
                ev.synchronize()
                if output == "jpeg":
                    files, sizes, files_d = host_out
                    for j, i in enumerate(idx):
                        n_ = int(sizes[j])
                        if n_ <= files.shape[1]:
                            results[i] = files[j, :n_].numpy().tobytes()
                        else:                                      # larger than the copied prefix: fetch this one file exactly
                            results[i] = files_d[j, :n_].cpu().numpy().tobytes()
                        self._jpeg_prefix = min(files_d.shape[1], max(self._jpeg_prefix, -(-(n_ * 5 // 4) // 65536) * 65536))
                    return
                for j, i in enumerate(idx):
                    results[i] = Image.fromarray(host_out[j].numpy().copy())

            trace = getattr(self, "_trace", None)          # scripts/e2e_probe.py: host seconds per phase
            import time as _time

            def mark(name, t0):
                if trace is not None:
                    trace.append((name, _time.perf_counter() - t0))
                return _time.perf_counter()

            for k, ((wh, n_exec, _), idx) in enumerate(chunks):
                t_ = _time.perf_counter()
                nb = len(idx)
                pad_to = mb if nb * 2 >= mb else 1 << (nb - 1).bit_length()       # ragged tail: reuse the full-size graph, or the next power of two
                host_in, host_out = self._host_buffers(mb, wh)[k & 1]
                same = all(images[i].size == wh for i in idx)
                if same:
                    for j, i in enumerate(idx):
                        host_in[j].copy_(torch.from_numpy(np.array(images[i].convert("RGB"))))
                    for j in range(nb, pad_to):
                        host_in[j].copy_(host_in[nb - 1])
                    d_img = host_in[:pad_to].to(self._dev, non_blocking=True)
                else:
                    parts = [self._to_device(images[i], wh) for i in idx]
                    d_img = torch.cat(parts + [parts[-1]] * (pad_to - nb), 0)
                t_ = mark("stage images (PIL->pinned->H2D)", t_)
                pad = [idx[-1]] * (pad_to - nb)
                pe, pl = self._encode_prompts([prompts[i] for i in idx + pad], [negs[i] for i in idx + pad])      # [B,2,77,D], [B,2,P]
                t_ = mark("encode prompts (launch)", t_)
                per_img = [self._draw_noises(seeds[i], n_exec, wh) for i in idx]
                per_img += [per_img[-1]] * (pad_to - nb)
                noises = [torch.cat([p[d] for p in per_img], 0) for d in range(len(per_img[0]))]
                t_ = mark("noise draws (launch)", t_)
                sel = lambda name: [st[name][i] for i in idx + pad]
                out = self._engine.edit_batch(d_img, pe, pl, noises, strength=sel("strength"), num_inference_steps=sel("num_inference_steps"),
                                              guidance_scale=sel("guidance_scale"), controlnet_conditioning_scale=sel("controlnet_conditioning_scale"),
                                              canny_low=sel("canny_low_threshold"), canny_high=sel("canny_high_threshold"), canny_blur=canny_gaussian_blur)
                t_ = mark("edit_batch (graph launch)", t_)
                if output == "jpeg":
                    # Encode on the GPU.  The file sizes are not known on the host yet, so a prefix of every file buffer is copied whose
                    # length adapts to the largest file seen so far (+25 %, starting at 1/8 of the worst case); a file that does not
                    # fit is fetched exactly in finalize().
                    files_d, sizes_d = ops.jpeg_encode(out.images[:nb], jpeg_quality)
                    pre = min(files_d.shape[1], self.__dict__.setdefault("_jpeg_prefix", max(files_d.shape[1] // 8, 1 << 16)))
                    key = ("jpeg", k & 1, nb, pre)
                    pinned = self.__dict__.setdefault("_pinned", {})
                    if key not in pinned:
                        for old in [q for q in pinned if isinstance(q, tuple) and q[:2] == key[:2]]:
                            del pinned[old]
                        pinned[key] = (torch.empty((nb, pre), dtype=torch.uint8).pin_memory(), torch.empty((nb,), dtype=torch.int32).pin_memory())
                    hf, hs = pinned[key]
                    hf.copy_(files_d[:, :pre], non_blocking=True)
                    hs.copy_(sizes_d, non_blocking=True)
                    host_out = (hf, hs, files_d)
                else:
                    host_out[:nb].copy_(out.images[:nb], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(stream)
                t_ = mark("D2H enqueue", t_)
                if pending is not None:
                    finalize(pending)                    # host work of the previous micro-batch overlaps this one's GPU time
                t_ = mark("finalize previous (wait + PIL)", t_)
                pending = (idx, host_out, ev)
            if pending is not None:
                finalize(pending)
        return results  # type: ignore[return-value]

    def warm_up(self, micro_batch: Optional[int] = None, *, size=None, **edit_kwargs) -> float:
        """Runs one dummy micro-batch with the given ``edit`` arguments so that the CUDA graph for that shape / schedule is captured and
        the pinned staging buffers exist before the first real call (sweeps call this during initialisation).  The graph serves every
        setting with the same size, executed step count and CFG on/off (guidance > 1), whatever the guidance, scales, thresholds.  ``size`` as in
        :meth:`edit`; ``"auto"`` warms up the square bucket.  Returns the seconds spent."""
        import time
        t0 = time.perf_counter()
        mb = int(micro_batch or self.MICRO_BATCH)
        wh = resolve_size(size, (self.OUT_SIZE, self.OUT_SIZE))
        dummy = [Image.new("RGB", wh, (127, 127, 127))] * mb
        self.edit_many(dummy, "warm-up", seed=0, micro_batch=mb, size=wh, **edit_kwargs)
        torch.cuda.synchronize(self._dev)
        return time.perf_counter() - t0

    def _host_buffers(self, mb: int, size=(OUT_SIZE, OUT_SIZE)):
        """Two (input, output) pairs of pinned uint8 staging buffers [mb,height,width,3] (allocated once per micro-batch size and image
        size = (width, height))."""
        cache = self.__dict__.setdefault("_pinned", {})
        w, h = size
        key = (mb, h, w)
        if key not in cache:
            cache[key] = [(torch.empty((mb, h, w, 3), dtype=torch.uint8).pin_memory(), torch.empty((mb, h, w, 3), dtype=torch.uint8).pin_memory())
                          for _ in range(2)]
        self._pinned_last = key
        return cache[key]

    def clear_memory(self):
        """Clear GPU memory cache (reference ``src/pipeline.py:276-279``).  Also drops every captured CUDA graph except the most
        recently used one (each holds a private memory pool) and the pinned staging buffers of every image size but the most recently
        used one (about 100 MB per size at 8 images per micro-batch), so a parameter sweep cannot grow memory without bound."""
        if str(self.device).startswith("cuda"):
            self._engine.release_graphs(keep=1)
            pinned = self.__dict__.get("_pinned", {})
            for key in [k for k in pinned if isinstance(k[0], int) and k != getattr(self, "_pinned_last", None)]:
                del pinned[key]
            with torch.cuda.device(self._dev):
                torch.cuda.empty_cache()

    def get_memory_usage(self):
        """``lora_pristine_gb``: the part of ``allocated_gb`` held by the pristine weight copies of active LoRA adapters (0 when the
        adapters are the ones the editor was built with)."""
        if str(self.device).startswith("cuda"):
            return {"allocated_gb": torch.cuda.memory_allocated(self._dev) / 1024 ** 3, "reserved_gb": torch.cuda.memory_reserved(self._dev) / 1024 ** 3,
                    "lora_pristine_gb": self.pipe.adapters.pristine_bytes() / 1024 ** 3}
        return {"allocated_gb": 0, "reserved_gb": 0}
