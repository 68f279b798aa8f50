"""LoRA adapters on a built engine: diffusers' ``load_lora_weights`` / ``set_adapters`` / ``delete_adapters`` /
``unload_lora_weights`` (the reference adds its LCM-LoRA with ``load_lora_weights``, ``src/pipeline.py:154``), applied to the packed
fp16 weights in place.

Every packed layout is a linear map T of the diffusers weight W (:mod:`.weights`), so the packed delta of the active adapters of one
module is itself a low-rank product: B' = [w_1 B_1 | w_2 B_2 | ...] (rows permuted for GEGLU) times A'' = T applied to the stacked A_i
(LayerNorm fold: centred A (.) gamma, plus the bias delta B' (A beta); conv: (kh, kw, cin) order; up-sample: four phase-summed factors).
That product runs on the tensor-core GEMM (``fie_gemm_f16``, the factors as fp16 hi + lo pairs) with the pristine packed weight as the
epilogue residual and the live weight as its output: live = fp16(pristine + B' A''), rounded once from fp32.  The 8-channel ``conv_in`` (fp16 hi + lo pair) is not
linear in W: it is rebuilt from hi + lo + delta.

* The weights w_i are relative to the engine as built: the load-time LCM-LoRA (SDXL) is adapter ``default_0`` at 1.0, already fused.
* Nothing is allocated before the first load.  A packed weight (and folded bias) is copied to a pristine buffer the first time a
  delta touches it; every change recomputes from those copies; when the active set is back to the built one every written module is
  copied back (byte for byte) and the copies are freed.
* Writes are in place on the current stream of the engine's device, so device pointers, and with them every captured CUDA graph,
  stay valid.  Only the modules an adapter targets (now or at the previous change) are written.
* The ControlNet and the VAE are never adapted (as in diffusers).  Text-encoder parts apply to the GPU CLIP towers when the editor runs
  them, and are otherwise ignored with a RuntimeWarning."""
from __future__ import annotations

import math
import warnings
from collections import OrderedDict
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

from . import checkpoints as K
from . import ops
from .weights import LoraTarget, conv3x3_layout, conv_up2x_layout, fold_layernorm_lora, pack_conv3x3_c8, unpack_conv3x3_c8

Tensor = torch.Tensor
Params = Dict[str, Tensor]
_TAPS = {"rows": 1, "conv3": 9, "up2x": 9, "c8": 9}


def _pad64(n: int) -> int:
    return (n + 63) // 64 * 64


def _names(x, what: str) -> List[str]:
    names = [x] if isinstance(x, str) else list(x)
    if not all(isinstance(n, str) for n in names):
        raise ValueError(f"{what}: adapter names must be strings")
    return names


class _Adapter:
    """One loaded adapter: {part: peft dict}, the factor its B matrices are scaled by, and its weight in the engine as built (1.0 for a
    LoRA fused at build time, 0.0 for one loaded since).  Deltas are tied to this object, never to its name: a name can be deleted and
    then given to another adapter."""
    _serial = 0

    def __init__(self, parts: Dict[str, Params], b_scale: float = 1.0, built: float = 0.0):
        self.parts, self.b_scale, self.built = parts, float(b_scale), float(built)
        _Adapter._serial += 1
        self.key = _Adapter._serial                       # identity of the factors cached on the device


class LoraAdapters:
    """The adapter state of one engine (and its GPU text encoders, if any).  ``base``: {name: (peft dict, B scale)} of the UNet LoRAs
    fused at build time (active at 1.0); ``text()`` returns the ``SDXLTextEncoders`` or None; ``on_change()`` runs after every change
    (the editor drops its prompt cache)."""

    def __init__(self, engine, base: Optional[Dict[str, Tuple[Params, float]]] = None, text: Optional[Callable] = None,
                 on_change: Optional[Callable] = None):
        self.engine = engine
        self._text = text or (lambda: None)
        self._on_change = on_change or (lambda: None)
        # the build-time adapters, kept after a delete_adapters: their factors are fused into the built weights
        self._built: "OrderedDict[str, _Adapter]" = OrderedDict((name, _Adapter({"unet": peft}, scale, built=1.0))
                                                                 for name, (peft, scale) in (base or {}).items())
        self._adapters: "OrderedDict[str, _Adapter]" = OrderedDict(self._built)
        self._weights: Dict[str, float] = {name: a.built for name, a in self._built.items()}     # active adapters -> weight
        self._targets: Optional[Dict[str, Dict[str, LoraTarget]]] = None
        self._dev_factors: Dict[Tuple[int, str, str], Tuple[Tensor, Tensor]] = {}  # (adapter key, part, module) -> (A, B) fp32 on the device
        self._pristine: Dict[int, Tensor] = {}                                      # data_ptr of a live buffer -> its copy as built
        self._written: set = set()                                                  # (part, module) that may hold a delta now
        self._deltas: Dict = {}                                                     # the deltas the live weights hold

    # ---- queries ----
    def get_active_adapters(self) -> List[str]:
        return list(self._weights)

    def get_list_adapters(self) -> Dict[str, List[str]]:
        out: Dict[str, List[str]] = {}
        for name, ad in self._adapters.items():
            for part in ad.parts:
                out.setdefault(part, []).append(name)
        return out

    def pristine_bytes(self) -> int:
        """Device bytes of the pristine copies (0 whenever the active set is the one the engine was built with)."""
        return sum(t.numel() * t.element_size() for t in self._pristine.values())

    # ---- changes ----
    def load_lora_weights(self, path_or_dict, adapter_name: Optional[str] = None, weight_name: Optional[str] = None):
        if adapter_name is None:
            i = len(self._adapters)
            while f"default_{i}" in self._adapters:
                i += 1
            adapter_name = f"default_{i}"
        if not isinstance(adapter_name, str) or not adapter_name:
            raise ValueError("load_lora_weights: adapter_name must be a non-empty string")
        if adapter_name in self._adapters:
            raise ValueError(f"load_lora_weights: an adapter named {adapter_name!r} is already loaded")
        parts = K.split_lora(K.read_lora(path_or_dict, weight_name))
        targets = self._all_targets()
        adapter: Dict[str, Params] = {}
        for part, sd in parts.items():
            if part not in targets:
                warnings.warn(f"load_lora_weights: the {part} part of adapter {adapter_name!r} is ignored: prompts do not come from the GPU text "
                              "encoders (synthetic embeddings or the prompt_encoder hook)", RuntimeWarning, stacklevel=3)
                continue
            peft = K.lora_to_peft(sd, self._param_names(part), part)
            self._check(part, peft, targets[part])
            if peft:
                adapter[part] = peft
        if not adapter and not (set(parts) - set(targets)):
            raise ValueError("load_lora_weights: no LoRA tensors found")
        self._commit(OrderedDict(self._adapters, **{adapter_name: _Adapter(adapter)}), dict(self._weights, **{adapter_name: 1.0}))

    def set_adapters(self, adapter_names, adapter_weights=None):
        names = _names(adapter_names, "set_adapters")
        unknown = [n for n in names if n not in self._adapters]
        if unknown:
            raise ValueError(f"set_adapters: unknown adapters {unknown}; loaded: {list(self._adapters)}")
        if len(set(names)) != len(names):
            raise ValueError(f"set_adapters: an adapter is named twice in {names}")
        if adapter_weights is None:
            ws = [1.0] * len(names)
        elif isinstance(adapter_weights, (int, float)) and not isinstance(adapter_weights, bool):
            ws = [adapter_weights] * len(names)
        else:
            try:
                ws = list(adapter_weights)
            except TypeError:
                raise ValueError(f"set_adapters: adapter_weights must be a number or one number per adapter, got {adapter_weights!r}") from None
            if len(ws) != len(names):
                raise ValueError(f"set_adapters: {len(ws)} weights for {len(names)} adapters")
        try:
            ws = [float(w) for w in ws]
        except (TypeError, ValueError):
            raise ValueError(f"set_adapters: adapter weights must be numbers, got {adapter_weights!r}") from None
        if not all(math.isfinite(w) for w in ws):
            raise ValueError(f"set_adapters: adapter weights must be finite, got {ws}")
        self._commit(self._adapters, dict(zip(names, ws)))

    def delete_adapters(self, adapter_names):
        names = _names(adapter_names, "delete_adapters")
        unknown = [n for n in names if n not in self._adapters]
        if unknown:
            raise ValueError(f"delete_adapters: unknown adapters {unknown}; loaded: {list(self._adapters)}")
        self._commit(OrderedDict((n, a) for n, a in self._adapters.items() if n not in names),
                     {n: w for n, w in self._weights.items() if n not in names})

    def unload_lora_weights(self):
        """Back to the engine as built: every adapter loaded since is removed and the load-time ones are active at 1.0."""
        self._commit(OrderedDict(self._built), {name: a.built for name, a in self._built.items()})

    # ---- internals ----
    def _all_targets(self) -> Dict[str, Dict[str, LoraTarget]]:
        if self._targets is None:
            t = {"unet": self.engine.unet.lora_targets()}
            te = self._text()
            if te is not None:
                t["text_encoder"], t["text_encoder_2"] = te.enc1.lora_targets(), te.enc2.lora_targets()
            self._targets = t
        return self._targets

    def _param_names(self, part: str) -> List[str]:
        if part == "unet":
            from . import synthetic as S
            with S.shapes_only():
                return list(S.make_unet_params(self.engine.unet.cfg))
        te = self._text()
        return (te.enc1 if part == "text_encoder" else te.enc2).param_names

    @staticmethod
    def _check(part: str, peft: Params, targets: Dict[str, LoraTarget]):
        """ValueError unless every module of ``peft`` has a packed form that takes a delta and factors of its shape."""
        for k, a in peft.items():
            if not k.endswith(".lora_A.weight"):
                continue
            mod = k[: -len(".lora_A.weight")]
            t = targets.get(mod)
            if t is None:
                raise ValueError(f"LoRA: {part} module {mod!r} has no packed form that can take a delta (only Linear / Conv2d weights can)")
            b = peft[mod + ".lora_B.weight"]
            r = a.shape[0]
            ok = b.shape[0] == t.out and b.numel() == t.out * r and a.numel() == r * t.inp * _TAPS[t.kind]
            if t.kind != "rows":
                ok = ok and a.dim() == 4 and tuple(a.shape[2:]) == (3, 3)
            if not ok:
                raise ValueError(f"LoRA: {part} module {mod!r}: factors A {tuple(a.shape)}, B {tuple(b.shape)} do not fit its weight "
                                 f"({t.out} x {t.inp}{' x 3 x 3' if t.kind != 'rows' else ''})")

    def _factors(self, ad: _Adapter, part: str, mod: str) -> Tuple[Tensor, Tensor]:
        key = (ad.key, part, mod)
        f = self._dev_factors.get(key)
        if f is None:
            peft = ad.parts[part]
            a, b = peft[mod + ".lora_A.weight"], peft[mod + ".lora_B.weight"]
            b = b.to(self.engine.dev, torch.float32).reshape(b.shape[0], -1)
            f = self._dev_factors[key] = (a.to(self.engine.dev, torch.float32).reshape(a.shape[0], -1).contiguous(),
                                          (b * ad.b_scale if ad.b_scale != 1.0 else b).contiguous())
        return f

    def _commit(self, adapters: "OrderedDict[str, _Adapter]", weights: Dict[str, float]):
        """Apply the state (adapters, active weights), then make it current.  If the device update fails, the previous state is written
        back and the error raised: the adapters stay as they were."""
        contrib = [(ad, weights.get(name, 0.0) - ad.built) for name, ad in adapters.items()]
        # a build-time adapter that is no longer loaded (deleted, or its name now taken by another adapter): minus its fused factors
        contrib += [(ad, -ad.built) for name, ad in self._built.items() if adapters.get(name) is not ad]
        deltas: Dict[Tuple[str, str], List[Tuple[float, _Adapter]]] = OrderedDict()
        for ad, w in contrib:
            if w == 0.0:
                continue
            for part, peft in ad.parts.items():
                for k in peft:
                    if k.endswith(".lora_A.weight"):
                        deltas.setdefault((part, k[: -len(".lora_A.weight")]), []).append((w, ad))
        try:
            self._apply(deltas)
        except BaseException:
            try:
                self._apply(self._deltas)
            except Exception:
                pass
            raise
        self._deltas = deltas
        self._adapters = adapters
        self._weights = dict(weights)
        used = {ad.key for ws in deltas.values() for _, ad in ws}
        for key in [k for k in self._dev_factors if k[0] not in used]:
            del self._dev_factors[key]
        self._on_change()

    def _apply(self, deltas: Dict[Tuple[str, str], List[Tuple[float, _Adapter]]]):
        """Write the packed weights for ``deltas`` = {(part, module): [(weight relative to the build, adapter), ...]}.  A module is
        recorded in ``_written`` before its first write, so a later change restores it even if this one stops part way."""
        targets = self._all_targets()
        with torch.cuda.device(self.engine.dev), torch.no_grad():
            for part, mod in self._written - set(deltas):
                self._restore(targets[part][mod])
            self._written &= set(deltas)
            for (part, mod), ws in deltas.items():
                t = targets[part][mod]
                for buf in (t.weight, t.bias):
                    if buf is not None and buf.data_ptr() not in self._pristine:
                        self._pristine[buf.data_ptr()] = buf.clone()
                self._written.add((part, mod))
                self._write(t, [(w,) + self._factors(ad, part, mod) for w, ad in ws])
        if not deltas:
            self._pristine.clear()

    @staticmethod
    def _rows(t: LoraTarget, buf: Tensor) -> Tensor:
        """The part of a live (or pristine) buffer that belongs to module ``t``."""
        if t.kind in ("up2x", "c8") or t.perm is not None:
            return buf
        return buf[t.row0:t.row0 + t.out]

    def _restore(self, t: LoraTarget):
        for buf in (t.weight, t.bias):
            if buf is not None:
                self._rows(t, buf).copy_(self._rows(t, self._pristine[buf.data_ptr()]))

    def _write(self, t: LoraTarget, fs: Sequence[Tuple[float, Tensor, Tensor]]):
        """live = fp16(pristine + B' A'') for the factors (w_i, A_i [r_i, in * taps], B_i [out, r_i])."""
        bc = torch.cat([w * b for w, _, b in fs], 1)                 # B' [out, R]
        ac = torch.cat([a for _, a, _ in fs], 0)                     # [R, in * taps]
        r = ac.shape[0]
        pw = self._pristine[t.weight.data_ptr()]
        if t.kind == "c8":                                            # fp16 hi + lo pair: rebuilt from the fp32 sum
            w32 = unpack_conv3x3_c8(pw, t.out, t.inp) + (bc @ ac).view(t.out, t.inp, 3, 3)
            t.weight.copy_(pack_conv3x3_c8(w32, pad_cout_to=t.weight.shape[0]))
            return
        ab = None
        if t.kind == "rows":
            ak = ac
            if t.ln is not None:
                ak, ab = fold_layernorm_lora(ac, *t.ln)
            ak = [ak]
        elif t.kind == "conv3":
            ak = [conv3x3_layout(ac.view(r, t.inp, 3, 3), pad_cin_to=t.weight.shape[1] // 9)]
        else:                                                         # up2x: one product per phase
            ak = list(conv_up2x_layout(ac.view(r, t.inp, 3, 3)))
        if t.perm is not None:
            bc = bc.index_select(0, t.perm)
        if ab is not None:
            pb = self._pristine[t.bias.data_ptr()]
            self._rows(t, t.bias).copy_(self._rows(t, pb) + bc @ ab)
        # fp16 operands as hi + lo pairs, [Bh | Bh | Bl] x [Ah; Al; Ah] along K: the product keeps ~22 bits of the fp32 factors (fp16
        # factors alone would err by 2^-11 of |B'| |A''|, many fp16 ulps of a weight near zero), so the one rounding of the epilogue
        # dominates.  K = 3 R, zero-padded to the GEMM's 64.
        kp = _pad64(3 * r)
        bh = bc.to(torch.float16)
        a16 = torch.zeros((bc.shape[0], kp), dtype=torch.float16, device=bc.device)
        a16[:, :r], a16[:, r:2 * r], a16[:, 2 * r:3 * r] = bh, bh, (bc - bh.float()).to(torch.float16)
        live, base = self._rows(t, t.weight), self._rows(t, pw)
        for p, a2 in enumerate(ak):
            at = a2.t()
            ah = at.to(torch.float16)
            w16 = torch.zeros((at.shape[0], kp), dtype=torch.float16, device=bc.device)
            w16[:, :r], w16[:, r:2 * r], w16[:, 2 * r:3 * r] = ah, (at - ah.float()).to(torch.float16), ah
            out, res = (live[p], base[p]) if t.kind == "up2x" else (live, base)
            ops.gemm(a16, w16, out=out, residual=res)
