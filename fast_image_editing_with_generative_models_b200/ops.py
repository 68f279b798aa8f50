"""Thin Python wrappers over the C-ABI: torch owns device memory and streams, the kernels do the work.

Activations are NHWC / token-major fp16 tensors.  Every wrapper raises if the CUDA library is unavailable.
The GEMM / convolution / GroupNorm / softmax / VAE-attention wrappers also take bf16 tensors (the bf16 VAE, DESIGN.md 3.11): a bf16
input goes to the ``*_bf16`` entry points, an fp16 input to the fp16 ones exactly as before.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

from . import _lib
from ._lib import Epilogue, check

ACT_NONE, ACT_SILU, ACT_GEGLU, ACT_GELU, ACT_QUICKGELU, ACT_RELU = 0, 1, 2, 3, 4, 5
LAUNCHES = 0  # number of our kernels launched through this module (bench reports it)
_KERNELS_PER_CALL = {"canny3": 4, "canny1": 3, "groupnorm": 2}


PROFILE = None  # set to a list to record (kernel family, algorithmic work, start event, end event) per call


def _count(n=1):
    global LAUNCHES
    LAUNCHES += n


class _prof:
    """Context manager: when ops.PROFILE is a list, brackets one C-ABI call with CUDA events on the launch stream."""

    def __init__(self, family: str, work: float, unit: str, tag: str = ""):
        self.on = PROFILE is not None
        if self.on:
            self.family, self.work, self.unit, self.tag = family, work, unit, tag
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)

    def __enter__(self):
        if self.on:
            self.e0.record()
        return self

    def __exit__(self, *a):
        if self.on:
            self.e1.record()
            PROFILE.append((self.family, self.work, self.unit, self.e0, self.e1, self.tag))
        return False


STAGES = []   # (name, event) marks recorded by stage() while PROFILE is a list


def stage(name: str):
    """Mark the start of a pipeline stage (Canny, VAE encode, denoising step k, VAE decode) on the launch stream; only when profiling."""
    if PROFILE is not None:
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        STAGES.append((name, e))


def stage_summary():
    """-> {stage: ms} between consecutive marks (the last mark must be 'end')."""
    torch.cuda.synchronize()
    out = {}
    for (n0, e0), (_, e1) in zip(STAGES[:-1], STAGES[1:]):
        out[n0] = out.get(n0, 0.0) + e0.elapsed_time(e1)
    return out


def profile_summary(by_tag: bool = False):
    """-> {family: dict(calls, ms, work, unit)} from the recorded events (synchronises)."""
    torch.cuda.synchronize()
    out = {}
    for fam, work, unit, e0, e1, tag in PROFILE or []:
        if by_tag:
            fam = f"{fam} {tag}"
        d = out.setdefault(fam, dict(calls=0, ms=0.0, work=0.0, unit=unit))
        d["calls"] += 1
        d["ms"] += e0.elapsed_time(e1)
        d["work"] += work
    return out


_DT = {torch.float16: _lib.DT_F16, torch.bfloat16: _lib.DT_BF16, torch.float32: _lib.DT_F32}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, dtype, name: str):
    if not t.is_cuda:
        raise _lib.FieError(f"{name}: expected a CUDA tensor (the B200 path has no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.FieError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise _lib.FieError(f"{name}: expected a contiguous tensor")


def canny(img_u8: torch.Tensor, low: int = 100, high: int = 200, out_channels: int = 1, gaussian_blur: bool = False) -> torch.Tensor:
    """uint8 [N,H,W,3] (RGB) or [N,H,W] (gray) -> uint8 edges [N,H,W] or [N,H,W,3] (0/255); == cv2.Canny.
    ``gaussian_blur`` (default off, as in the reference): gray -> cv2.GaussianBlur(gray, (5, 5), 0) -> Canny."""
    _req(img_u8, torch.uint8, "canny")
    if gaussian_blur:
        gray = rgb_to_gray(img_u8) if img_u8.dim() == 4 else img_u8
        img_u8 = gaussian_blur5(gray)
    in_ch = 3 if img_u8.dim() == 4 else 1
    n, h, w = img_u8.shape[:3]
    L = _lib.lib()
    ws_bytes = L.fie_canny_workspace_bytes(n, h, w)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=img_u8.device)
    out = torch.empty((n, h, w, 3) if out_channels == 3 else (n, h, w), dtype=torch.uint8, device=img_u8.device)
    with _prof("canny", float(n) * h * w * (in_ch + out_channels), "B"):
        check(L.fie_canny_u8(_p(img_u8), _p(out), n, h, w, in_ch, out_channels, int(low), int(high), _p(ws), ws_bytes, _stream()), "fie_canny_u8")
    _count(3)
    return out


def rgb_to_gray(img_u8: torch.Tensor) -> torch.Tensor:
    """uint8 [N,H,W,3] -> uint8 [N,H,W]; == cv2.cvtColor(img, cv2.COLOR_RGB2GRAY)."""
    _req(img_u8, torch.uint8, "rgb_to_gray")
    n, h, w, c = img_u8.shape
    if c != 3:
        raise _lib.FieError("rgb_to_gray: RGB input expected")
    out = torch.empty((n, h, w), dtype=torch.uint8, device=img_u8.device)
    check(_lib.lib().fie_rgb_to_gray_u8(_p(img_u8), _p(out), n, h, w, _stream()), "fie_rgb_to_gray_u8")
    _count()
    return out


def gaussian_blur5(img_u8: torch.Tensor) -> torch.Tensor:
    """uint8 [N,H,W] or [N,H,W,3] -> same shape; bit-exact with cv2.GaussianBlur(img, (5, 5), 0)."""
    _req(img_u8, torch.uint8, "gaussian_blur5")
    c = img_u8.shape[3] if img_u8.dim() == 4 else 1
    n, h, w = img_u8.shape[:3]
    out = torch.empty_like(img_u8)
    with _prof("gaussian_blur5", 2.0 * img_u8.numel(), "B"):
        check(_lib.lib().fie_gaussian_blur5_u8(_p(img_u8), _p(out), n, h, w, c, _stream()), "fie_gaussian_blur5_u8")
    _count()
    return out


_JPEG_WS = {}


def jpeg_encode(img_u8: torch.Tensor, quality: int = 75):
    """uint8 [N,H,W,3] (CUDA) -> (uint8 [N, stride] buffer of N JPEG files, int32 [N] file sizes), byte-identical to
    ``PIL.Image.fromarray(img).save(f, "JPEG", quality=quality)`` (baseline, 4:2:0).  See :func:`jpeg_bytes` for the host side."""
    _req(img_u8, torch.uint8, "jpeg_encode")
    n, h, w, c = img_u8.shape
    if c != 3:
        raise _lib.FieError("jpeg_encode: RGB images expected")
    L = _lib.lib()
    stride = L.fie_jpeg_max_bytes(h, w)
    nbytes = L.fie_jpeg_workspace_bytes(n, h, w)
    key = (str(img_u8.device), n, h, w)
    ws = _JPEG_WS.get(key)
    if ws is None:
        _JPEG_WS.clear()
        ws = _JPEG_WS[key] = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=img_u8.device)
    out = torch.empty((n, stride), dtype=torch.uint8, device=img_u8.device)
    sizes = torch.empty((n,), dtype=torch.int32, device=img_u8.device)
    with _prof("jpeg_encode", float(img_u8.numel()), "B"):
        check(L.fie_jpeg_encode_u8(_p(img_u8), n, h, w, int(quality), _p(out), stride, _p(sizes), _p(ws), nbytes, _stream()), "fie_jpeg_encode_u8")
    _count(7)
    return out, sizes


def jpeg_bytes(img_u8: torch.Tensor, quality: int = 75):
    """-> list of N ``bytes`` objects (the JPEG files).  Two small D2H copies: the sizes, then only the used prefix of the buffer."""
    out, sizes = jpeg_encode(img_u8, quality)
    sz = sizes.cpu().tolist()
    m = max(sz) if sz else 0
    host = out[:, :m].cpu().numpy()
    return [host[i, :sz[i]].tobytes() for i in range(len(sz))]


_RS_TABLES = {}


def resize_pillow(img_u8: torch.Tensor, out_h: int, out_w: int, filter_name: str = "lanczos") -> torch.Tensor:
    """uint8 [N,H,W,3] (CUDA) -> uint8 [N,out_h,out_w,3], bit-identical to PIL ``Image.resize((out_w, out_h), Image.LANCZOS | BICUBIC)``."""
    from .resize import pillow_tables
    _req(img_u8, torch.uint8, "resize_pillow")
    n, h, w, c = img_u8.shape
    if c != 3:
        raise _lib.FieError("resize_pillow: RGB images expected")
    dev = img_u8.device
    key = (filter_name, h, w, out_h, out_w, str(dev))
    if key not in _RS_TABLES:
        bx, kx, ksx = pillow_tables(w, out_w, filter_name)
        by, ky, ksy = pillow_tables(h, out_h, filter_name)
        _RS_TABLES[key] = (bx.to(dev), kx.to(dev), ksx, by.to(dev), ky.to(dev), ksy)
    bx, kx, ksx, by, ky, ksy = _RS_TABLES[key]
    out = torch.empty((n, out_h, out_w, 3), dtype=torch.uint8, device=dev)
    tmp = torch.empty((n, h, out_w, 3), dtype=torch.uint8, device=dev) if (out_w != w and out_h != h) else None
    with _prof("resize", float(img_u8.numel() + out.numel()), "B"):
        check(_lib.lib().fie_resample_lanczos_u8(_p(img_u8), _p(out), _p(tmp), n, h, w, out_h, out_w, _p(bx), _p(kx), ksx, _p(by), _p(ky), ksy, _stream()),
              "fie_resample_lanczos_u8")
    _count((out_w != w) + (out_h != h))
    return out


def resize_lanczos(img_u8: torch.Tensor, out_h: int, out_w: int) -> torch.Tensor:
    return resize_pillow(img_u8, out_h, out_w, "lanczos")


def _f3(vals):
    return None if vals is None else (ctypes.c_float * 3)(*[float(v) for v in vals])


def resize_aa_normalize(img: torch.Tensor, out_h: int, out_w: int, mean=None, std=None) -> torch.Tensor:
    """uint8 (read as v/255) or fp32 [N,H,W,3] -> fp32 [N,out_h,out_w,3]: torchvision ``Resize(antialias=True)`` (bilinear) followed by
    ``Normalize(mean, std)`` — DinoDistanceMetric._to_tensor, reference ``src/metrics.py:124-136``."""
    from .resize import aa_bilinear_tables
    if img.dtype not in (torch.uint8, torch.float32) or not img.is_cuda or not img.is_contiguous() or img.shape[-1] != 3:
        raise _lib.FieError("resize_aa_normalize: contiguous uint8 / fp32 CUDA [N,H,W,3] expected")
    n, h, w, _ = img.shape
    dev = img.device
    key = ("aa", h, w, out_h, out_w, str(dev))
    if key not in _RS_TABLES:
        bx, kx, ksx = aa_bilinear_tables(w, out_w)
        by, ky, ksy = aa_bilinear_tables(h, out_h)
        _RS_TABLES[key] = (bx.to(dev), kx.to(dev), ksx, by.to(dev), ky.to(dev), ksy)
    bx, kx, ksx, by, ky, ksy = _RS_TABLES[key]
    out = torch.empty((n, out_h, out_w, 3), dtype=torch.float32, device=dev)
    tmp = torch.empty((n, h, out_w, 3), dtype=torch.float32, device=dev) if out_w != w else None
    check(_lib.lib().fie_resample_f32(_p(img), int(img.dtype == torch.uint8), _p(out), _p(tmp), n, h, w, out_h, out_w, _p(bx), _p(kx), ksx, _p(by), _p(ky), ksy,
                                      _f3(mean), _f3(std), _stream()), "fie_resample_f32")
    _count(1 + (out_w != w))
    return out


def ssim_u8(a: torch.Tensor, b: torch.Tensor, kernel_size: int = 11, sigma: float = 1.5, k1: float = 0.01, k2: float = 0.03) -> torch.Tensor:
    """uint8 [N,H,W,C] pairs -> fp64 [N] mean SSIM (torchmetrics ``StructuralSimilarityIndexMeasure(data_range=1.0)`` per image)."""
    _req(a, torch.uint8, "ssim_u8"); _req(b, torch.uint8, "ssim_u8")
    if a.shape != b.shape or a.dim() != 4:
        raise _lib.FieError("ssim_u8: two [N,H,W,C] images of one shape expected")
    n, h, w, c = a.shape
    out = torch.empty((n,), dtype=torch.float64, device=a.device)
    check(_lib.lib().fie_ssim_u8(_p(a), _p(b), n, h, w, c, kernel_size, float(sigma), float(k1), float(k2), _p(out), _stream()), "fie_ssim_u8")
    _count()
    return out / float(c * (h - kernel_size + 1) * (w - kernel_size + 1))


def sqdiff_u8(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """uint8 [N,...] pairs -> int64 [N] exact sums of squared byte differences."""
    _req(a, torch.uint8, "sqdiff_u8"); _req(b, torch.uint8, "sqdiff_u8")
    if a.shape != b.shape:
        raise _lib.FieError("sqdiff_u8: shapes differ")
    n = a.shape[0]
    out = torch.empty((n,), dtype=torch.int64, device=a.device)
    check(_lib.lib().fie_sqdiff_u8(_p(a), _p(b), n, a.numel() // n, _p(out), _stream()), "fie_sqdiff_u8")
    _count()
    return out


def patchify(img: torch.Tensor, patch: int, mean=None, std=None) -> torch.Tensor:
    """uint8 (v/255) or fp32 [N,H,W,3] -> fp16 [N*(H/P)*(W/P), P*P*3] patch rows (K order py, px, c), optionally normalised."""
    if img.dtype not in (torch.uint8, torch.float32) or not img.is_cuda or not img.is_contiguous() or img.shape[-1] != 3:
        raise _lib.FieError("patchify: contiguous uint8 / fp32 CUDA [N,H,W,3] expected")
    n, h, w, _ = img.shape
    out = torch.empty((n * (h // patch) * (w // patch), patch * patch * 3), dtype=torch.float16, device=img.device)
    check(_lib.lib().fie_patchify_f16(_p(img), int(img.dtype == torch.uint8), _p(out), n, h, w, patch, _f3(mean), _f3(std), _stream()), "fie_patchify_f16")
    _count()
    return out


def vit_assemble(patches: torch.Tensor, cls: torch.Tensor, pos: torch.Tensor, n: int) -> torch.Tensor:
    """patch rows fp16 [n*np, c] + class token [c] + position embeddings [np+1, c] -> tokens fp16 [n*(np+1), c]."""
    for t in (patches, cls, pos):
        _req(t, torch.float16, "vit_assemble")
    c = patches.shape[-1]
    npatch = patches.shape[0] // n
    if pos.shape[0] != npatch + 1 or pos.shape[-1] != c or cls.numel() != c:
        raise _lib.FieError("vit_assemble: position embeddings must be [n_patches + 1, c]")
    out = torch.empty((n * (npatch + 1), c), dtype=torch.float16, device=patches.device)
    check(_lib.lib().fie_vit_assemble_f16(_p(patches), _p(cls), _p(pos), _p(out), n, npatch, c, _stream()), "fie_vit_assemble_f16")
    _count()
    return out


def l2norm_rows(x: torch.Tensor, out: Optional[torch.Tensor] = None, eps: float = 1e-4) -> torch.Tensor:
    """fp16 [rows, c] (row stride allowed) -> rows / max(|row|, eps)."""
    if x.dtype != torch.float16 or not x.is_cuda or x.stride(-1) != 1:
        raise _lib.FieError("l2norm_rows: fp16 CUDA rows with unit inner stride required")
    rows, c = x.shape
    if out is None:
        out = torch.empty((rows, c), dtype=torch.float16, device=x.device)
    check(_lib.lib().fie_l2norm_rows_f16(_p(x), x.stride(0), _p(out), out.stride(0), rows, c, float(eps), _stream()), "fie_l2norm_rows_f16")
    _count()
    return out


def sqdiff_f32(a: torch.Tensor, b: torch.Tensor, rows: int, cols: int) -> torch.Tensor:
    """fp32 matrices (row strides allowed) -> fp64 [1] sum of squared differences over the leading rows x cols window."""
    for t in (a, b):
        if t.dtype != torch.float32 or not t.is_cuda or t.stride(-1) != 1:
            raise _lib.FieError("sqdiff_f32: fp32 CUDA rows with unit inner stride required")
    out = torch.empty((1,), dtype=torch.float64, device=a.device)
    check(_lib.lib().fie_sqdiff_f32(_p(a), a.stride(0), _p(b), b.stride(0), rows, cols, _p(out), _stream()), "fie_sqdiff_f32")
    _count()
    return out


def cosine_rows(a: torch.Tensor, b: torch.Tensor, eps: float = 1e-8) -> torch.Tensor:
    """fp16 [rows, c] pairs -> fp32 [rows] cosine similarities."""
    for t in (a, b):
        if t.dtype != torch.float16 or not t.is_cuda or t.stride(-1) != 1:
            raise _lib.FieError("cosine_rows: fp16 CUDA rows with unit inner stride required")
    rows, c = a.shape
    out = torch.empty((rows,), dtype=torch.float32, device=a.device)
    check(_lib.lib().fie_cosine_rows_f16(_p(a), a.stride(0), _p(b), b.stride(0), _p(out), rows, c, float(eps), _stream()), "fie_cosine_rows_f16")
    _count()
    return out


def im2col3x3(x: torch.Tensor, stride: int = 1, pad: int = 1, shift=None, scale=None, kpad: Optional[int] = None) -> torch.Tensor:
    """fp16 [N,H,W,C] (channel-strided views allowed) or the uint8 RGB network input -> fp16 [N*OH*OW, kpad >= 9C] (K order ky, kx, c;
    default kpad = 9C rounded up to 8, columns beyond 9C zero)."""
    if x.dtype not in (torch.uint8, torch.float16) or not x.is_cuda or x.stride(-1) != 1:
        raise _lib.FieError("im2col3x3: fp16 / uint8 CUDA NHWC tensor required")
    n, h, w, c = x.shape
    ld = x.stride(-2)
    if (h > 1 and x.stride(1) != w * ld) or (n > 1 and x.stride(0) != h * w * ld):        # (the stride of a size-1 dimension is arbitrary)
        raise _lib.FieError("im2col3x3: only the channel dimension may be strided")
    oh, ow = (h + 2 * pad - 3) // stride + 1, (w + 2 * pad - 3) // stride + 1
    kpad = (9 * c + 7) // 8 * 8 if kpad is None else int(kpad)
    out = torch.empty((n * oh * ow, kpad), dtype=torch.float16, device=x.device)
    check(_lib.lib().fie_im2col3x3_f16(_p(x), int(x.dtype == torch.uint8), ld, _p(out), n, h, w, c, stride, pad, kpad, _f3(shift), _f3(scale), _stream()),
          "fie_im2col3x3_f16")
    _count()
    return out


def maxpool3s2_ceil(x: torch.Tensor) -> torch.Tensor:
    """fp16 [N,H,W,C] -> MaxPool2d(3, 2, ceil_mode=True)."""
    _req(x, torch.float16, "maxpool3s2_ceil")
    n, h, w, c = x.shape
    oh, ow = (h - 2) // 2 + 1, (w - 2) // 2 + 1
    out = torch.empty((n, oh, ow, c), dtype=torch.float16, device=x.device)
    check(_lib.lib().fie_maxpool3s2_ceil_f16(_p(x), _p(out), n, h, w, c, _stream()), "fie_maxpool3s2_ceil_f16")
    _count()
    return out


def lpips_layer(f0: torch.Tensor, f1: torch.Tensor, lin: torch.Tensor) -> torch.Tensor:
    """fp16 [N,H,W,C] feature pairs, lin fp32 [C] -> fp64 [N]: spatial mean of sum_c lin[c] (unit(f0) - unit(f1))^2."""
    _req(f0, torch.float16, "lpips_layer"); _req(f1, torch.float16, "lpips_layer"); _req(lin, torch.float32, "lpips_layer")
    n, h, w, c = f0.shape
    if f1.shape != f0.shape or lin.numel() != c:
        raise _lib.FieError("lpips_layer: shape mismatch")
    out = torch.empty((n,), dtype=torch.float64, device=f0.device)
    check(_lib.lib().fie_lpips_layer_f16(_p(f0), _p(f1), _p(lin), n, h * w, c, _p(out), _stream()), "fie_lpips_layer_f16")
    _count()
    return out / float(h * w)


def preprocess(img_u8: torch.Tensor, c_out: int = 4, normalize: bool = True) -> torch.Tensor:
    _req(img_u8, torch.uint8, "preprocess")
    n, h, w, _ = img_u8.shape
    out = torch.empty((n, h, w, c_out), dtype=torch.float16, device=img_u8.device)
    check(_lib.lib().fie_preprocess_u8_to_f16(_p(img_u8), _p(out), n, h, w, c_out, int(normalize), _stream()), "fie_preprocess_u8_to_f16")
    _count()
    return out


def preprocess_pad8(img_u8: torch.Tensor, normalize: bool = True) -> torch.Tensor:
    """uint8 [N,H,W,3] -> fp16 zero-padded [N,H+2,W+8,8] (input layout of :func:`conv3x3_c8`)."""
    _req(img_u8, torch.uint8, "preprocess_pad8")
    n, h, w, _ = img_u8.shape
    out = torch.empty((n, h + 2, w + 8, 8), dtype=torch.float16, device=img_u8.device)
    check(_lib.lib().fie_preprocess_u8_to_f16_pad8(_p(img_u8), _p(out), n, h, w, int(normalize), _stream()), "fie_preprocess_u8_to_f16_pad8")
    _count()
    return out


def pad8(x4: torch.Tensor) -> torch.Tensor:
    """fp16 [N,H,W,4] -> zero-padded fp16 [N,H+2,W+8,8] (input layout of :func:`conv3x3_c8`)."""
    _req(x4, torch.float16, "pad8")
    n, h, w, c = x4.shape
    if c != 4:
        raise _lib.FieError("pad8: 4-channel input expected")
    out = torch.empty((n, h + 2, w + 8, 8), dtype=torch.float16, device=x4.device)
    check(_lib.lib().fie_pad8_f16(_p(x4), _p(out), n, h, w, _stream()), "fie_pad8_f16")
    _count()
    return out


def postprocess(x: torch.Tensor) -> torch.Tensor:
    """fp16 [N,H,W,C>=3] -> uint8 [N,H,W,3]."""
    _req(x, torch.float16, "postprocess")
    n, h, w, c = x.shape
    out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=x.device)
    check(_lib.lib().fie_postprocess_f16_to_u8(_p(x), c, _p(out), n, h, w, _stream()), "fie_postprocess_f16_to_u8")
    _count()
    return out


def add(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _req(a, torch.float16, "add"); _req(b, torch.float16, "add")
    out = torch.empty_like(a) if out is None else out
    with _prof("add", 6.0 * a.numel(), "B"):
        check(_lib.lib().fie_add_f16(_p(a), _p(b), _p(out), a.numel(), _stream()), "fie_add_f16")
    _count()
    return out


def silu(a: torch.Tensor) -> torch.Tensor:
    _req(a, torch.float16, "silu")
    out = torch.empty_like(a)
    check(_lib.lib().fie_silu_f16(_p(a), _p(out), a.numel(), _stream()), "fie_silu_f16")
    _count()
    return out


def upsample2x(x: torch.Tensor) -> torch.Tensor:
    _req(x, torch.float16, "upsample2x")
    n, h, w, c = x.shape
    out = torch.empty((n, 2 * h, 2 * w, c), dtype=torch.float16, device=x.device)
    with _prof("upsample2x", 2.0 * out.numel() + 2.0 * x.numel(), "B"):
        check(_lib.lib().fie_upsample2x_f16(_p(x), _p(out), n, h, w, c, _stream()), "fie_upsample2x_f16")
    _count()
    return out


def embed_tokens(ids: torch.Tensor, tok: torch.Tensor, pos: torch.Tensor) -> torch.Tensor:
    """ids int32 [B, T] -> fp16 [B*T, C] = tok[ids] + pos[t]  (CLIPTextEmbeddings)."""
    _req(ids, torch.int32, "embed_tokens"); _req(tok, torch.float16, "embed_tokens"); _req(pos, torch.float16, "embed_tokens")
    b, t = ids.shape
    c = tok.shape[1]
    out = torch.empty((b * t, c), dtype=torch.float16, device=ids.device)
    check(_lib.lib().fie_embed_tokens_f16(_p(ids), _p(tok), _p(pos), _p(out), b * t, t, c, tok.shape[0], _stream()), "fie_embed_tokens_f16")
    _count()
    return out


def sincos_embedding(vals, dim: int, device) -> torch.Tensor:
    vals = [float(v) for v in vals]
    arr = (ctypes.c_float * len(vals))(*vals)
    out = torch.empty((len(vals), dim), dtype=torch.float16, device=device)
    check(_lib.lib().fie_sincos_embedding(arr, len(vals), dim, _p(out), _stream()), "fie_sincos_embedding")
    _count()
    return out


def softmax_rows(s: torch.Tensor, scale: float, out: Optional[torch.Tensor] = None, out_dtype=torch.float16) -> torch.Tensor:
    """Row softmax of fp32 scores (scaled here) or fp16 scores (pre-scaled by the GEMM epilogue: pass scale = 1) -> fp16
    (fp32 scores: or bf16, by ``out_dtype`` or the dtype of ``out``)."""
    if s.dtype not in (torch.float32, torch.float16):
        raise _lib.FieError("softmax_rows: fp32 or fp16 scores expected")
    _req(s, s.dtype, "softmax_rows")
    rows, cols = s.shape
    out = torch.empty((rows, cols), dtype=out_dtype, device=s.device) if out is None else out
    f16 = s.dtype == torch.float16
    if out.dtype not in (torch.float16, torch.bfloat16) or (f16 and out.dtype != torch.float16):
        raise _lib.FieError("softmax_rows: fp16 output, or bf16 output of fp32 scores")
    with _prof("softmax_rows", (4.0 if f16 else 6.0) * rows * cols, "B"):
        fn = _lib.lib().fie_softmax_rows_f16 if f16 else (_lib.lib().fie_softmax_rows_f32_to_bf16 if out.dtype == torch.bfloat16
                                                           else _lib.lib().fie_softmax_rows_f32_to_f16)
        check(fn(_p(s), s.stride(0), _p(out), out.stride(0), rows, cols, float(scale), _stream()), "fie_softmax_rows")
    _count()
    return out


def softmax_rows_exp(s: torch.Tensor, scale: float = 1.0, out: Optional[torch.Tensor] = None):
    """fp16 scores [rows, cols] -> (P' = exp(scale (s - rowmax)) fp16, 1 / rowsum fp32 [rows]); pass the latter as ``row_scale`` of the
    P V GEMM.  In place when ``out is s``."""
    _req(s, torch.float16, "softmax_rows_exp")
    rows, cols = s.shape
    out = torch.empty((rows, cols), dtype=torch.float16, device=s.device) if out is None else out
    inv = torch.empty((rows,), dtype=torch.float32, device=s.device)
    with _prof("softmax_rows", 4.0 * rows * cols, "B"):
        check(_lib.lib().fie_softmax_rows_exp_f16(_p(s), s.stride(0), _p(out), out.stride(0), _p(inv), rows, cols, float(scale), _stream()), "fie_softmax_rows_exp_f16")
    _count()
    return out, inv


def _gn_stats_ok(n_out: int, groups: int, rows_per_image: int, ldd: int) -> bool:
    """Can the GEMM epilogue accumulate the GroupNorm statistics of its output? (see fie_epilogue.gn_stats)"""
    if groups <= 0 or n_out % groups or n_out % 32 or ldd % 16 or rows_per_image % 32:
        return False
    cpg = n_out // groups
    return cpg in GN_FUSE_CPG


# Channels-per-group for which the producing epilogue accumulates the GroupNorm statistics.  Measured on B200 (SDXL VAE, batch 8):
# the extra epilogue work costs more than the saved statistics pass for 4 and 8 channels per group (narrow-N convolutions are
# epilogue-sensitive), and wins for 16 and 32; the kernel supports {4, 8, 16, 32}.
GN_FUSE_CPG = tuple(int(t) for t in os.environ.get("FIE_GN_FUSE_CPG", "16,32").split(",") if t)    # (8 measured neutral on B200)


def _gn_stats_alloc(out: torch.Tensor, n_img: int, groups: int) -> torch.Tensor:
    st = torch.zeros((n_img, groups, 2), dtype=torch.int64, device=out.device)
    out._gn_stats = (st, groups)          # picked up by groupnorm() on this very tensor object
    return st


def zeros_i64(shape, device) -> torch.Tensor:
    """Zeroed int64 statistics workspace (one memset node; device memory is torch's job)."""
    return torch.zeros(shape, dtype=torch.int64, device=device)


def groupnorm(x0: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, silu: bool, groups: int = 32,
              x1: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x0 [N,H,W,C0] (+ optional concatenated x1 [N,H,W,C1]) -> [N,H,W,C0+C1] normalised (+SiLU).  If x0 was produced by a
    GEMM / conv call with ``gn_groups=groups``, its statistics already exist and only the apply pass runs.  bf16 inputs take the
    range-safe statistics of fie_groupnorm_bf16."""
    if x0.dtype == torch.bfloat16:
        return _groupnorm_bf16(x0, gamma, beta, eps, silu, groups, x1)
    _req(x0, torch.float16, "groupnorm")
    n = x0.shape[0]
    c0 = x0.shape[-1]
    hw = x0.numel() // (n * c0)
    c1 = 0
    if x1 is not None:
        _req(x1, torch.float16, "groupnorm")
        c1 = x1.shape[-1]
    out = torch.empty(tuple(x0.shape[:-1]) + (c0 + c1,), dtype=torch.float16, device=x0.device)
    pre = getattr(x0, "_gn_stats", None) if x1 is None else None
    ready = pre is not None and pre[1] == groups and pre[0].shape[0] == n
    stats = pre[0] if ready else torch.empty((n, groups, 2), dtype=torch.int64, device=x0.device)
    with _prof("groupnorm", 4.0 * out.numel(), "B", f"[{n},{hw},{c0}+{c1}]" + (" fused-stats" if ready else "")):
        check(_lib.lib().fie_groupnorm_f16(_p(x0), c0, _p(x1), c1, _p(out), n, hw, groups, _p(gamma), _p(beta), float(eps), int(silu),
                                            _p(stats), int(ready), _stream()), "fie_groupnorm_f16")
    # launches: apply only (producer statistics), the single-pass slab kernel (default policy of csrc/norm.cu: the (image, group) slab fits
    # one CTA's shared memory), or statistics + apply
    cpg = (c0 + c1) // groups
    slab = (not ready) and cpg % 2 == 0 and hw >= 64 and hw * cpg * 2 <= 192 * 1024 and os.environ.get("FIE_GN_SLAB", "1") != "0"
    _count(1 if (ready or slab) else 2)
    return out


def _groupnorm_bf16(x0, gamma, beta, eps, silu, groups, x1):
    _req(x0, torch.bfloat16, "groupnorm")
    n = x0.shape[0]
    c0 = x0.shape[-1]
    hw = x0.numel() // (n * c0)
    c1 = 0
    if x1 is not None:
        _req(x1, torch.bfloat16, "groupnorm")
        c1 = x1.shape[-1]
    out = torch.empty(tuple(x0.shape[:-1]) + (c0 + c1,), dtype=torch.bfloat16, device=x0.device)
    L = _lib.lib()
    nbytes = L.fie_groupnorm_bf16_workspace_bytes(n, hw, c0 + c1, groups)
    ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=x0.device)
    with _prof("groupnorm", 4.0 * out.numel(), "B", f"[{n},{hw},{c0}+{c1}] bf16"):
        check(L.fie_groupnorm_bf16(_p(x0), c0, _p(x1), c1, _p(out), n, hw, groups, _p(gamma), _p(beta), float(eps), int(silu), _p(ws), ws.numel(),
                                   _stream()), "fie_groupnorm_bf16")
    cpg = (c0 + c1) // groups
    slab = cpg % 2 == 0 and hw >= 64 and hw * cpg * 2 <= 192 * 1024 and os.environ.get("FIE_GN_SLAB", "1") != "0"
    _count(1 if slab else 2)
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    _req(x, torch.float16, "layernorm")
    c = x.shape[-1]
    rows = x.numel() // c
    out = torch.empty_like(x)
    with _prof("layernorm", 4.0 * out.numel(), "B", f"[{rows},{c}]"):
        check(_lib.lib().fie_layernorm_f16(_p(x), _p(out), rows, c, _p(gamma), _p(beta), float(eps), _stream()), "fie_layernorm_f16")
    _count()
    return out


def _epilogue(col_bias=None, row_bias=None, rows_per_group=1, m_bias=None, residual=None, scale=1.0, act=ACT_NONE, out_f32=False, gn=None,
              ln_out=None, ln_in=None, row_scale=None):
    ep = Epilogue()
    ep.col_bias = _p(col_bias); ep.row_bias = _p(row_bias); ep.rows_per_group = int(rows_per_group)
    ep.ld_row_bias = row_bias.stride(-2) if (row_bias is not None and row_bias.dim() >= 2) else 0
    ep.m_bias = _p(m_bias)
    ep.residual = _p(residual); ep.ld_res = residual.stride(-2) if residual is not None else 0
    ep.scale = float(scale); ep.act = int(act); ep.out_f32 = int(out_f32)
    if gn is not None:                      # (stats tensor, groups, rows per image)
        ep.gn_stats = _p(gn[0]); ep.gn_groups = int(gn[1]); ep.gn_rows_per_image = int(gn[2])
    if ln_out is not None:                  # int64 [M, 2] row statistics of the output, zeroed by the caller
        ep.ln_stats_out = _p(ln_out)
    if ln_in is not None:                   # (int64 [M, 2] statistics of the A rows, eps)
        ep.ln_stats_in = _p(ln_in[0]); ep.ln_eps = float(ln_in[1])
    if row_scale is not None:
        ep.row_scale = _p(row_scale)
    return ep


def gemm(a: torch.Tensor, w: torch.Tensor, *, a1: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, n_valid: Optional[int] = None,
         col_bias=None, row_bias=None, rows_per_group=1, m_bias=None, residual=None, scale=1.0, act=ACT_NONE, out_f32=False,
         gn_groups: int = 0, gn_rows: int = 0, ln_out: Optional[torch.Tensor] = None, ln_in=None,
         row_scale: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """D = epilogue(A @ W^T).  a: [..., K] fp16 rows (row stride may exceed K), w: [N, K] fp16; optional a1 continues K.
    ln_out: zeroed int64 [M, 2] that receives the LayerNorm statistics of the output rows.  ln_in = (stats, eps): the A rows are
    layer-normalised on the fly (w / col_bias from weights.fold_layernorm).
    bf16 a / w (/ a1): fie_gemm_bf16, whose output is bf16 by default, else ``out_dtype`` / the dtype of ``out`` (fp16, bf16, fp32)."""
    bf = a.dtype == torch.bfloat16
    if bf:
        if w.dtype != torch.bfloat16 or (a1 is not None and a1.dtype != torch.bfloat16) or not a.is_cuda:
            raise _lib.FieError("gemm: bf16 A needs bf16 W (and A1) CUDA tensors")
    elif a.dtype != torch.float16 or w.dtype != torch.float16 or not a.is_cuda:
        raise _lib.FieError("gemm: fp16 CUDA tensors required")
    k0 = a.shape[-1]
    m = a.numel() // k0
    lda = a.stride(-2) if a.dim() >= 2 else k0
    n, k = w.shape
    k_split, lda1 = 0, 0
    if a1 is not None:
        k_split = k0
        lda1 = a1.stride(-2)
        assert k0 + a1.shape[-1] == k
    else:
        assert k0 == k, (k0, k)
    n_out = n // 2 if act == ACT_GEGLU else n
    if not bf and out_dtype not in (None, torch.float16):
        raise _lib.FieError("gemm: fp16 operands give fp16 (or, with out_f32, fp32) output")
    if out is None:
        odt = torch.float32 if out_f32 else (out_dtype or a.dtype)
        out = torch.empty(tuple(a.shape[:-1]) + (n_out,), dtype=odt, device=a.device)
    if bf:
        out_f32 = out.dtype == torch.float32
    ldd = out.stride(-2) if out.dim() >= 2 else n_out
    gn = None
    if gn_groups and gn_rows and not out_f32 and not bf and m % gn_rows == 0 and _gn_stats_ok(n_out, gn_groups, gn_rows, ldd):
        gn = (_gn_stats_alloc(out, m // gn_rows, gn_groups), gn_groups, gn_rows)
    if ln_out is not None and (ln_out.dtype != torch.int64 or ln_out.numel() != 2 * m or not ln_out.is_contiguous()):
        raise _lib.FieError("gemm: ln_out must be a contiguous int64 [M, 2] tensor")
    if ln_in is not None and (ln_in[0].dtype != torch.int64 or ln_in[0].numel() != 2 * m or not ln_in[0].is_contiguous()):
        raise _lib.FieError("gemm: ln_in = (contiguous int64 [M, 2] statistics, eps)")
    if row_scale is not None and (row_scale.dtype != torch.float32 or row_scale.numel() != m or not row_scale.is_contiguous()):
        raise _lib.FieError("gemm: row_scale must be a contiguous fp32 [M] tensor")
    ep = _epilogue(col_bias, row_bias, rows_per_group, m_bias, residual, scale, act, out_f32, gn, ln_out, ln_in, row_scale)
    ep.ln_dim = k
    with _prof("gemm", 2.0 * m * n * k, "FLOP", f"M{m} N{n} K{k} act{act} res{int(residual is not None)} f32{int(out_f32)}" + (" bf16" if bf else "")):
        if bf:
            check(_lib.lib().fie_gemm_bf16(_p(a), lda, _p(a1), lda1, k_split, _p(w), _p(out), ldd, m, n, k, ctypes.byref(ep), _DT[out.dtype], _stream()),
                  "fie_gemm_bf16")
        else:
            check(_lib.lib().fie_gemm_f16(_p(a), lda, _p(a1), lda1, k_split, _p(w), _p(out), ldd, m, n, k, ctypes.byref(ep), _stream()), "fie_gemm_f16")
    _count()
    return out


def _req_any(x: torch.Tensor, w: torch.Tensor, name: str) -> bool:
    """Activation and packed weight both fp16 (-> False) or both bf16 (-> True)."""
    if x.dtype == torch.bfloat16:
        _req(x, torch.bfloat16, name)
        if w.dtype != torch.bfloat16:
            raise _lib.FieError(f"{name}: bf16 activations need bf16 weights")
        return True
    _req(x, torch.float16, name)
    return False


def conv3x3(x: torch.Tensor, w: torch.Tensor, *, stride: int = 1, pad_mode: int = 0, cout_valid: Optional[int] = None,
            out: Optional[torch.Tensor] = None, col_bias=None, row_bias=None, rows_per_group=1, residual=None, scale=1.0, act=ACT_NONE,
            gn_groups: int = 0) -> torch.Tensor:
    """x [N,H,W,Cin] fp16, w packed [Cout, 9*Cin] fp16 -> [N,H/stride,W/stride,cout_valid].  bf16 x / w: fie_conv3x3_bf16, output in
    the dtype of ``out`` (default bf16); GroupNorm statistics are then left to the GroupNorm kernel."""
    bf = _req_any(x, w, "conv3x3")
    n, h, wd, cin = x.shape
    cout = w.shape[0]
    assert w.shape[1] == 9 * cin, (w.shape, cin)
    cv = cout if cout_valid is None else cout_valid
    if out is None:
        out = torch.empty((n, h // stride, wd // stride, cv), dtype=x.dtype, device=x.device)
    gn = None
    ohw = (h // stride) * (wd // stride)
    if gn_groups and not bf and cv == cout and _gn_stats_ok(cout, gn_groups, ohw, out.stride(-2)):
        gn = (_gn_stats_alloc(out, n, gn_groups), gn_groups, ohw)
    ep = _epilogue(col_bias, row_bias, rows_per_group, None, residual, scale, act, False, gn)
    with _prof("conv3x3", 2.0 * n * (h // stride) * (wd // stride) * cv * 9 * cin, "FLOP", f"[{n},{h},{wd},{cin}]->{cv} s{stride}" + (" bf16" if bf else "")):
        if bf:
            check(_lib.lib().fie_conv3x3_bf16(_p(x), _p(w), _p(out), out.stride(-2), n, h, wd, cin, cout, cv, stride, pad_mode, ctypes.byref(ep),
                                              _DT[out.dtype], _stream()), "fie_conv3x3_bf16")
        else:
            check(_lib.lib().fie_conv3x3_f16(_p(x), _p(w), _p(out), out.stride(-2), n, h, wd, cin, cout, cv, stride, pad_mode, ctypes.byref(ep), _stream()),
                  "fie_conv3x3_f16")
    _count()
    return out


def conv_up2x(x: torch.Tensor, w4: torch.Tensor, *, col_bias=None, out: Optional[torch.Tensor] = None, gn_groups: int = 0) -> torch.Tensor:
    """Fused nearest-2x upsample + conv3x3.  x [N,H,W,Cin], w4 packed [4, Cout, 4*Cin] (weights.pack_conv_up2x) -> [N,2H,2W,Cout].
    bf16 x / w4: fie_conv_up2x_bf16 (output dtype of ``out``, default bf16)."""
    bf = _req_any(x, w4, "conv_up2x")
    n, h, wd, cin = x.shape
    cout = w4.shape[1]
    assert w4.shape[0] == 4 and w4.shape[2] == 4 * cin, (w4.shape, cin)
    if out is None:
        out = torch.empty((n, 2 * h, 2 * wd, cout), dtype=x.dtype, device=x.device)
    gn = None
    if gn_groups and not bf and _gn_stats_ok(cout, gn_groups, h * wd, out.stride(-2)):
        gn = (_gn_stats_alloc(out, n, gn_groups), gn_groups, h * wd)       # rows of each phase launch are INPUT pixels: h*w per image
    ep = _epilogue(col_bias, gn=gn)
    with _prof("conv_up2x", 2.0 * n * 4 * h * wd * cout * 4 * cin, "FLOP", f"[{n},{h},{wd},{cin}]->{cout}" + (" bf16" if bf else "")):
        if bf:
            check(_lib.lib().fie_conv_up2x_bf16(_p(x), _p(w4), _p(out), out.stride(-2), n, h, wd, cin, cout, ctypes.byref(ep), _DT[out.dtype], _stream()),
                  "fie_conv_up2x_bf16")
        else:
            check(_lib.lib().fie_conv_up2x_f16(_p(x), _p(w4), _p(out), out.stride(-2), n, h, wd, cin, cout, ctypes.byref(ep), _stream()), "fie_conv_up2x_f16")
    _count(4)
    return out


def conv3x3_c8(xp: torch.Tensor, w: torch.Tensor, *, cout_valid: Optional[int] = None, col_bias=None, act=ACT_NONE, gn_groups: int = 0,
               residual: Optional[torch.Tensor] = None, out_dtype=torch.float16) -> torch.Tensor:
    """Tensor-core conv_in.  xp: zero-padded [N,H+2,W+8,8] fp16 (:func:`preprocess_pad8`), w: [Cout, 384] (weights.pack_conv3x3_c8)
    -> [N,H,W,cout_valid] fp16, or bf16 with ``out_dtype=torch.bfloat16`` (fie_conv3x3_c8_bf16: the operands stay fp16)."""
    _req(xp, torch.float16, "conv3x3_c8")
    n, hp, wp, c = xp.shape
    assert c == 8 and w.shape[1] == 384, (xp.shape, w.shape)
    h, wd = hp - 2, wp - 8
    cout = w.shape[0]
    cv = cout if cout_valid is None else cout_valid
    bf = out_dtype == torch.bfloat16
    out = torch.empty((n, h, wd, cv), dtype=out_dtype, device=xp.device)
    gn = None
    if gn_groups and not bf and cv == cout and _gn_stats_ok(cout, gn_groups, h * wd, out.stride(-2)):
        gn = (_gn_stats_alloc(out, n, gn_groups), gn_groups, h * wd)
    ep = _epilogue(col_bias, act=act, gn=gn, residual=residual)
    with _prof("conv_in_c8", 2.0 * out.numel() + 2.0 * xp.numel(), "B", f"[{n},{h},{wd},8]->{cv}" + (" bf16" if bf else "")):
        if bf:
            check(_lib.lib().fie_conv3x3_c8_bf16(_p(xp), _p(w), _p(out), out.stride(-2), n, h, wd, cout, cv, ctypes.byref(ep), _DT[out.dtype], _stream()),
                  "fie_conv3x3_c8_bf16")
        else:
            check(_lib.lib().fie_conv3x3_c8_f16(_p(xp), _p(w), _p(out), out.stride(-2), n, h, wd, cout, cv, ctypes.byref(ep), _stream()), "fie_conv3x3_c8_f16")
    _count()
    return out


def conv3x3_cin4(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], cout: int, ld_out: Optional[int] = None, act=ACT_NONE) -> torch.Tensor:
    """x [N,H,W,4] fp16, w fp32 [cout,3,3,4] -> [N,H,W,ld_out] fp16 (channels >= cout zero)."""
    _req(x, torch.float16, "conv3x3_cin4")
    n, h, wd, c = x.shape
    assert c == 4
    ld = cout if ld_out is None else ld_out
    out = torch.empty((n, h, wd, ld), dtype=torch.float16, device=x.device)
    with _prof("conv_cin4", 2.0 * out.numel() + 2.0 * x.numel(), "B"):
        check(_lib.lib().fie_conv3x3_cin4_f16(_p(x), _p(w), _p(bias), _p(out), ld, n, h, wd, cout, int(act), _stream()), "fie_conv3x3_cin4_f16")
    _count()
    return out


def attention_d64(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, b: int, heads: int, nq: int, nkv: int, out: Optional[torch.Tensor] = None,
                  scale: float = 0.125, causal: bool = False) -> torch.Tensor:
    """q [b*nq, >=heads*64] (row-strided views allowed), k/v [b*nkv, ...] -> [b*nq, heads*64]."""
    for t in (q, k, v):
        if t.dtype != torch.float16 or not t.is_cuda or t.stride(-1) != 1:
            raise _lib.FieError("attention_d64: fp16 CUDA tensors with unit inner stride required")
    if out is None:
        out = torch.empty((b * nq, heads * 64), dtype=torch.float16, device=q.device)
    with _prof("attention", 4.0 * b * heads * nq * nkv * 64, "FLOP", f"b{b} h{heads} nq{nq} nkv{nkv}"):
        fn = _lib.lib().fie_attention_d64_causal_f16 if causal else _lib.lib().fie_attention_d64_f16
        check(fn(_p(q), q.stride(-2), _p(k), k.stride(-2), _p(v), v.stride(-2), _p(out), out.stride(-2),
                                                b, heads, nq, nkv, float(scale), _stream()), "fie_attention_d64_f16")
    _count()
    return out


_VAE_WS = {}


def attention_vae(q: torch.Tensor, k: torch.Tensor, vt: torch.Tensor, scale: float, out: Optional[torch.Tensor] = None, f32_scores: bool = False,
                  chunk_rows: int = 0) -> torch.Tensor:
    """softmax(scale q k^T) v for ONE image of the VAE mid-block attention (1 head): q, k [ntok, d] fp16, vt [d, ntok] fp16 (V transposed)
    -> [ntok, d].  One C-ABI call (fie_attn_vae_d512_f16); the score workspace is cached per (device, shape).  bf16 q, k, vt:
    fie_attn_vae_d512_bf16, bf16 output, always fp32 scores."""
    bf = q.dtype == torch.bfloat16
    for t in (q, k, vt):
        _req(t, torch.bfloat16 if bf else torch.float16, "attention_vae")
    f32_scores = f32_scores or bf
    ntok, d = q.shape
    if out is None:
        out = torch.empty((ntok, d), dtype=q.dtype, device=q.device)
    L = _lib.lib()
    nbytes = L.fie_attn_vae_workspace_bytes(ntok, int(chunk_rows), int(f32_scores))
    key = (str(q.device), nbytes)
    ws = _VAE_WS.get(key)
    if ws is None or torch.cuda.is_current_stream_capturing():
        ws = torch.empty(nbytes, dtype=torch.uint8, device=q.device)       # (inside a graph capture: owned by the graph's pool)
        if not torch.cuda.is_current_stream_capturing():
            _VAE_WS.clear()
            _VAE_WS[key] = ws
    with _prof("vae_attention", 4.0 * ntok * ntok * d, "FLOP", f"ntok{ntok} d{d} f32{int(f32_scores)}" + (" bf16" if bf else "")):
        if bf:
            check(L.fie_attn_vae_d512_bf16(_p(q), q.stride(0), _p(k), k.stride(0), _p(vt), _p(out), out.stride(0), ntok, d, float(scale), int(chunk_rows),
                                           _p(ws), nbytes, _stream()), "fie_attn_vae_d512_bf16")
        else:
            check(L.fie_attn_vae_d512_f16(_p(q), q.stride(0), _p(k), k.stride(0), _p(vt), _p(out), out.stride(0), ntok, d, float(scale), int(f32_scores),
                                          int(chunk_rows), _p(ws), nbytes, _stream()), "fie_attn_vae_d512_f16")
    nchunks = 1 if chunk_rows <= 0 else -(-ntok // chunk_rows)
    _count(3 * nchunks)
    return out


def vae_sample_add_noise(moments: torch.Tensor, xi: torch.Tensor, noise: torch.Tensor, scaling: float, sqrt_a: float, sqrt_1ma: float):
    """moments [N,H,W,>=8] fp16, xi/noise [N,H,W,4] fp16 -> noisy latents [N,H,W,4] as (fp32 state, fp16 copy for the UNet)."""
    _req(moments, torch.float16, "vae_sample_add_noise")
    out32 = torch.empty(xi.shape, dtype=torch.float32, device=xi.device)
    out16 = torch.empty_like(xi)
    npx = xi.numel() // 4
    check(_lib.lib().fie_vae_sample_add_noise(_p(moments), moments.shape[-1], _p(xi), _p(noise), _p(out32), _p(out16), npx, float(scaling), float(sqrt_a),
                                               float(sqrt_1ma), _stream()), "fie_vae_sample_add_noise")
    _count()
    return out32, out16


def cfg_lcm_step(eps_u: torch.Tensor, eps_c: torch.Tensor, x32: torch.Tensor, noise: Optional[torch.Tensor], guidance: float, c: dict):
    """eps_u/eps_c: [N,H,W,ld] fp16 views (first 4 channels used); x32 [N,H,W,4] fp32 latent state; c = LCM step coefficients
    -> (fp32 state, fp16 copy)."""
    _req(x32, torch.float32, "cfg_lcm_step")
    out32 = torch.empty_like(x32)
    out16 = torch.empty(x32.shape, dtype=torch.float16, device=x32.device)
    npx = x32.numel() // 4
    check(_lib.lib().fie_cfg_lcm_step(_p(eps_u), _p(eps_c), eps_u.stride(-2), _p(x32), _p(noise), _p(out32), _p(out16), npx, float(guidance), float(c["sqrt_a"]),
                                       float(c["sqrt_1ma"]), float(c["c_skip"]), float(c["c_out"]), float(c["sqrt_a_prev"]), float(c["sqrt_1ma_prev"]),
                                       int(bool(c["last"])), _stream()), "fie_cfg_lcm_step")
    _count()
    return out32, out16
