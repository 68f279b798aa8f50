"""Load-time weight layout transforms for the CUDA kernels (the cold path of ``FastEditor.__init__``,
reference ``src/pipeline.py:45-181``): conv weights to [Cout][kh][kw][Cin], GEGLU row interleave, LayerNorm fold, LoRA fuse.

Every transform has two implementations with the same result: on CUDA tensors the library's own kernels (``csrc/pack.cu``,
``fie_pack_* / fie_fold_layernorm_f16 / fie_fuse_lora_f32`` — SURVEY 8(b) ``fie_pack_weights_*``; no ATen / cuBLAS compute kernel
runs at load time), on CPU tensors plain torch ops (``EditEngine(pack_on_host=True)`` and the CPU tests, which are also what
``tests/test_gpu_kernels.py`` checks the kernels against).  ``dtype=torch.bfloat16`` gives the same layouts with bf16 elements (the bf16
VAE; ``fie_pack_*_bf16``)."""
from __future__ import annotations

from typing import Optional, Tuple

import torch

import os

from . import _lib

NATIVE = os.environ.get("FIE_NATIVE_PACK", "1") != "0"      # 0: torch ops also on CUDA tensors (debugging / A-B)


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


def _bf(dtype) -> bool:
    if dtype not in (torch.float16, torch.bfloat16):
        raise ValueError(f"packed weights are fp16 or bf16, not {dtype}")
    return dtype == torch.bfloat16


def cast_f16(w: torch.Tensor, dtype=torch.float16) -> torch.Tensor:
    """fp32 [N, K] -> fp16 (or bf16) [N, K] (a Linear / 1x1-conv weight as the GEMM's B operand)."""
    bf = _bf(dtype)
    if not (w.is_cuda and NATIVE):
        return w.to(dtype).contiguous()
    w = _f32(w)
    n, k = w.shape[0], w.numel() // w.shape[0]
    out = torch.empty(w.shape, dtype=dtype, device=w.device)
    fn = "fie_pack_rows_bf16" if bf else "fie_pack_rows_f16"
    with torch.cuda.device(w.device):
        _lib.check(getattr(_lib.lib(), fn)(w.data_ptr(), None, None, out.data_ptr(), None, n, k, _stream(w)), fn)
    return out


def pack_conv3x3(w: torch.Tensor, pad_cout_to: Optional[int] = None, pad_cin_to: Optional[int] = None, dtype=torch.float16) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> fp16 (or bf16) [Cout_p, 9*Cin_p] with K order (kh, kw, cin); zero padding of channels on request."""
    bf = _bf(dtype)
    cout, cin = w.shape[:2]
    cp = pad_cin_to or cin
    op = pad_cout_to or cout
    if w.is_cuda and NATIVE:
        w = _f32(w)
        out = torch.empty((op, 9 * cp), dtype=dtype, device=w.device)
        fn = "fie_pack_conv3x3_bf16" if bf else "fie_pack_conv3x3_f16"
        with torch.cuda.device(w.device):
            _lib.check(getattr(_lib.lib(), fn)(w.data_ptr(), out.data_ptr(), cout, cin, op, cp, _stream(w)), fn)
        return out
    out = torch.zeros((op, 3, 3, cp), dtype=dtype, device=w.device)
    out[:cout, :, :, :cin] = w.permute(0, 2, 3, 1).to(dtype)
    return out.reshape(op, 9 * cp).contiguous()


def pack_conv3x3_c8(w: torch.Tensor, pad_cout_to: Optional[int] = None) -> torch.Tensor:
    """[Cout, Cin<=8, 3, 3] -> fp16 [Cout_p, 3*2*64] for the tensor-core conv_in (fie_conv3x3_c8_f16): per kernel row kh two
    64-wide K blocks (hi, lo) whose element kw*8 + c is w[co, c, kh, kw]; the other 40 positions (padded pixels 3..7 of the
    window) are zero.  hi = fp16(w), lo = fp16(w - hi): the fp32 conv_in weights survive the fp16 tensor-core path to ~2^-22."""
    cout, cin = w.shape[:2]
    assert cin <= 8
    op = pad_cout_to or cout
    if w.is_cuda and NATIVE:
        w = _f32(w)
        out = torch.empty((op, 384), dtype=torch.float16, device=w.device)
        with torch.cuda.device(w.device):
            _lib.check(_lib.lib().fie_pack_conv3x3_c8_f16(w.data_ptr(), out.data_ptr(), cout, cin, op, _stream(w)), "fie_pack_conv3x3_c8_f16")
        return out
    w32 = w.float().permute(0, 2, 3, 1)                                            # [co][kh][kw][c]
    hi = w32.to(torch.float16)
    lo = (w32 - hi.float()).to(torch.float16)
    out = torch.zeros((op, 3, 2, 8, 8), dtype=torch.float16, device=w.device)     # [co][kh][hi|lo][pixel][channel]
    out[:cout, :, 0, :3, :cin] = hi
    out[:cout, :, 1, :3, :cin] = lo
    return out.reshape(op, 3 * 2 * 64).contiguous()


def pack_conv_up2x(w: torch.Tensor, dtype=torch.float16) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> fp16 (or bf16) [4, Cout, 4*Cin]: phase (a, b) weights of nearest-2x-upsample + conv3x3.
    Output row 2i+a reads input rows {i-1, i} (a = 0) or {i, i+1} (a = 1); the 3x3 taps that fall on the same input row are
    summed (in fp32): a=0 -> [W0, W1+W2], a=1 -> [W0+W1, W2]; identically for columns.  K order (ty, tx, cin)."""
    bf = _bf(dtype)
    if w.is_cuda and NATIVE:
        w = _f32(w)
        cout, cin = w.shape[:2]
        out = torch.empty((4, cout, 4 * cin), dtype=dtype, device=w.device)
        fn = "fie_pack_conv_up2x_bf16" if bf else "fie_pack_conv_up2x_f16"
        with torch.cuda.device(w.device):
            _lib.check(getattr(_lib.lib(), fn)(w.data_ptr(), out.data_ptr(), cout, cin, _stream(w)), fn)
        return out
    w = w.float()
    rows = {0: [w[:, :, 0], w[:, :, 1] + w[:, :, 2]], 1: [w[:, :, 0] + w[:, :, 1], w[:, :, 2]]}   # each [Cout, Cin, 3(kw)]
    out = []
    for a in (0, 1):
        for b in (0, 1):
            taps = []
            for ty in (0, 1):
                r = rows[a][ty]
                cols = [r[:, :, 0], r[:, :, 1] + r[:, :, 2]] if b == 0 else [r[:, :, 0] + r[:, :, 1], r[:, :, 2]]
                taps += cols                                   # (ty, tx) order, each [Cout, Cin]
            out.append(torch.stack(taps, dim=1).reshape(w.shape[0], -1))
    return torch.stack(out, 0).to(dtype).contiguous()


def pack_geglu(w: torch.Tensor, b: Optional[torch.Tensor]) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """GEGLU projection [8C, C] (value rows first, gate rows second) -> rows interleaved per accumulator tile:
    tile j = [value rows j*h..(j+1)*h | gate rows 4C+j*h..], h = fie_geglu_block_n(8C)/2."""
    n = w.shape[0]
    half = n // 2
    h = _lib.lib().fie_geglu_block_n(n) // 2
    assert half % h == 0
    idx = torch.arange(n, device=w.device).view(2, half // h, h).permute(1, 0, 2).reshape(-1)
    wp = w.index_select(0, idx).contiguous()
    bp = None if b is None else b.index_select(0, idx).float().contiguous()
    return wp, bp


def fold_layernorm(w: torch.Tensor, b: Optional[torch.Tensor], gamma: torch.Tensor, beta: Optional[torch.Tensor]):
    """LayerNorm (gamma, beta over K) followed by Linear(W [N, K], b) as ONE GEMM on the un-normalised rows (fie_epilogue
    ln_stats_in).  With W' = W (.) gamma and its rows centred over K, W'' = W' - mean_k(W'):
        sum_k x_k W''_nk = sum_k (x_k - mean(x)) W'_nk,   so   LN(x) W^T + b = rstd(x) * (x W''^T) + (b + W beta)
    and the epilogue only has to scale each row by its 1/sigma.  Returns (W'' fp16 [N, K], bias fp32 [N])."""
    if w.is_cuda and NATIVE:
        w = _f32(w)
        n, k = w.shape
        w16 = torch.empty((n, k), dtype=torch.float16, device=w.device)
        bias = torch.empty((n,), dtype=torch.float32, device=w.device)
        g32 = _f32(gamma.to(w.device))
        b32 = None if b is None else _f32(b.to(w.device))
        be32 = None if beta is None else _f32(beta.to(w.device))
        with torch.cuda.device(w.device):
            _lib.check(_lib.lib().fie_fold_layernorm_f16(w.data_ptr(), None if b32 is None else b32.data_ptr(), g32.data_ptr(),
                                                         None if be32 is None else be32.data_ptr(), w16.data_ptr(), bias.data_ptr(), n, k, _stream(w)),
                       "fie_fold_layernorm_f16")
        return w16, bias
    w32 = w.float() * gamma.float()[None, :]
    w16 = (w32 - w32.mean(dim=1, keepdim=True)).to(torch.float16).contiguous()
    bias = torch.zeros(w.shape[0], dtype=torch.float32, device=w.device) if b is None else b.float().clone()
    if beta is not None:
        bias = bias + w.float() @ beta.float()
    return w16, bias.contiguous()


def fuse_lora(w: torch.Tensor, lora_a: torch.Tensor, lora_b: torch.Tensor, scale: float) -> torch.Tensor:
    """W' = W + scale * B A  (re-association of the reference's unfused peft path, src/pipeline.py:154).
    Linear: A [r, in], B [out, r].  Conv: A [r, in, k, k], B [out, r, 1, 1]."""
    if w.is_cuda and NATIVE:
        out = w.float().clone().contiguous()                       # fp32 master copy, fused in place
        a32, b32 = _f32(lora_a.to(w.device)), _f32(lora_b.to(w.device))
        cout, rank = out.shape[0], a32.shape[0]
        cols = out.numel() // cout
        assert a32.numel() == rank * cols and b32.numel() == cout * rank, (tuple(w.shape), tuple(lora_a.shape), tuple(lora_b.shape))
        with torch.cuda.device(w.device):
            _lib.check(_lib.lib().fie_fuse_lora_f32(out.data_ptr(), a32.data_ptr(), b32.data_ptr(), float(scale), cout, rank, cols, _stream(w)),
                       "fie_fuse_lora_f32")
        return out
    w32 = w.float()
    if w.dim() == 4:
        delta = torch.einsum("or,rikl->oikl", lora_b.float()[:, :, 0, 0], lora_a.float())
    else:
        delta = lora_b.float() @ lora_a.float()
    return w32 + scale * delta
