"""Float64 reference, per-element error bound, inputs and tile forms for the tensor-core GEMM (k_gemm_conv, csrc/gemm_conv.cu).
No GPU needed.

The reference is the epilogue contract of include/fie_b200.h computed in float64 from the exact fp16 / bf16 operand values:
    acc = A B^T                                  (a two-source A is the concatenation [A0 | A1] along K)
    pre = row_scale[m] acc + col_bias[n] + row_bias[m // rows_per_group][n] + m_bias[m]
    v   = act(pre) * scale + residual[m, n]
GEGLU reads B in the per-tile interleaved layout of weights.pack_geglu: output column j h + i takes the value from accumulator
column 2 j h + i (with col_bias and row_bias) and the gate from column 2 j h + h + i (with col_bias only), v = value gelu(gate).

Error model of a correct kernel against that reference, per element:
- accumulation in fp32 (tcgen05, K = 16 per instruction): one rounding of the running sum per 16-wide K step, at most one ulp
  (rounded or truncated), so |err| <= gamma_K sum_k |a_k b_k| |row_scale| with gamma_K = (ceil(K / 16) + 2) 2^-23;
- the epilogue adds the biases in fp32: at most three roundings, <= 2^-22 (|row_scale acc| + |col| + |row| + |m_bias|);
- both go through the activation with its largest slope: 1.13 for the erf GELU, 1.10 for SiLU and quick-GELU, 1 for ReLU
  and none; GEGLU by the product rule, |gelu(g)| e_val + |val| (1.13 e_gate + approximation error of gelu(g));
- the activation's own approximation error: relative 2^-20 for the MUFU exp / reciprocal, plus 2^-22 |x| relative for SiLU and
  quick-GELU (the exp argument x log2(e) is rounded to fp32), plus 2^-22 |x| absolute for the erf GELU (0.5 |x| times the
  1.5e-7 absolute error of the Abramowitz-Stegun erfc);
- times |scale|, plus 2^-23 (|scale act| + |residual|) for the fp32 product and residual add;
- output rounding: half an ulp, 2^-11 relative for fp16, 2^-8 for bf16, 2^-24 for fp32.  Values just above a power of two
  reach that, so the bound allows u_out (|ref| + error) with u_out one whole ulp (2^-10, 2^-7, 2^-23) to keep the margin of
  two below; plus 2^-24 absolute, which covers fp16 subnormals (rounded by 2^-25 absolute) and the underflow of the
  activations' tails.
The CPU emulation of the kernel's arithmetic below (emulate()) stays within half of this bound on every generator; rounding the
accumulator or v to fp16 too early, scaling after the residual, adding m_bias after the activation or a tanh GELU exceed it
(tests/test_gemm_cases_cpu.py).
"""
import contextlib
import math
from dataclasses import dataclass, replace
from typing import Optional

import torch

# activation codes of include/fie_b200.h (FIE_ACT_*)
NONE, SILU, GEGLU, GELU, QUICKGELU, RELU = 0, 1, 2, 3, 4, 5
ACT_NAMES = {NONE: "none", SILU: "silu", GELU: "gelu", QUICKGELU: "quickgelu", RELU: "relu", GEGLU: "geglu"}
SLOPE = {NONE: 1.0, SILU: 1.10, GELU: 1.13, QUICKGELU: 1.10, RELU: 1.0}
U_OUT = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7, torch.float32: 2.0 ** -23}      # one ulp: twice the rounding
ABS = 2.0 ** -24
SQRT1_2 = 0.7071067811865476


def gamma_k(k):
    return (math.ceil(k / 16) + 2) * 2.0 ** -23


def geglu_block_n(n):
    """fie_geglu_block_n (gemm_conv.cu), restated so that the CPU tests need no library."""
    return 256 if n % 256 == 0 else (128 if n % 128 == 0 else 64)


def geglu_columns(n, device=None):
    """(value, gate) accumulator columns of the N/2 output columns of a packed GEGLU weight [N, K]."""
    h = geglu_block_n(n) // 2
    o = torch.arange(n // 2, device=device)
    val = (o // h) * 2 * h + o % h
    return val, val + h


@dataclass
class Epi:
    """One epilogue: the keyword arguments of ops.gemm (tensors on the device of the operands, or None)."""
    col_bias: Optional[torch.Tensor] = None
    row_bias: Optional[torch.Tensor] = None
    rows_per_group: int = 1
    m_bias: Optional[torch.Tensor] = None
    row_scale: Optional[torch.Tensor] = None
    residual: Optional[torch.Tensor] = None
    scale: float = 1.0
    act: int = NONE

    def kwargs(self):
        return dict(col_bias=self.col_bias, row_bias=self.row_bias, rows_per_group=self.rows_per_group, m_bias=self.m_bias,
                    row_scale=self.row_scale, residual=self.residual, scale=self.scale, act=self.act)

    def to(self, dev):
        f = lambda t: None if t is None else t.to(dev)
        return replace(self, col_bias=f(self.col_bias), row_bias=f(self.row_bias), m_bias=f(self.m_bias), row_scale=f(self.row_scale),
                       residual=f(self.residual))


# ------------------------------------------------------------------ activations (float64, and the kernel's forms in fp32)
def act64(x, act):
    if act == NONE:
        return x
    if act == SILU:
        return x * torch.sigmoid(x)
    if act == GELU:
        return gelu64(x)
    if act == QUICKGELU:
        return x * torch.sigmoid(1.702 * x)
    if act == RELU:
        return x.clamp_min(0.0)
    raise ValueError(act)


def gelu64(x):
    return 0.5 * x * torch.special.erfc(-x * SQRT1_2)


def act_approx(x, y, act):
    """Bound on the approximation error of the kernel's activation at pre-activation x (y = act64(x))."""
    if act in (NONE, RELU):
        return torch.zeros_like(x)
    if act == GELU:
        return 2.0 ** -20 * y.abs() + 2.0 ** -22 * x.abs()
    k = 1.702 if act == QUICKGELU else 1.0
    return y.abs() * (2.0 ** -20 + 2.0 ** -22 * k * x.abs())


# ------------------------------------------------------------------ reference and bound
def reference(a, w, ep, a1=None, r0=0, r1=None):
    """Float64 reference of rows r0:r1, on a's device.  Returns a dict: out (v), err (the error model above before the output
    rounding), acc (row_scale acc), pre and act (act(pre)); for GEGLU also val_pre and gate_pre, with pre and acc the value's."""
    r1 = a.shape[0] if r1 is None else r1
    a = a[r0:r1]
    x = torch.cat([a, a1[r0:r1]], dim=1) if a1 is not None else a
    x, w = x.to(torch.float64), w.to(a.device, torch.float64)
    k = x.shape[1]
    acc = x @ w.t()
    sab = x.abs() @ w.abs().t()
    rs = ep.row_scale[r0:r1].double()[:, None] if ep.row_scale is not None else None
    if rs is not None:
        acc, sab = acc * rs, sab * rs.abs()
    n = w.shape[0]
    col = ep.col_bias.double()[None, :] if ep.col_bias is not None else torch.zeros((1, n), dtype=torch.float64, device=a.device)
    if ep.row_bias is not None:
        g = torch.arange(r0, r1, device=a.device) // ep.rows_per_group
        row = ep.row_bias.double()[g, :n]
    else:
        row = torch.zeros((1, n), dtype=torch.float64, device=a.device)
    mb = ep.m_bias[r0:r1].double()[:, None] if ep.m_bias is not None else torch.zeros((1, 1), dtype=torch.float64, device=a.device)
    res = ep.residual[r0:r1].double() if ep.residual is not None else None
    gk = gamma_k(k)
    d = {}
    if ep.act == GEGLU:
        vc, gc = geglu_columns(n, a.device)
        val = acc[:, vc] + col[:, vc] + row[:, vc]
        gate = acc[:, gc] + col[:, gc]
        e_val = gk * sab[:, vc] + 2.0 ** -22 * (acc[:, vc].abs() + col[:, vc].abs() + row[:, vc].abs())
        e_gate = gk * sab[:, gc] + 2.0 ** -22 * (acc[:, gc].abs() + col[:, gc].abs())
        gg = gelu64(gate)
        y = val * gg
        e = gg.abs() * e_val + val.abs() * (1.13 * e_gate + act_approx(gate, gg, GELU)) + 1.13 * e_val * e_gate + 2.0 ** -24 * y.abs()
        d.update(val_pre=val, gate_pre=gate, pre=val, acc=acc[:, vc])
    else:
        pre = acc + col + row + mb
        y = act64(pre, ep.act)
        e_pre = gk * sab + 2.0 ** -22 * (acc.abs() + col.abs() + row.abs() + mb.abs())
        e = SLOPE[ep.act] * e_pre + act_approx(pre, y, ep.act)
        d.update(pre=pre, acc=acc)
    out = y * ep.scale
    e = e * abs(ep.scale) + 2.0 ** -23 * out.abs()
    if res is not None:
        out = out + res
        e = e + 2.0 ** -23 * res.abs()
    d.update(out=out, err=e, act=y)
    return d


def expected(a, w, ep, out_dtype=torch.float16, a1=None, max_elems=1 << 25):
    """(ref, tol), float64 [M, N_out] on a's device, computed in row chunks of at most max_elems accumulator elements."""
    m, n = a.shape[0], w.shape[0]
    step = max(1, max_elems // n)
    refs, tols = [], []
    for r0 in range(0, m, step):
        d = reference(a, w, ep, a1, r0, min(m, r0 + step))
        refs.append(d["out"])
        tols.append(tolerance(d["out"], d["err"], out_dtype))
    return torch.cat(refs), torch.cat(tols)


def tolerance(ref, err, out_dtype):
    return err + U_OUT[out_dtype] * (ref.abs() + err) + ABS


def err_ratio(out, ref, tol):
    """max over elements of |out - ref| / tol; inf if out has a non-finite value."""
    if not bool(torch.isfinite(out).all()):
        return math.inf
    return float(((out.to(ref.device).double() - ref).abs() / tol).max())


# ------------------------------------------------------------------ emulation of the kernel's arithmetic (fp32 torch)
def _r16(x, dt):
    return x.to(dt).to(torch.float32)


def gelu_as32(x):
    """gelu_erf_f of fie_common.cuh in fp32 (rcp / ex2 exact to fp32 rounding)."""
    z = x.abs() * 0.70710678118654752440
    t = 1.0 / (0.3275911 * z + 1.0)
    pl = 1.061405429 * t - 1.453152027
    pl = pl * t + 1.421413741
    pl = pl * t - 0.284496736
    pl = pl * t + 0.254829592
    e = torch.exp2(-1.4426950408889634 * z * z)
    q = pl * t * e
    return 0.5 * x * torch.where(x < 0, q, 2.0 - q)


def gelu_tanh32(x):
    return 0.5 * x * (1.0 + torch.tanh(0.7978845608028654 * (x + 0.044715 * x * x * x)))


def _act32(x, act, mutant):
    if act == NONE:
        return x
    if act == SILU:
        return x / (1.0 + torch.exp2(-1.4426950408889634 * x))
    if act == QUICKGELU:
        return x / (1.0 + torch.exp2((-1.702 * 1.4426950408889634) * x))
    if act == GELU:
        return gelu_tanh32(x) if mutant == "tanh_gelu" else gelu_as32(x)
    if act == RELU:
        return x.clamp_min(0.0)
    raise ValueError(act)


def accumulate32(x, w):
    """fp32 accumulation of x w^T (operands exact in fp32) in 16-wide K steps: the product sum of each step is exact (float64), the
    running sum is rounded to fp32 once per step."""
    x, w = x.double(), w.double()
    acc = torch.zeros((x.shape[0], w.shape[0]), dtype=torch.float32)
    for k0 in range(0, x.shape[1], 16):
        acc = (acc.double() + x[:, k0:k0 + 16] @ w[:, k0:k0 + 16].t()).float()
    return acc


MUTANTS = ("early_acc_round", "early_res_round", "scale_after_residual", "m_bias_after_act", "tanh_gelu")


def emulate(a, w, ep, out_dtype=torch.float16, a1=None, mutant=None):
    """The fast-path epilogue of k_gemm_conv in fp32 on the CPU: v = fma(acc, row_scale, col + row); v += m_bias; act; v *= scale;
    v += residual; round to out_dtype.  mutant (one of MUTANTS) injects a known defect."""
    x = torch.cat([a, a1], dim=1) if a1 is not None else a
    n = w.shape[0]
    acc = accumulate32(x, w)
    if mutant == "early_acc_round":
        acc = _r16(acc, torch.float16)
    col = ep.col_bias.float() if ep.col_bias is not None else torch.zeros(n)
    row = ep.row_bias.float()[torch.arange(x.shape[0]) // ep.rows_per_group, :n] if ep.row_bias is not None else torch.zeros(n)
    b = col + row
    rs = ep.row_scale.float()[:, None] if ep.row_scale is not None else torch.ones((1, 1))
    v = (acc.double() * rs.double() + b.double()).float()            # fmaf
    if ep.act == GEGLU:
        vc, gc = geglu_columns(n)
        gate = (acc[:, gc].double() * rs.double() + col[gc].double()).float()
        v = v[:, vc] * gelu_as32(gate)
    else:
        mb = ep.m_bias.float()[:, None] if ep.m_bias is not None else None
        if mb is not None and mutant != "m_bias_after_act":
            v = v + mb
        v = _act32(v, ep.act, mutant)
        if mb is not None and mutant == "m_bias_after_act":
            v = v + mb
    if mutant != "scale_after_residual":
        v = v * ep.scale
    if ep.residual is not None:
        if mutant == "early_res_round":
            v = _r16(v, out_dtype)
        v = v + ep.residual.float()
    if mutant == "scale_after_residual":
        v = v * ep.scale
    return v.to(out_dtype)


# ------------------------------------------------------------------ input generators (seeded, CPU tensors)
def _gen(seed):
    return torch.Generator("cpu").manual_seed(seed)


def _randn(shape, g, scale=1.0):
    return torch.randn(shape, generator=g) * scale


def generic(m, n, k, seed, dtype=torch.float16, act=NONE, m_bias=True, row_scale=False, residual=True, scale=0.5,
            rows_per_group=256):
    """N(0, 1) A, W / sqrt(K), N(0, 1) col / row / m biases, N(0, 1) residual.  Returns (a, w, Epi)."""
    g = _gen(seed)
    a = _randn((m, k), g).to(dtype)
    w = (_randn((n, k), g) / math.sqrt(k)).to(dtype)
    out16 = torch.bfloat16 if dtype == torch.bfloat16 else torch.float16
    ep = Epi(col_bias=_randn((n,), g), row_bias=_randn(((m + rows_per_group - 1) // rows_per_group, n), g), rows_per_group=rows_per_group,
             m_bias=_randn((m,), g) if m_bias else None, row_scale=(0.25 + torch.rand((m,), generator=g) * 2) if row_scale else None,
             residual=_randn((m, n), g).to(out16) if residual else None, scale=scale, act=act)
    return a, w, ep


def cancelling_acc(m, n, k, seed, dtype=torch.float16, act=NONE):
    """Rows of A share a large common vector u (|u_k| ~ 4) plus 2^-6 noise, and col_bias[n] = -(u . w_n) (in float64, of the
    rounded operands): |acc| is typically a hundred or more times |pre|, so an accumulator rounded to the output type before the bias is added
    is off by ~2^-11 |acc|, far above the bound.  No residual, scale 1."""
    g = _gen(seed)
    u = (torch.rand((k,), generator=g) * 2 + 3) * torch.where(torch.rand((k,), generator=g) < 0.5, -1.0, 1.0)
    a = (u[None, :] + _randn((m, k), g, 2.0 ** -6)).to(dtype)
    w = (_randn((n, k), g) / math.sqrt(k)).to(dtype)
    col = -(u.to(dtype).double() @ w.double().t())
    return a, w, Epi(col_bias=col.float(), act=act)


def cancelling_residual(m, n, k, seed, dtype=torch.float16, act=NONE, scale=0.5, out_dtype=torch.float16):
    """Generic A, W and biases, and residual = -round(v) with v = act(pre) * scale in float64: the output is the rounding
    residue of v, so rounding v to the output type before the residual add returns 0 instead."""
    a, w, ep = generic(m, n, k, seed, dtype, act=act, m_bias=False, residual=False, scale=scale)
    v = reference(a, w, ep)["out"]
    return a, w, replace(ep, residual=(-v).to(out_dtype))


def activation_sweep(m, n, k, seed, dtype=torch.float16, act=GELU, lo=-90.0, hi=20.0):
    """pre covers [lo, hi] densely through col_bias (a linear ramp over the N columns, shifted by a fraction of a step per row
    through m_bias), with a small A W (|acc| ~ 0.06): the GELU negative tail, SiLU / quick-GELU where exp(-x) overflows, and
    ReLU's kink at 0.  No residual, scale 1."""
    g = _gen(seed)
    a = _randn((m, k), g, 0.25).to(dtype)
    w = (_randn((n, k), g, 0.25) / math.sqrt(k)).to(dtype)
    step = (hi - lo) / n
    col = torch.linspace(lo, hi - step, n)
    mb = torch.rand((m,), generator=g) * step
    return a, w, Epi(col_bias=col, m_bias=mb, act=act)


GENERATORS = {"generic": generic, "cancelling_acc": cancelling_acc, "cancelling_residual": cancelling_residual,
              "activation_sweep": activation_sweep}


# ------------------------------------------------------------------ tile forms
def forms(geglu_n=None):
    """Every (cg, kps, mt, block_n) the kernel can run: block_n a multiple of 32 up to 256 / mt; for a GEGLU projection with
    N = geglu_n weight rows only its packed tile width fie_geglu_block_n(N) (so mt = 2 only when that is <= 128)."""
    out = []
    for cg in (1, 2):
        for kps in (1, 2):
            for mt in (1, 2):
                bns = [geglu_block_n(geglu_n)] if geglu_n else list(range(32, 256 // mt + 1, 32))
                out += [(cg, kps, mt, bn) for bn in bns if bn <= 256 // mt]
    return out


def form_code(cg, kps, mt):
    """First argument of fie_tune_gemm: cg in bits 0-1, kps in bits 2-3, mt in bits 8-9."""
    return cg | kps << 2 | mt << 8


@contextlib.contextmanager
def forced_form(lib, cg=0, kps=0, mt=0, block_n=0):
    """Force the next GEMMs onto one tile form (0 = the library's choice); always restores the default."""
    lib.fie_tune_gemm(form_code(cg, kps, mt), block_n)
    try:
        yield
    finally:
        lib.fie_tune_gemm(0, 0)
