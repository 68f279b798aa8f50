// Shared helpers for the fie_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/fie_b200.h"

namespace fie {

// Thread-local last-error string (the only mutable global state of the library).
void set_error(const char* fmt, ...);
int  check_launch(const char* what);   // returns FIE_OK or FIE_ERR_CUDA after cudaGetLastError()

#define FIE_REQUIRE(cond, ...)                                   \
    do { if (!(cond)) { fie::set_error(__VA_ARGS__); return FIE_ERR_INVALID; } } while (0)

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// Per-device one-time state: cudaFuncSetAttribute and the SM count belong to a DEVICE, and one process may drive several GPUs
// (FastEditor(device="cuda:1")), so every "done once" flag in this library is an array indexed by the current device.
constexpr int kMaxDevices = 64;
int current_device();        // cudaGetDevice, clamped to [0, kMaxDevices)
int device_sm_count();       // multiprocessor count of the current device (cached per device)

// x * sigmoid(x) with two MUFU ops (ex2, rcp); the IEEE division it replaces cost ~10 extra issue slots per element.
__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.0f + __expf(-x)); }
// Exact (erf) GELU, 0.5 x (1 + erf(x / sqrt 2)), with erfc from Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7, far below
// the fp16 rounding of the result): q = erfc(|z|) = poly5(t) exp(-z^2), t = 1 / (1 + p |z|).  Written on the erfc side
// so the negative tail (1 + erf = q) has no cancellation.  ~14 issue slots and 2 MUFU instead of erff's ~30 + branch.
__device__ __forceinline__ float gelu_erf_f(float x) {
    const float z = fabsf(x) * 0.70710678118654752440f;
    float t;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
    float pl = fmaf(1.061405429f, t, -1.453152027f);
    pl = fmaf(pl, t, 1.421413741f);
    pl = fmaf(pl, t, -0.284496736f);
    pl = fmaf(pl, t, 0.254829592f);
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * z * z));
    const float q = pl * t * e;
    return 0.5f * x * (x < 0.0f ? q : 2.0f - q);
}

// Packed fp32x2 arithmetic (FFMA2 / FADD2 / FMUL2, new on sm_100): one issue slot for two elements.  Measured on B200
// (scripts/micro/mufu_mix.cu): a packed instruction occupies the FMA pipe for 2 cycles -- the FLOP rate of scalar fp32 -- so the
// gain is in issue slots, which MUFU-heavy element-wise code (8 clk per MUFU warp instruction) is short of.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f32x2 pack2u(uint32_t lo, uint32_t hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 ffma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.ftz.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f32x2 fmul2(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 fadd2(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 fadd2_rm(f32x2 a, f32x2 b) { f32x2 r; asm("add.rm.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 fsub2(f32x2 a, f32x2 b) { f32x2 r; asm("sub.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }

// SiLU of a pair: y / (1 + 2^(-y log2 e)) with ONE MUFU per element (ex2); the reciprocal is a bit-trick seed (12 % error)
// refined by three packed Newton steps r <- r (2 - d r) (error^2 each: 1.4e-2, 2e-4, 4e-8) instead of a second MUFU.
__device__ __forceinline__ void silu2(float& y0, float& y1) {
    float e0, e1;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fminf(-1.4426950408889634f * y0, 126.0f)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fminf(-1.4426950408889634f * y1, 126.0f)));
    const f32x2 d = fadd2(pack2(e0, e1), pack2(1.0f, 1.0f));
    float d0, d1;
    unpack2(d, d0, d1);
    f32x2 r = pack2(__int_as_float(0x7EF311C7 - __float_as_int(d0)), __int_as_float(0x7EF311C7 - __float_as_int(d1)));
    const f32x2 two = pack2(2.0f, 2.0f), nd = pack2(-d0, -d1);
    r = fmul2(r, ffma2(nd, r, two));
    r = fmul2(r, ffma2(nd, r, two));
    r = fmul2(r, ffma2(nd, r, two));
    unpack2(fmul2(pack2(y0, y1), r), y0, y1);
}

__device__ __forceinline__ float quick_gelu_f(float x) { return __fdividef(x, 1.0f + __expf(-1.702f * x)); }

// Two 16-bit floats in one 32-bit word: fp16 (BF = false) or bf16 (BF = true), round to nearest even.
template <bool BF> __device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    if constexpr (BF) { const __nv_bfloat162 h = __floats2bfloat162_rn(a, b); return *reinterpret_cast<const uint32_t*>(&h); }
    else { const __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<const uint32_t*>(&h); }
}
template <bool BF> __device__ __forceinline__ float2 unpack_h2(uint32_t u) {
    if constexpr (BF) return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
    else return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
template <bool BF> __device__ __forceinline__ float h_to_f(uint16_t u) {
    if constexpr (BF) return __bfloat162float(__ushort_as_bfloat16(u));
    else return __half2float(__ushort_as_half(u));
}
template <bool BF> __device__ __forceinline__ uint16_t f_to_h(float v) {
    if constexpr (BF) return __bfloat16_as_ushort(__float2bfloat16_rn(v));
    else return __half_as_ushort(__float2half_rn(v));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace fie
