// Memory-bound helper kernels: pre/post-processing, residual adds, nearest upsample, sinusoidal embedding,
// row softmax, VAE posterior sample + add_noise, fused CFG + LCMScheduler.step.
// All use 128-bit accesses where the layout allows and grid-stride loops sized to the SM count.
#include "fie_common.cuh"

namespace fie {

static inline int grid_for(long long work_items, int block) {
    long long b = (work_items + block - 1) / block;
    long long cap = 148ll * 8;
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

// ---- VaeImageProcessor.preprocess: u8 HWC -> fp16 NHWC (x/127.5 - 1 computed as 2*(x/255)-1 in fp32) ----
__global__ void __launch_bounds__(256) k_pre(const uint8_t* __restrict__ in, __half* __restrict__ out, long long npix, int c_out, int normalize) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (long long)gridDim.x * blockDim.x) {
        float v[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) { float x = (float)in[i * 3 + c] / 255.0f; v[c] = normalize ? 2.0f * x - 1.0f : x; }
        __half* o = out + i * c_out;
        if (c_out == 4) {
            __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], 0.0f);
            uint2 u; u.x = *reinterpret_cast<uint32_t*>(&a); u.y = *reinterpret_cast<uint32_t*>(&b);
            *reinterpret_cast<uint2*>(o) = u;
        } else {
            for (int c = 0; c < c_out; ++c) o[c] = __float2half_rn(c < 3 ? v[c] : 0.0f);
        }
    }
}

// Same conversion into the zero-padded 8-channel layout [n][h+2][w+8][8] the tensor-core conv_in reads (real pixel (y, x) at
// (y+1, x+1)); one thread writes one 16-byte padded pixel, borders and channels 3..7 as zeros.
__global__ void __launch_bounds__(256) k_pre_pad8(const uint8_t* __restrict__ in, uint4* __restrict__ out, int n, int h, int w, int normalize) {
    const int wp = w + 8, hp = h + 2;
    const long long total = (long long)n * hp * wp;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int xx = (int)(i % wp) - 1; const long long t = i / wp; const int yy = (int)(t % hp) - 1; const long long img = t / hp;
        uint4 u = make_uint4(0, 0, 0, 0);
        if (xx >= 0 && xx < w && yy >= 0 && yy < h) {
            const uint8_t* px = in + ((img * h + yy) * w + xx) * 3;
            float v[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) { float x = (float)px[c] / 255.0f; v[c] = normalize ? 2.0f * x - 1.0f : x; }
            __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], 0.0f);
            u.x = *reinterpret_cast<uint32_t*>(&a); u.y = *reinterpret_cast<uint32_t*>(&b);
        }
        out[i] = u;
    }
}

// fp16 [n,h,w,4] (latents) -> the same zero-padded 8-channel layout [n][h+2][w+8][8] (channels 4..7 and borders zero)
__global__ void __launch_bounds__(256) k_pad8_f16(const uint2* __restrict__ in, uint4* __restrict__ out, int n, int h, int w) {
    const int wp = w + 8, hp = h + 2;
    const long long total = (long long)n * hp * wp;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int xx = (int)(i % wp) - 1; const long long t = i / wp; const int yy = (int)(t % hp) - 1; const long long img = t / hp;
        uint4 u = make_uint4(0, 0, 0, 0);
        if (xx >= 0 && xx < w && yy >= 0 && yy < h) { const uint2 v = __ldg(in + (img * h + yy) * w + xx); u.x = v.x; u.y = v.y; }
        out[i] = u;
    }
}

// ---- VaeImageProcessor.postprocess: clamp(x/2+0.5,0,1) -> round(x*255) -> u8 ----
__global__ void __launch_bounds__(256) k_post(const __half* __restrict__ in, int ld, uint8_t* __restrict__ out, long long npix) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            // the reference computes x/2+0.5 and the clamp in the model dtype (fp16), then *255 and round in fp32
            __half hx = __float2half_rn(__half2float(in[i * ld + c]) / 2.0f);
            hx = __float2half_rn(__half2float(hx) + 0.5f);
            float x = fminf(fmaxf(__half2float(hx), 0.0f), 1.0f);
            out[i * 3 + c] = (uint8_t)rintf(x * 255.0f);
        }
    }
}

__global__ void __launch_bounds__(256) k_add(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ o, long long n8) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
        uint4 x = __ldg(a + i), y = __ldg(b + i), r;
        const __half2* xh = reinterpret_cast<const __half2*>(&x); const __half2* yh = reinterpret_cast<const __half2*>(&y);
        __half2* rh = reinterpret_cast<__half2*>(&r);
#pragma unroll
        for (int j = 0; j < 4; ++j) { float2 fa = __half22float2(xh[j]), fb = __half22float2(yh[j]); rh[j] = __floats2half2_rn(fa.x + fb.x, fa.y + fb.y); }
        o[i] = r;
    }
}

__global__ void __launch_bounds__(256) k_silu(const uint4* __restrict__ a, uint4* __restrict__ o, long long n8) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
        uint4 x = __ldg(a + i), r;
        const __half2* xh = reinterpret_cast<const __half2*>(&x); __half2* rh = reinterpret_cast<__half2*>(&r);
#pragma unroll
        for (int j = 0; j < 4; ++j) { float2 f = __half22float2(xh[j]); rh[j] = __floats2half2_rn(silu_f(f.x), silu_f(f.y)); }
        o[i] = r;
    }
}

__global__ void __launch_bounds__(256) k_up2x(const uint4* __restrict__ x, uint4* __restrict__ o, int n, int h, int w, int c8) {
    const long long total = (long long)n * 2 * h * 2 * w * c8;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        int cv = (int)(i % c8); long long t = i / c8;
        int ox = (int)(t % (2 * w)); t /= (2 * w);
        int oy = (int)(t % (2 * h)); int img = (int)(t / (2 * h));
        o[i] = __ldg(x + (((long long)img * h + (oy >> 1)) * w + (ox >> 1)) * c8 + cv);
    }
}

struct SinCosArgs { float vals[64]; };
__global__ void k_sincos(SinCosArgs a, int count, int dim, __half* __restrict__ out) {
    const int half = dim / 2;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count * half; i += gridDim.x * blockDim.x) {
        int r = i / half, j = i % half;
        float freq = expf(-logf(10000.0f) * (float)j / (float)half);
        float arg = a.vals[r] * freq;
        out[r * dim + j] = __float2half_rn(cosf(arg));
        out[r * dim + half + j] = __float2half_rn(sinf(arg));
    }
}

// one CTA per row; cols up to 64K.  T = float (raw scores, scaled here) or __half (scores already scaled by the GEMM epilogue).
template <typename T> struct Vec4;
template <> struct Vec4<float> { static __device__ __forceinline__ float4 ld(const float* p) { return *reinterpret_cast<const float4*>(p); } };
template <> struct Vec4<__half> {
    static __device__ __forceinline__ float4 ld(const __half* p) {
        const uint2 u = *reinterpret_cast<const uint2*>(p);
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
        return make_float4(a.x, a.y, b.x, b.y);
    }
};
__device__ __forceinline__ float ex2_f(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }

// Single-pass form for rows of at most 256 x 4 x NV columns: the row lives in registers (NV independent vector loads in flight
// per thread), one block reduction for the max and one for the sum.
// OBF: the probabilities are stored as bf16 instead of fp16 (the bf16 VAE).
template <typename T, int NV, bool OBF = false>
__global__ void __launch_bounds__(256) k_softmax_rows_reg(const T* __restrict__ s, long long ld_in, uint16_t* __restrict__ p, long long ld_out, int cols, float scale) {
    __shared__ float red[8];
    __shared__ float bc;
    const T* row = s + (long long)blockIdx.x * ld_in;
    uint16_t* orow = p + (long long)blockIdx.x * ld_out;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    float4 v[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const int i = (k * 256 + tid) * 4;
        v[k] = i + 4 <= cols ? Vec4<T>::ld(row + i) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < NV; ++k) mx = fmaxf(mx, fmaxf(fmaxf(v[k].x, v[k].y), fmaxf(v[k].z, v[k].w)));
    mx = warp_max(mx);
    if (lane == 0) red[wid] = mx;
    __syncthreads();
    if (tid == 0) { float m = red[0]; for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]); bc = m; }
    __syncthreads();
    mx = bc;
    const float sl2 = scale * 1.4426950408889634f, off = -mx * sl2;
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        v[k].x = exp2f(fmaf(v[k].x, sl2, off)); v[k].y = exp2f(fmaf(v[k].y, sl2, off)); v[k].z = exp2f(fmaf(v[k].z, sl2, off)); v[k].w = exp2f(fmaf(v[k].w, sl2, off));
        sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
    sum = warp_sum(sum);
    __syncthreads();
    if (lane == 0) red[wid] = sum;
    __syncthreads();
    if (tid == 0) { float t = 0; for (int i = 0; i < 8; ++i) t += red[i]; bc = 1.0f / t; }
    __syncthreads();
    const float inv = bc;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const int i = (k * 256 + tid) * 4;
        if (i + 4 <= cols) {
            uint2 u; u.x = pack_h2<OBF>(v[k].x * inv, v[k].y * inv); u.y = pack_h2<OBF>(v[k].z * inv, v[k].w * inv);
            *reinterpret_cast<uint2*>(orow + i) = u;
        }
    }
}

// exp-only form for fp16 scores (rows of at most 256 x 4 x NV columns): writes P' = exp2((s - rowmax) * scale * log2 e) <= 1 as fp16 and
// 1 / sum(P') per row; the normalisation is applied exactly, in fp32, by the epilogue of the P V GEMM (fie_epilogue.row_scale).
// The row stays in registers as packed fp16 (the maximum of fp16 values is exact in fp16), so the kernel needs half the registers
// of the normalising form, one block reduction before the stores instead of two, and keeps four to five CTAs per SM in flight.
template <int NV>
__global__ void __launch_bounds__(256, 4) k_softmax_rows_exp(const __half* __restrict__ s, long long ld_in, __half* __restrict__ p, long long ld_out,
                                                             float* __restrict__ inv_sum, int cols, float scale) {
    __shared__ float red[8];
    __shared__ float bc;
    const __half* row = s + (long long)blockIdx.x * ld_in;
    __half* orow = p + (long long)blockIdx.x * ld_out;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint2 v[NV];
    const __half2 ninf = __float2half2_rn(-INFINITY);
    __half2 m2 = ninf;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const int i = (k * 256 + tid) * 4;
        if (i + 4 <= cols) v[k] = *reinterpret_cast<const uint2*>(row + i);
        else { v[k].x = *reinterpret_cast<const uint32_t*>(&ninf); v[k].y = v[k].x; }
    }
#pragma unroll
    for (int k = 0; k < NV; ++k) m2 = __hmax2(m2, __hmax2(*reinterpret_cast<const __half2*>(&v[k].x), *reinterpret_cast<const __half2*>(&v[k].y)));
    float mx = warp_max(fmaxf(__low2float(m2), __high2float(m2)));
    if (lane == 0) red[wid] = mx;
    __syncthreads();
    if (tid == 0) { float m = red[0]; for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]); bc = m; }
    __syncthreads();
    mx = bc;
    const float sl2 = scale * 1.4426950408889634f, off = -mx * sl2;
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const int i = (k * 256 + tid) * 4;
        if (i + 4 <= cols) {
            const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v[k].x)), b = __half22float2(*reinterpret_cast<const __half2*>(&v[k].y));
            const __half2 pa = __floats2half2_rn(ex2_f(fmaf(a.x, sl2, off)), ex2_f(fmaf(a.y, sl2, off)));
            const __half2 pb = __floats2half2_rn(ex2_f(fmaf(b.x, sl2, off)), ex2_f(fmaf(b.y, sl2, off)));
            const float2 ra = __half22float2(pa), rb = __half22float2(pb);        // the row sum is the sum of what the GEMM will read
            sum += (ra.x + ra.y) + (rb.x + rb.y);
            uint2 u; u.x = *reinterpret_cast<const uint32_t*>(&pa); u.y = *reinterpret_cast<const uint32_t*>(&pb);
            *reinterpret_cast<uint2*>(orow + i) = u;
        }
    }
    sum = warp_sum(sum);
    __syncthreads();
    if (lane == 0) red[wid] = sum;
    __syncthreads();
    if (tid == 0) { float t = 0; for (int i = 0; i < 8; ++i) t += red[i]; inv_sum[blockIdx.x] = 1.0f / t; }
}

template <typename T, bool OBF = false>
__global__ void __launch_bounds__(256) k_softmax_rows(const T* __restrict__ s, long long ld_in, uint16_t* __restrict__ p, long long ld_out, int cols, float scale) {
    __shared__ float red[8];
    __shared__ float bc;
    const T* row = s + (long long)blockIdx.x * ld_in;
    uint16_t* orow = p + (long long)blockIdx.x * ld_out;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    float mx = -INFINITY;
    for (int i = tid * 4; i < cols; i += 1024) {
        if (i + 4 <= cols) { float4 v = Vec4<T>::ld(row + i); mx = fmaxf(mx, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w))); }
        else for (int j = i; j < cols; ++j) mx = fmaxf(mx, to_f(row[j]));
    }
    mx = warp_max(mx);
    if (lane == 0) red[wid] = mx;
    __syncthreads();
    if (tid == 0) { float m = red[0]; for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]); bc = m; }
    __syncthreads();
    mx = bc;
    const float sl2 = scale * 1.4426950408889634f;
    float sum = 0.f;
    for (int i = tid * 4; i < cols; i += 1024) {
        if (i + 4 <= cols) { float4 v = Vec4<T>::ld(row + i); sum += exp2f((v.x - mx) * sl2) + exp2f((v.y - mx) * sl2) + exp2f((v.z - mx) * sl2) + exp2f((v.w - mx) * sl2); }
        else for (int j = i; j < cols; ++j) sum += exp2f((to_f(row[j]) - mx) * sl2);
    }
    sum = warp_sum(sum);
    __syncthreads();
    if (lane == 0) red[wid] = sum;
    __syncthreads();
    if (tid == 0) { float t = 0; for (int i = 0; i < 8; ++i) t += red[i]; bc = 1.0f / t; }
    __syncthreads();
    const float inv = bc;
    for (int i = tid * 4; i < cols; i += 1024) {
        if (i + 4 <= cols) {
            float4 v = Vec4<T>::ld(row + i);
            uint2 u;
            u.x = pack_h2<OBF>(exp2f((v.x - mx) * sl2) * inv, exp2f((v.y - mx) * sl2) * inv);
            u.y = pack_h2<OBF>(exp2f((v.z - mx) * sl2) * inv, exp2f((v.w - mx) * sl2) * inv);
            *reinterpret_cast<uint2*>(orow + i) = u;
        } else for (int j = i; j < cols; ++j) orow[j] = f_to_h<OBF>(exp2f((to_f(row[j]) - mx) * sl2) * inv);
    }
}

// z0 = (mean + exp(0.5*clamp(logvar,-30,20))*xi)*scaling ; x = sqrt_a*z0 + sqrt_1ma*noise.  The latent STATE is kept in fp32
// across the scheduler steps (out32); out16 is the fp16 copy the UNet / ControlNet read.  (diffusers keeps the state in the model
// dtype; the fp32 state removes one fp16 rounding of |x| <= 16, i.e. up to 4e-3, per step from the final latents.)
__global__ void __launch_bounds__(256) k_vae_sample(const __half* __restrict__ mom, int ld_m, const __half* __restrict__ xi, const __half* __restrict__ noise,
                                                    float* __restrict__ out32, __half* __restrict__ out16, long long npx, float scaling, float sa, float s1) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npx * 4; i += (long long)gridDim.x * blockDim.x) {
        long long px = i >> 2; int c = (int)(i & 3);
        const float mean = __half2float(mom[px * ld_m + c]);
        const float logvar = fminf(fmaxf(__half2float(mom[px * ld_m + 4 + c]), -30.0f), 20.0f);
        const float z = (mean + expf(0.5f * logvar) * __half2float(xi[i])) * scaling;
        const float r = sa * z + s1 * __half2float(noise[i]);
        out32[i] = r; out16[i] = __float2half_rn(r);
    }
}

__global__ void __launch_bounds__(256) k_cfg_lcm(const __half* __restrict__ eu, const __half* __restrict__ ec, int ld_e, const float* __restrict__ x,
                                                 const __half* __restrict__ noise, float* __restrict__ out32, __half* __restrict__ out16, long long npx, float g,
                                                 float sa, float s1, float c_skip, float c_out, float sap, float s1p, int last) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npx * 4; i += (long long)gridDim.x * blockDim.x) {
        long long px = i >> 2; int c = (int)(i & 3);
        float u = __half2float(eu[px * ld_e + c]), cc = __half2float(ec[px * ld_e + c]);
        float eps = u + g * (cc - u);
        float xv = x[i];
        float x0 = (xv - s1 * eps) / sa;
        float den = c_out * x0 + c_skip * xv;
        float r = last ? den : sap * den + s1p * __half2float(noise[i]);
        out32[i] = r; out16[i] = __float2half_rn(r);
    }
}

// token + position embedding: one 16-byte vector per thread
__global__ void __launch_bounds__(256) k_embed_tokens(const int* __restrict__ ids, const uint4* __restrict__ tok, const uint4* __restrict__ pos, uint4* __restrict__ out,
                                                      long long rows, int seq_len, int cv, int vocab) {
    const long long total = rows * cv;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / cv; const int v = (int)(i - r * cv);
        int id = ids[r]; id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
        const uint4 a = __ldg(tok + (long long)id * cv + v), b = __ldg(pos + (long long)(r % seq_len) * cv + v);
        uint4 o; const __half2* ah = reinterpret_cast<const __half2*>(&a); const __half2* bh = reinterpret_cast<const __half2*>(&b); __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
        for (int j = 0; j < 4; ++j) { const float2 fa = __half22float2(ah[j]), fb = __half22float2(bh[j]); oh[j] = __floats2half2_rn(fa.x + fb.x, fa.y + fb.y); }
        out[i] = o;
    }
}

}  // namespace fie
using namespace fie;

extern "C" int fie_embed_tokens_f16(const int* ids, const void* tok, const void* pos, void* out, long long rows, int seq_len, int c, int vocab, void* stream) {
    FIE_REQUIRE(ids && tok && pos && out && rows > 0 && seq_len > 0 && c > 0 && (c % 8) == 0 && vocab > 0, "fie_embed_tokens_f16: bad args");
    k_embed_tokens<<<grid_for(rows * (c / 8), 256), 256, 0, (cudaStream_t)stream>>>(ids, (const uint4*)tok, (const uint4*)pos, (uint4*)out, rows, seq_len, c / 8, vocab);
    return check_launch("fie_embed_tokens_f16");
}

extern "C" int fie_preprocess_u8_to_f16(const void* img, void* out, int n, int h, int w, int c_out, int normalize, void* stream) {
    FIE_REQUIRE(img && out && n > 0 && h > 0 && w > 0 && c_out >= 3, "fie_preprocess_u8_to_f16: bad args");
    long long npix = (long long)n * h * w;
    k_pre<<<grid_for(npix, 256), 256, 0, (cudaStream_t)stream>>>((const uint8_t*)img, (__half*)out, npix, c_out, normalize);
    return check_launch("fie_preprocess_u8_to_f16");
}
extern "C" int fie_preprocess_u8_to_f16_pad8(const void* img, void* out, int n, int h, int w, int normalize, void* stream) {
    FIE_REQUIRE(img && out && n > 0 && h > 0 && w > 0, "fie_preprocess_u8_to_f16_pad8: bad args");
    const long long total = (long long)n * (h + 2) * (w + 8);
    k_pre_pad8<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const uint8_t*)img, (uint4*)out, n, h, w, normalize);
    return check_launch("fie_preprocess_u8_to_f16_pad8");
}
extern "C" int fie_pad8_f16(const void* x4, void* out, int n, int h, int w, void* stream) {
    FIE_REQUIRE(x4 && out && n > 0 && h > 0 && w > 0, "fie_pad8_f16: bad args");
    const long long total = (long long)n * (h + 2) * (w + 8);
    k_pad8_f16<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const uint2*)x4, (uint4*)out, n, h, w);
    return check_launch("fie_pad8_f16");
}
extern "C" int fie_postprocess_f16_to_u8(const void* x, int ld, void* out, int n, int h, int w, void* stream) {
    FIE_REQUIRE(x && out && n > 0 && h > 0 && w > 0 && ld >= 3, "fie_postprocess_f16_to_u8: bad args");
    long long npix = (long long)n * h * w;
    k_post<<<grid_for(npix, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)x, ld, (uint8_t*)out, npix);
    return check_launch("fie_postprocess_f16_to_u8");
}
extern "C" int fie_add_f16(const void* a, const void* b, void* out, long long count, void* stream) {
    FIE_REQUIRE(a && b && out && count > 0 && (count % 8) == 0, "fie_add_f16: count must be a positive multiple of 8");
    k_add<<<grid_for(count / 8, 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)a, (const uint4*)b, (uint4*)out, count / 8);
    return check_launch("fie_add_f16");
}
extern "C" int fie_silu_f16(const void* a, void* out, long long count, void* stream) {
    FIE_REQUIRE(a && out && count > 0 && (count % 8) == 0, "fie_silu_f16: count must be a positive multiple of 8");
    k_silu<<<grid_for(count / 8, 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)a, (uint4*)out, count / 8);
    return check_launch("fie_silu_f16");
}
extern "C" int fie_upsample2x_f16(const void* x, void* out, int n, int h, int w, int c, void* stream) {
    FIE_REQUIRE(x && out && n > 0 && h > 0 && w > 0 && c > 0 && (c % 8) == 0, "fie_upsample2x_f16: c must be a multiple of 8");
    long long total = (long long)n * 4 * h * w * (c / 8);
    k_up2x<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)x, (uint4*)out, n, h, w, c / 8);
    return check_launch("fie_upsample2x_f16");
}
extern "C" int fie_sincos_embedding(const float* host_vals, int count, int dim, void* out, void* stream) {
    FIE_REQUIRE(host_vals && out && count > 0 && count <= 64 && dim > 0 && (dim % 2) == 0, "fie_sincos_embedding: bad args");
    SinCosArgs a; for (int i = 0; i < 64; ++i) a.vals[i] = i < count ? host_vals[i] : 0.f;
    k_sincos<<<ceil_div((long long)count * dim / 2, 128), 128, 0, (cudaStream_t)stream>>>(a, count, dim, (__half*)out);
    return check_launch("fie_sincos_embedding");
}
extern "C" int fie_softmax_rows_f32_to_f16(const void* s, long long ld_in, void* p, long long ld_out, long long rows, int cols, float scale, void* stream) {
    FIE_REQUIRE(s && p && rows > 0 && rows < (1ll << 31) && cols > 0 && (ld_in % 4) == 0 && (ld_out % 4) == 0, "fie_softmax_rows: bad args");
    if ((cols % 4) == 0 && cols <= 16384) k_softmax_rows_reg<float, 16><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>((const float*)s, ld_in, (uint16_t*)p, ld_out, cols, scale);
    else k_softmax_rows<float><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>((const float*)s, ld_in, (uint16_t*)p, ld_out, cols, scale);
    return check_launch("fie_softmax_rows_f32_to_f16");
}
extern "C" int fie_softmax_rows_f32_to_bf16(const void* s, long long ld_in, void* p, long long ld_out, long long rows, int cols, float scale, void* stream) {
    FIE_REQUIRE(s && p && rows > 0 && rows < (1ll << 31) && cols > 0 && (ld_in % 4) == 0 && (ld_out % 4) == 0, "fie_softmax_rows_f32_to_bf16: bad args");
    if ((cols % 4) == 0 && cols <= 16384) k_softmax_rows_reg<float, 16, true><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>((const float*)s, ld_in, (uint16_t*)p, ld_out, cols, scale);
    else k_softmax_rows<float, true><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>((const float*)s, ld_in, (uint16_t*)p, ld_out, cols, scale);
    return check_launch("fie_softmax_rows_f32_to_bf16");
}
extern "C" int fie_softmax_rows_f16(const void* s, long long ld_in, void* p, long long ld_out, long long rows, int cols, float scale, void* stream) {
    FIE_REQUIRE(s && p && rows > 0 && rows < (1ll << 31) && cols > 0 && (ld_in % 4) == 0 && (ld_out % 4) == 0, "fie_softmax_rows_f16: bad args");
    if ((cols % 4) == 0 && cols <= 16384) k_softmax_rows_reg<__half, 16><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>((const __half*)s, ld_in, (uint16_t*)p, ld_out, cols, scale);
    else k_softmax_rows<__half><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>((const __half*)s, ld_in, (uint16_t*)p, ld_out, cols, scale);
    return check_launch("fie_softmax_rows_f16");
}
extern "C" int fie_softmax_rows_exp_f16(const void* s, long long ld_in, void* p, long long ld_out, float* inv_sum, long long rows, int cols, float scale, void* stream) {
    FIE_REQUIRE(s && p && inv_sum && rows > 0 && rows < (1ll << 31) && cols > 0 && (cols % 4) == 0 && cols <= 16384 && (ld_in % 4) == 0 && (ld_out % 4) == 0,
                "fie_softmax_rows_exp_f16: bad args (cols must be a multiple of 4, <= 16384)");
    k_softmax_rows_exp<16><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>((const __half*)s, ld_in, (__half*)p, ld_out, inv_sum, cols, scale);
    return check_launch("fie_softmax_rows_exp_f16");
}
extern "C" int fie_vae_sample_add_noise(const void* moments, int ld_m, const void* xi, const void* noise, float* x_out_f32, void* x_out_f16,
                                        long long count_px, float scaling, float sqrt_a, float sqrt_1ma, void* stream) {
    FIE_REQUIRE(moments && xi && noise && x_out_f32 && x_out_f16 && count_px > 0 && ld_m >= 8, "fie_vae_sample_add_noise: bad args");
    k_vae_sample<<<grid_for(count_px * 4, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)moments, ld_m, (const __half*)xi, (const __half*)noise,
                                                                                x_out_f32, (__half*)x_out_f16, count_px, scaling, sqrt_a, sqrt_1ma);
    return check_launch("fie_vae_sample_add_noise");
}
extern "C" int fie_cfg_lcm_step(const void* eps_u, const void* eps_c, int ld_e, const float* x_f32, const void* noise, float* x_out_f32, void* x_out_f16,
                                long long count_px, float guidance, float sqrt_a, float sqrt_1ma, float c_skip, float c_out,
                                float sqrt_a_prev, float sqrt_1ma_prev, int last, void* stream) {
    FIE_REQUIRE(eps_u && eps_c && x_f32 && x_out_f32 && x_out_f16 && count_px > 0 && ld_e >= 4 && (last || noise), "fie_cfg_lcm_step: bad args");
    k_cfg_lcm<<<grid_for(count_px * 4, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)eps_u, (const __half*)eps_c, ld_e, x_f32,
                                                                              (const __half*)noise, x_out_f32, (__half*)x_out_f16, count_px, guidance, sqrt_a, sqrt_1ma,
                                                                              c_skip, c_out, sqrt_a_prev, sqrt_1ma_prev, last);
    return check_launch("fie_cfg_lcm_step");
}
