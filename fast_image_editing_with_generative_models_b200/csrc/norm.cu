// GroupNorm(+SiLU) and LayerNorm on NHWC / token-major fp16 activations (memory-bound).
//   GroupNorm: pass 1 accumulates per-(image, group) sum / sum-of-squares (fp32 per thread, then 2^-20 fixed-point
//   64-bit integer atomics in shared and global memory: integer addition is associative, so the statistics - and with
//   them the whole edit - are bit-reproducible run to run); pass 2 applies (x-mean)*rstd*gamma+beta (+SiLU) and writes
//   fp16.  Pass 1 is skipped when the producing GEMM / convolution already accumulated the statistics in its epilogue.  An optional second source realises the torch.cat([h, skip]) of the UNet up blocks so the
//   concatenated tensor is only ever written once, already normalised.
//   bf16 activations (the bf16 VAE) can exceed the fixed-point range, so their statistics are per-chunk (count, mean, M2) partials
//   merged in a fixed order with Chan's formula instead (k_gn_partials + k_gn_apply<true>): deterministic and free of cancellation.
//   LayerNorm: one warp per row, row kept in registers, two-pass mean / variance in fp32.
// Replaces F.group_norm / F.silu / F.layer_norm in diffusers ResnetBlock2D, Transformer2DModel, BasicTransformerBlock.
#include "fie_common.cuh"
#include <string.h>
#include <type_traits>

namespace fie {

// 2^-20 fixed point in a 64-bit two's-complement integer: exact, order-independent accumulation (|sum| < 2^43).
__device__ __forceinline__ unsigned long long gn_fix(float v) { return (unsigned long long)__float2ll_rn(v * 1048576.0f); }

struct GNArgs {
    const uint4* x0; const uint4* x1; uint4* out;
    int c0v, c1v, cv;          // channel vectors (8 fp16) per source / total
    long long hw; int groups; int cpg;   // channels per group
    const float* gamma; const float* beta; float eps; int silu; unsigned long long* stats;
    int rows_per_cta; int rows_in_flight;
    float* parts;              // bf16 path: (count, mean, M2) per [image][chunk][group]; chunk = blockIdx.x of the row partition
    int chunks;
};

// Row partition of the two-kernel path (depends only on n, hw and the channel vectors): rows_in_flight rows per sweep, enough CTAs
// to cover the machine a few times, at least rows_in_flight * 4 rows each.
static void gn_partition(int n, long long hw, int cv, int* rows_in_flight, int* rows_per_cta, int* chunks) {
    int rif = 512 / cv; if (rif < 1) rif = 1;
    const long long want = (148ll * 4 + n - 1) / n;
    long long rpc = (hw + want - 1) / want;
    if (rpc < (long long)rif * 4) rpc = (long long)rif * 4;
    *rows_in_flight = rif; *rows_per_cta = (int)rpc; *chunks = (int)((hw + rpc - 1) / rpc);
}

// Chan et al.'s pairwise update: (na, ma, qa) <- merge with (nb, mb, qb); q = sum of squared deviations from the mean (M2).
template <typename F>
__device__ __forceinline__ void chan_merge(F& na, F& ma, F& qa, F nb, F mb, F qb) {
    if (nb == F(0)) return;
    const F n = na + nb, d = mb - ma;
    ma += d * (nb / n);
    qa += qb + d * d * (na * nb / n);
    na = n;
}

// bf16 statistics pass: CTA (chunk, image) -> one (count, mean, M2) per group over its rows.  Each thread accumulates, per channel,
// sums of (x - shift) and (x - shift)^2 with shift = the first element it reads (so |mean - shift| is of the order of sigma and the
// fp32 sums do not cancel when |mean| >> sigma), turns them into (count, mean, M2), and the partials are merged per group in a fixed
// order (row slot, then channel): the result depends only on the data, never on scheduling.
__global__ void __launch_bounds__(512) k_gn_partials(GNArgs a) {
    __shared__ float pm[512 * 8], pq[512 * 8];
    __shared__ float pn[512];
    const int img = blockIdx.y;
    const int v = threadIdx.x % a.cv, rsub = threadIdx.x / a.cv;
    float cnt = 0.f;
    if (rsub < a.rows_in_flight) {
        float k[8], s[8], q[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { k[j] = 0.f; s[j] = 0.f; q[j] = 0.f; }
        const long long r0 = (long long)blockIdx.x * a.rows_per_cta;
        const long long r1 = min(r0 + (long long)a.rows_per_cta, a.hw);
        const bool first = v < a.c0v;
        const uint4* src = first ? a.x0 + (long long)img * a.hw * a.c0v + v : a.x1 + (long long)img * a.hw * a.c1v + (v - a.c0v);
        const int stride = first ? a.c0v : a.c1v;
        const long long step = a.rows_in_flight;
        long long r = r0 + rsub;
        if (r < r1) {
            const uint4 u = __ldg(src + r * stride);
            const uint32_t* h = reinterpret_cast<const uint32_t*>(&u);
#pragma unroll
            for (int j = 0; j < 4; ++j) { const float2 f = unpack_h2<true>(h[j]); k[2 * j] = f.x; k[2 * j + 1] = f.y; }
        }
        auto acc = [&](const uint4& u) {
            const uint32_t* h = reinterpret_cast<const uint32_t*>(&u);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 f = unpack_h2<true>(h[j]);
                const float d0 = f.x - k[2 * j], d1 = f.y - k[2 * j + 1];
                s[2 * j] += d0; q[2 * j] = fmaf(d0, d0, q[2 * j]); s[2 * j + 1] += d1; q[2 * j + 1] = fmaf(d1, d1, q[2 * j + 1]);
            }
        };
        for (; r + 3 * step < r1; r += 4 * step) {          // 4 independent 128-bit loads in flight per thread
            uint4 u[4];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) u[kk] = __ldg(src + (r + kk * step) * stride);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) acc(u[kk]);
            cnt += 4.f;
        }
        for (; r < r1; r += step) { acc(__ldg(src + r * stride)); cnt += 1.f; }
        const int base = (rsub * a.cv + v) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float mj = cnt > 0.f ? s[j] / cnt : 0.f;
            pm[base + j] = k[j] + mj;
            pq[base + j] = fmaxf(fmaf(-s[j], mj, q[j]), 0.f);
        }
        if (v == 0) pn[rsub] = cnt;
    }
    __syncthreads();
    for (int g = threadIdx.x; g < a.groups; g += blockDim.x) {
        float n = 0.f, m = 0.f, m2 = 0.f;
        for (int rs = 0; rs < a.rows_in_flight; ++rs) {
            const float nb = pn[rs];
            for (int c = g * a.cpg; c < (g + 1) * a.cpg; ++c) chan_merge(n, m, m2, nb, pm[rs * a.cv * 8 + c], pq[rs * a.cv * 8 + c]);
        }
        float* o = a.parts + (((long long)img * a.chunks + blockIdx.x) * a.groups + g) * 3;
        o[0] = n; o[1] = m; o[2] = m2;
    }
}


__global__ void __launch_bounds__(512) k_gn_stats(GNArgs a) {
    __shared__ unsigned long long gs[64], gq[64];
    const int img = blockIdx.y;
    const int v = threadIdx.x % a.cv, rsub = threadIdx.x / a.cv;
    for (int i = threadIdx.x; i < 2 * a.groups; i += blockDim.x) { if (i < a.groups) gs[i] = 0ull; else gq[i - a.groups] = 0ull; }
    __syncthreads();
    float s[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] = 0.f; q[j] = 0.f; }
    if (rsub < a.rows_in_flight) {
        const long long r0 = (long long)blockIdx.x * a.rows_per_cta;
        const long long r1 = min(r0 + (long long)a.rows_per_cta, a.hw);
        const bool first = v < a.c0v;
        const uint4* src = first ? a.x0 + (long long)img * a.hw * a.c0v + v : a.x1 + (long long)img * a.hw * a.c1v + (v - a.c0v);
        const int stride = first ? a.c0v : a.c1v;
        const long long step = a.rows_in_flight;
        long long r = r0 + rsub;
        for (; r + 3 * step < r1; r += 4 * step) {          // 4 independent 128-bit loads in flight per thread
            uint4 u[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) u[k] = __ldg(src + (r + k * step) * stride);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const __half2* h = reinterpret_cast<const __half2*>(&u[k]);
#pragma unroll
                for (int j = 0; j < 4; ++j) { float2 f = __half22float2(h[j]); s[2 * j] += f.x; q[2 * j] += f.x * f.x; s[2 * j + 1] += f.y; q[2 * j + 1] += f.y * f.y; }
            }
        }
        for (; r < r1; r += step) {
            uint4 u = __ldg(src + r * stride);
            const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
            for (int j = 0; j < 4; ++j) { float2 f = __half22float2(h[j]); s[2 * j] += f.x; q[2 * j] += f.x * f.x; s[2 * j + 1] += f.y; q[2 * j + 1] += f.y * f.y; }
        }
        // channels v*8 .. v*8+7 -> groups
        if (a.cpg >= 8 && (a.cpg % 8) == 0) {
            float ts = 0.f, tq = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) { ts += s[j]; tq += q[j]; }
            int g = (v * 8) / a.cpg;
            atomicAdd(&gs[g], gn_fix(ts)); atomicAdd(&gq[g], gn_fix(tq));
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) { int g = (v * 8 + j) / a.cpg; atomicAdd(&gs[g], gn_fix(s[j])); atomicAdd(&gq[g], gn_fix(q[j])); }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < a.groups; i += blockDim.x) {
        atomicAdd(&a.stats[((long long)img * a.groups + i) * 2], gs[i]);
        atomicAdd(&a.stats[((long long)img * a.groups + i) * 2 + 1], gq[i]);
    }
}

// BF = false: fp16 activations, statistics in the int64 fixed-point sums.  BF = true: bf16 activations, statistics merged here from the
// chunk partials of k_gn_partials (chunk order, fp64) by the first `groups` threads of every CTA.
template <bool BF>
__global__ void __launch_bounds__(512, 2) k_gn_apply(GNArgs a) {
    const int img = blockIdx.y;
    const int v = threadIdx.x % a.cv, rsub = threadIdx.x / a.cv;
    float ga[8], be[8], mu[8], rs[8];
    if constexpr (BF) {
        __shared__ float g_mu[64], g_rs[64];
        for (int g = threadIdx.x; g < a.groups; g += blockDim.x) {
            double n = 0.0, m = 0.0, m2 = 0.0;
            const float* pp = a.parts + (long long)img * a.chunks * a.groups * 3 + g * 3;
            for (int ch = 0; ch < a.chunks; ++ch, pp += a.groups * 3) chan_merge(n, m, m2, (double)pp[0], (double)pp[1], (double)pp[2]);
            g_mu[g] = (float)m;
            g_rs[g] = rsqrtf((float)(m2 / n) + a.eps);
        }
        __syncthreads();
        if (rsub >= a.rows_in_flight) return;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = v * 8 + j, g = c / a.cpg;
            mu[j] = g_mu[g]; rs[j] = g_rs[g];
            ga[j] = __ldg(a.gamma + c); be[j] = __ldg(a.beta + c);
        }
    } else {
    if (rsub >= a.rows_in_flight) return;
    // mean / variance in double from the exact integer sums: E[x^2] - mean^2 cancels badly in fp32 when |mean| >> sigma.
    // A sum of squares that wrapped the 64-bit fixed-point range (group RMS beyond ~1450 over a 1024^2 x 4-channel group) shows up
    // as a negative integer and is turned into NaN -- loud instead of silently wrong.
    const double inv_cnt = 1.0 / ((double)a.hw * (double)a.cpg * 1048576.0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        int c = v * 8 + j, g = c / a.cpg;
        const long long isum = (long long)a.stats[((long long)img * a.groups + g) * 2], isq = (long long)a.stats[((long long)img * a.groups + g) * 2 + 1];
        const double mean = (double)isum * inv_cnt;
        const double var = fmax(fma(-mean, mean, (double)isq * inv_cnt), 0.0);
        mu[j] = (float)mean; rs[j] = isq < 0 ? __int_as_float(0x7fc00000) : rsqrtf((float)var + a.eps);
        ga[j] = __ldg(a.gamma + c); be[j] = __ldg(a.beta + c);
    }
    }
    const long long r0 = (long long)blockIdx.x * a.rows_per_cta;
    const long long r1 = min(r0 + (long long)a.rows_per_cta, a.hw);
    const bool first = v < a.c0v;
    const uint4* src = first ? a.x0 + (long long)img * a.hw * a.c0v + v : a.x1 + (long long)img * a.hw * a.c1v + (v - a.c0v);
    const int stride = first ? a.c0v : a.c1v;
    uint4* dst = a.out + (long long)img * a.hw * a.cv + v;
    // fold the affine transform: y = x * sc + sh
    float sc[8], sh[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j] = rs[j] * ga[j]; sh[j] = fmaf(-mu[j], sc[j], be[j]); }
    auto apply = [&](const uint4& u) -> uint4 {
        uint4 o;
        const uint32_t* h = reinterpret_cast<const uint32_t*>(&u);
        uint32_t* oh = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float2 f = unpack_h2<BF>(h[j]);
            float y0 = fmaf(f.x, sc[2 * j], sh[2 * j]), y1 = fmaf(f.y, sc[2 * j + 1], sh[2 * j + 1]);
            if (a.silu) silu2(y0, y1);
            oh[j] = pack_h2<BF>(y0, y1);
        }
        return o;
    };
    const long long step = a.rows_in_flight;
    long long r = r0 + rsub;
    for (; r + 3 * step < r1; r += 4 * step) {
        uint4 u[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) u[k] = __ldg(src + (r + k * step) * stride);
#pragma unroll
        for (int k = 0; k < 4; ++k) dst[(r + k * step) * a.cv] = apply(u[k]);
    }
    for (; r < r1; r += step) dst[r * a.cv] = apply(__ldg(src + r * stride));
}

// ---- Single-pass GroupNorm for slabs that fit in shared memory (the UNet / ControlNet norms: 10..80 channels per group over
// 1024..16384 pixels = 80 KB .. 1.3 MB per (image, group)) ----
// One thread-block CLUSTER per (image, group): each CTA loads its share of the group's rows into shared memory ONCE (one global read),
// the cluster reduces the mean and then the centred sum of squares over distributed shared memory (two-pass variance: no E[x^2] - mean^2
// cancellation, deterministic, independent of the batch size), and every CTA normalises its rows out of shared memory (one global
// write).  Replaces memset + k_gn_stats + k_gn_apply (two reads, one write, integer atomics) for these shapes, whose channel counts per
// group (10, 20, 30, 40, 60, 80) do not fit the producer-epilogue statistics either.
struct GNSlabArgs {
    const __half2* x0; const __half2* x1; __half2* out;
    int c0h, c1h, ch;          // channel PAIRS per source / total
    int cpgh;                  // channel pairs per group
    long long hw; int rows_per_cta;
    const float* gamma; const float* beta; float eps; int silu;
};

__device__ __forceinline__ float cluster_sum(float v, float* slots /* [32 warps + 8 ranks] */, int nranks, uint32_t rank) {
    // CTA reduction (warp shuffles + shared memory), then every rank reads all ranks' partials over DSMEM in rank order
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0) slots[wid] = v;
    __syncthreads();
    if (wid == 0) {
        float t = lane < nw ? slots[lane] : 0.f;
        t = warp_sum(t);
        if (lane == 0) slots[32 + rank] = t;           // this CTA's partial, published at slot 32 + own rank
    }
    if (nranks == 1) { __syncthreads(); return slots[32 + rank]; }
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    float tot = 0.f;
    for (int r = 0; r < nranks; ++r) {
        uint32_t remote; float pv;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"((uint32_t)__cvta_generic_to_shared(&slots[32 + r])), "r"(r));
        asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(pv) : "r"(remote) : "memory");
        tot += pv;
    }
    // the partial slots are rewritten by the next reduction: nobody may still be reading them
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    return tot;
}

// VEC = channel pairs per memory access (2: 64-bit accesses when the group width is a multiple of 4 channels, else 1: 32-bit).
// Thread (rsub, v) owns vector v of the rows rsub, rsub + step, ...: UNROLL independent loads are in flight per thread (one CTA per SM:
// the latency has to be covered by instruction-level parallelism, not by occupancy).
template <int VEC, bool BF>
__global__ void __launch_bounds__(1024, 1) k_gn_slab(GNSlabArgs a, int nranks) {
    extern __shared__ __align__(16) uint8_t gn_smem[];
    __shared__ float slots[48];
    typedef typename std::conditional<VEC == 2, uint2, uint32_t>::type vec_t;
    constexpr int UNROLL = 8;
    vec_t* slab = reinterpret_cast<vec_t*>(gn_smem);                   // [rows_per_cta][vpr]
    uint32_t rank = 0;
    if (nranks > 1) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int group = blockIdx.x / nranks, img = blockIdx.y;
    const long long r0 = (long long)rank * a.rows_per_cta;
    const int nrows = (int)max(min(r0 + (long long)a.rows_per_cta, a.hw) - r0, 0ll);
    const int vpr = a.cpgh / VEC;                                       // vectors per row of the group
    const int step = blockDim.x / vpr;                                  // rows covered by the CTA per sweep
    const int v = threadIdx.x % vpr, rsub = threadIdx.x / vpr;
    const bool active = rsub < step;
    const int c = group * a.cpgh + v * VEC;                             // first channel pair of this thread's vector
    const bool first = c < a.c0h;                                       // (c0 is a multiple of 8 channels: a vector never straddles the sources)
    const vec_t* src = first ? reinterpret_cast<const vec_t*>(a.x0 + ((long long)img * a.hw + r0) * a.c0h + c)
                             : reinterpret_cast<const vec_t*>(a.x1 + ((long long)img * a.hw + r0) * a.c1h + (c - a.c0h));
    const long long sstride = (first ? a.c0h : a.c1h) / VEC;            // row stride of the source in vectors
    auto sum2 = [](vec_t u, float& s) {
        const uint32_t* h = reinterpret_cast<const uint32_t*>(&u);
#pragma unroll
        for (int j = 0; j < VEC; ++j) { const float2 f = unpack_h2<BF>(h[j]); s += f.x + f.y; }
    };
    // ---- load (one global read) ----
    float s = 0.f;
    if (active) {
        int r = rsub;
        for (; r + (UNROLL - 1) * step < nrows; r += UNROLL * step) {
            vec_t u[UNROLL];
#pragma unroll
            for (int k = 0; k < UNROLL; ++k) u[k] = __ldg(src + (long long)(r + k * step) * sstride);
#pragma unroll
            for (int k = 0; k < UNROLL; ++k) { slab[(r + k * step) * vpr + v] = u[k]; sum2(u[k], s); }
        }
        for (; r < nrows; r += step) { const vec_t u = __ldg(src + (long long)r * sstride); slab[r * vpr + v] = u; sum2(u, s); }
    }
    const float cnt = (float)a.hw * (float)(2 * a.cpgh);
    const float mean = cluster_sum(s, slots, nranks, rank) / cnt;
    float q = 0.f;
    if (active)
        for (int r = rsub; r < nrows; r += step) {                       // own elements only: no barrier needed after the load loop
            const vec_t u = slab[r * vpr + v];
            const uint32_t* h = reinterpret_cast<const uint32_t*>(&u);
#pragma unroll
            for (int j = 0; j < VEC; ++j) { const float2 f = unpack_h2<BF>(h[j]); const float d0 = f.x - mean, d1 = f.y - mean; q = fmaf(d0, d0, fmaf(d1, d1, q)); }
        }
    const float var = cluster_sum(q, slots, nranks, rank) / cnt;
    const float rstd = rsqrtf(var + a.eps);
    // ---- apply from shared memory (one global write): y = x * sc + sh ----
    if (active) {
        float sc[2 * VEC], sh[2 * VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const float2 ga = __ldg(reinterpret_cast<const float2*>(a.gamma) + c + j), be = __ldg(reinterpret_cast<const float2*>(a.beta) + c + j);
            sc[2 * j] = rstd * ga.x; sc[2 * j + 1] = rstd * ga.y;
            sh[2 * j] = fmaf(-mean, sc[2 * j], be.x); sh[2 * j + 1] = fmaf(-mean, sc[2 * j + 1], be.y);
        }
        vec_t* dst = reinterpret_cast<vec_t*>(a.out + ((long long)img * a.hw + r0) * a.ch + c);
        const long long dstride = a.ch / VEC;
        for (int r = rsub; r < nrows; r += step) {
            vec_t u = slab[r * vpr + v];
            uint32_t* h = reinterpret_cast<uint32_t*>(&u);
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                const float2 f = unpack_h2<BF>(h[j]);
                float y0 = fmaf(f.x, sc[2 * j], sh[2 * j]), y1 = fmaf(f.y, sc[2 * j + 1], sh[2 * j + 1]);
                if (a.silu) silu2(y0, y1);
                h[j] = pack_h2<BF>(y0, y1);
            }
            dst[(long long)r * dstride] = u;
        }
    }
}

// ---- LayerNorm: a warp owns a strided set of rows; gamma / beta live in shared memory (one global read per CTA instead of
// four 128-bit loads per data vector and row), and the next row is already in flight while the current one is reduced ----
template <int MAXV>
__global__ void __launch_bounds__(256) k_layernorm(const uint4* __restrict__ x, uint4* __restrict__ out, long long rows, int cv,
                                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps) {
    extern __shared__ float4 gb[];                        // [2 * cv] gamma (two float4 per vector), then [2 * cv] beta
    for (int i = threadIdx.x; i < 2 * cv; i += blockDim.x) {
        gb[i] = __ldg(reinterpret_cast<const float4*>(gamma) + i);
        gb[2 * cv + i] = __ldg(reinterpret_cast<const float4*>(beta) + i);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long wstride = (long long)gridDim.x * (blockDim.x >> 5);
    long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const float c = (float)(cv * 8), inv_c = 1.0f / c;
    uint4 cur[MAXV], nxt[MAXV];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) { const int v = lane + i * 32; cur[i] = (row < rows && v < cv) ? __ldg(x + row * cv + v) : make_uint4(0, 0, 0, 0); }
    for (; row < rows; row += wstride) {
        const long long rn = row + wstride;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) { const int v = lane + i * 32; nxt[i] = (rn < rows && v < cv) ? __ldg(x + rn * cv + v) : make_uint4(0, 0, 0, 0); }
        float vals[MAXV][8];
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            const __half2* h = reinterpret_cast<const __half2*>(&cur[i]);
#pragma unroll
            for (int j = 0; j < 4; ++j) { float2 f = __half22float2(h[j]); vals[i][2 * j] = f.x; vals[i][2 * j + 1] = f.y; sum += f.x + f.y; }
        }
        const float mean = warp_sum(sum) * inv_c;          // lanes beyond cv contributed zeros
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            if (lane + i * 32 < cv) {
#pragma unroll
                for (int j = 0; j < 8; ++j) { float d = vals[i][j] - mean; sq += d * d; }
            }
        }
        const float rstd = rsqrtf(warp_sum(sq) * inv_c + eps);
        uint4* dst = out + row * cv;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            const int v = lane + i * 32;
            if (v < cv) {
                const float4 g0 = gb[2 * v], g1 = gb[2 * v + 1], b0 = gb[2 * cv + 2 * v], b1 = gb[2 * cv + 2 * v + 1];
                const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
                const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                uint4 o; __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    oh[j] = __floats2half2_rn((vals[i][2 * j] - mean) * rstd * g[2 * j] + b[2 * j], (vals[i][2 * j + 1] - mean) * rstd * g[2 * j + 1] + b[2 * j + 1]);
                dst[v] = o;
            }
        }
#pragma unroll
        for (int i = 0; i < MAXV; ++i) cur[i] = nxt[i];
    }
}

// Largest cluster size the single-pass slab kernel may use (0: always the two-kernel path); fie_tune_groupnorm_slab sets it.
// Measured on B200 (scripts/gn_bench.py, SDXL batch-8 shapes): with one CTA the slab kernel wins (82.6 -> 57.4 us on
// [16,1024,1280+640], 90 -> 75 us on [16,4096,640]); clusters of 4-8 CTAs (one CTA per SM, barrier-separated phases) LOSE
// against the streaming two-kernel path (309 -> 644 us on [16,16384,640+320]), so by default only slabs that fit one CTA take it.
static int g_gn_slab_mode = 1;

// Single-pass slab kernel when the (image, group) slab of every image fits the shared memory of <= g_gn_slab_mode CTAs.
// Returns FIE_OK when it launched, an error code, or 1 when the shape does not qualify (the caller takes the two-kernel path).
template <bool BF>
static int gn_try_slab(const void* x0, int c0, const void* x1, int c1, void* out, int n, long long hw, int groups,
                       const float* gamma, const float* beta, float eps, int fuse_silu, cudaStream_t stream) {
    const int c = c0 + c1;
    const int cpg = c / groups;
    const long long slab_bytes = hw * cpg * 2;
    constexpr long long kCtaBytes = 192 * 1024;
    if (!(g_gn_slab_mode && (cpg % 2) == 0 && (c0 % 2) == 0 && (c1 % 2) == 0 && slab_bytes <= 8 * kCtaBytes && hw >= 64 &&
          ((reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta)) & 7) == 0))
        return 1;
    int nranks = 1; while ((long long)nranks * kCtaBytes < slab_bytes) nranks <<= 1;
    if (nranks > g_gn_slab_mode) return 1;
    GNSlabArgs g;
    g.x0 = (const __half2*)x0; g.x1 = (const __half2*)x1; g.out = (__half2*)out;
    g.c0h = c0 / 2; g.c1h = c1 / 2; g.ch = c / 2; g.cpgh = cpg / 2; g.hw = hw;
    g.rows_per_cta = (int)((hw + nranks - 1) / nranks);
    g.gamma = gamma; g.beta = beta; g.eps = eps; g.silu = fuse_silu;
    const size_t smem = (size_t)g.rows_per_cta * g.cpgh * sizeof(__half2);
    static bool attr_dev[kMaxDevices] = {false};
    bool& attr = attr_dev[current_device()];
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(k_gn_slab<1, BF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCtaBytes + 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_gn_slab<2, BF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCtaBytes + 1024);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(k_gn_slab): %s", cudaGetErrorString(e)); return FIE_ERR_CUDA; }
        attr = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(groups * nranks), (unsigned)n); cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = nranks; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    // 64-bit accesses need 4-channel-aligned groups and sources (c0 % 8 == 0 is already required; c1 likewise)
    const bool vec2 = (cpg % 4) == 0;
    cudaError_t e = vec2 ? cudaLaunchKernelEx(&cfg, k_gn_slab<2, BF>, g, nranks) : cudaLaunchKernelEx(&cfg, k_gn_slab<1, BF>, g, nranks);
    if (e != cudaSuccess) { set_error("cudaLaunchKernelEx(k_gn_slab): %s", cudaGetErrorString(e)); cudaGetLastError(); return FIE_ERR_CUDA; }
    return check_launch(BF ? "fie_groupnorm_bf16 (slab)" : "fie_groupnorm_f16 (slab)");
}

static GNArgs gn_args(const void* x0, int c0, const void* x1, int c1, void* out, int n, long long hw, int groups,
                      const float* gamma, const float* beta, float eps, int fuse_silu) {
    GNArgs a;
    memset(&a, 0, sizeof(a));
    const int c = c0 + c1;
    a.x0 = (const uint4*)x0; a.x1 = (const uint4*)x1; a.out = (uint4*)out;
    a.c0v = c0 / 8; a.c1v = c1 / 8; a.cv = c / 8; a.hw = hw; a.groups = groups; a.cpg = c / groups;
    a.gamma = gamma; a.beta = beta; a.eps = eps; a.silu = fuse_silu;
    gn_partition(n, hw, a.cv, &a.rows_in_flight, &a.rows_per_cta, &a.chunks);
    return a;
}

}  // namespace fie
using namespace fie;

extern "C" void fie_tune_groupnorm_slab(int max_cluster) { fie::g_gn_slab_mode = max_cluster < 0 ? 0 : (max_cluster > 8 ? 8 : max_cluster); }

extern "C" int fie_groupnorm_f16(const void* x0, int c0, const void* x1, int c1, void* out, int n, long long hw, int groups,
                                 const float* gamma, const float* beta, float eps, int fuse_silu, void* stats_ws, int stats_ready, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    FIE_REQUIRE(x0 && out && gamma && beta && stats_ws, "fie_groupnorm_f16: null pointer");
    if (!x1) c1 = 0;
    const int c = c0 + c1;
    FIE_REQUIRE(n > 0 && n <= 65535 && hw > 0 && c0 > 0 && (c0 % 8) == 0 && (c1 % 8) == 0, "fie_groupnorm_f16: channels must be multiples of 8");
    FIE_REQUIRE(groups > 0 && groups <= 64 && (c % groups) == 0, "fie_groupnorm_f16: bad groups");
    FIE_REQUIRE(c / 8 <= 512, "fie_groupnorm_f16: too many channels (%d)", c);
    FIE_REQUIRE(!(stats_ready && c1), "fie_groupnorm_f16: producer statistics cannot cover a concatenated second source");
    if (!stats_ready) {
        const int rc = gn_try_slab<false>(x0, c0, x1, c1, out, n, hw, groups, gamma, beta, eps, fuse_silu, stream);
        if (rc <= 0) return rc;
    }
    GNArgs a = gn_args(x0, c0, x1, c1, out, n, hw, groups, gamma, beta, eps, fuse_silu);
    a.stats = (unsigned long long*)stats_ws;
    const int threads = ((a.cv * a.rows_in_flight + 31) / 32) * 32;
    dim3 grid((unsigned)a.chunks, n);
    if (!stats_ready) {
        cudaError_t e = cudaMemsetAsync(stats_ws, 0, sizeof(unsigned long long) * 2 * groups * n, stream);
        if (e != cudaSuccess) { set_error("fie_groupnorm_f16: memset: %s", cudaGetErrorString(e)); return FIE_ERR_CUDA; }
        k_gn_stats<<<grid, threads, 0, stream>>>(a);
    }
    k_gn_apply<false><<<grid, threads, 0, stream>>>(a);
    return check_launch("fie_groupnorm_f16");
}

extern "C" size_t fie_groupnorm_bf16_workspace_bytes(int n, long long hw, int c, int groups) {
    if (n <= 0 || hw <= 0 || c < 8 || groups <= 0) return 0;
    int rif, rpc, chunks;
    gn_partition(n, hw, c / 8, &rif, &rpc, &chunks);
    return (((size_t)n * chunks * groups * 3 * sizeof(float)) + 255) / 256 * 256;
}

extern "C" int fie_groupnorm_bf16(const void* x0, int c0, const void* x1, int c1, void* out, int n, long long hw, int groups,
                                  const float* gamma, const float* beta, float eps, int fuse_silu, void* workspace, size_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    FIE_REQUIRE(x0 && out && gamma && beta && workspace, "fie_groupnorm_bf16: null pointer");
    if (!x1) c1 = 0;
    const int c = c0 + c1;
    FIE_REQUIRE(n > 0 && n <= 65535 && hw > 0 && c0 > 0 && (c0 % 8) == 0 && (c1 % 8) == 0, "fie_groupnorm_bf16: channels must be multiples of 8");
    FIE_REQUIRE(groups > 0 && groups <= 64 && (c % groups) == 0, "fie_groupnorm_bf16: bad groups");
    FIE_REQUIRE(c / 8 <= 512, "fie_groupnorm_bf16: too many channels (%d)", c);
    FIE_REQUIRE(workspace_bytes >= fie_groupnorm_bf16_workspace_bytes(n, hw, c, groups), "fie_groupnorm_bf16: workspace too small");
    FIE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "fie_groupnorm_bf16: workspace must be 256-byte aligned");
    const int rc = gn_try_slab<true>(x0, c0, x1, c1, out, n, hw, groups, gamma, beta, eps, fuse_silu, stream);
    if (rc <= 0) return rc;
    GNArgs a = gn_args(x0, c0, x1, c1, out, n, hw, groups, gamma, beta, eps, fuse_silu);
    a.parts = (float*)workspace;
    const int threads = ((a.cv * a.rows_in_flight + 31) / 32) * 32;
    dim3 grid((unsigned)a.chunks, n);
    k_gn_partials<<<grid, threads, 0, stream>>>(a);
    k_gn_apply<true><<<grid, threads, 0, stream>>>(a);
    return check_launch("fie_groupnorm_bf16");
}

extern "C" int fie_layernorm_f16(const void* x, void* out, long long rows, int c, const float* gamma, const float* beta, float eps, void* stream) {
    FIE_REQUIRE(x && out && gamma && beta && rows > 0 && c > 0 && (c % 8) == 0 && c <= 2048, "fie_layernorm_f16: c must be a multiple of 8, <= 2048");
    const int cv = c / 8;
    FIE_REQUIRE(((reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta)) & 15) == 0, "fie_layernorm_f16: gamma / beta must be 16-byte aligned");
    long long blocks = (rows + 7) / 8;
    const long long cap = 148ll * 2;                      // two resident CTAs per SM (128 registers x 256 threads); each warp strides over its rows
    if (blocks > cap) blocks = cap;
    const unsigned grid = (unsigned)blocks;
    const size_t smem = (size_t)4 * cv * sizeof(float4);
    if (cv <= 64) k_layernorm<2><<<grid, 256, smem, (cudaStream_t)stream>>>((const uint4*)x, (uint4*)out, rows, cv, gamma, beta, eps);
    else if (cv <= 160) k_layernorm<5><<<grid, 256, smem, (cudaStream_t)stream>>>((const uint4*)x, (uint4*)out, rows, cv, gamma, beta, eps);
    else k_layernorm<8><<<grid, 256, smem, (cudaStream_t)stream>>>((const uint4*)x, (uint4*)out, rows, cv, gamma, beta, eps);
    return check_launch("fie_layernorm_f16");
}
