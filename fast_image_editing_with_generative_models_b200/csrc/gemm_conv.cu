// Persistent, warp-specialised tcgen05 GEMM / implicit-GEMM 3x3 convolution for sm_100a.
//
//   D[M, N] = epilogue( A[M, K] * B[N, K]^T )     fp16 (or bf16) operands, fp32 accumulators in TMEM
//
// Replaces F.linear / F.conv2d (cuBLASLt / cuDNN) in every diffusers module on the reference's edit path
// (UNet2DConditionModel, ControlNetModel, AutoencoderKL; reference call site src/pipeline.py:261-272).
//
// Data movement: TMA (cp.async.bulk.tensor) with 128-byte swizzle into a ring of shared-memory stages.
//   GEMM mode:  A tile = 2-D box {64 k, 128 rows} of the row-major activation matrix.
//   CONV mode:  A tile = 4-D box {64 ch, bw, bh, bn} (bw*bh*bn = 128 output pixels) of the NHWC activation,
//               shifted by the filter tap; zero padding comes from TMA out-of-bounds fill, so im2col is never
//               materialised.  Stride-2 convolutions read four parity-split views of the input.
//   CONV im2col mode (widths the box cannot tile: not a multiple of 128 and not a divisor of 128): A tile = 128 consecutive
//               output pixels in raster order (n, y, x), wrapping across rows and images, loaded by TMA im2col mode with the
//               tap as the im2col offset; the map's bounding box gives the zero padding.
//   B tile = 2-D box {64 k, block_n rows} of the packed weight matrix [N][K].
// Math: one elected thread issues tcgen05.mma (M=128, N=block_n, K=16) into a double-buffered TMEM accumulator.
// Epilogue: 4 warps read TMEM (tcgen05.ld 32x32b), fuse bias / time-embedding broadcast / SiLU / GEGLU /
//           scale / residual, and store fp16 (or bf16 / fp32) rows.
//
// Warp roles (384 threads): w0-7 epilogue, w8 TMA producer, w9 MMA issuer, w10 TMEM allocator, w11 idle.
#include "tc_common.cuh"

#ifndef FIE_GEMM_SETMAXNREG
#define FIE_GEMM_SETMAXNREG 1
#endif

namespace fie {

// Warp roles.  The epilogue warps get the LOW warp ids: the SM's warp scheduler favours higher ids among ready warps, and the
// single-thread TMA producer / MMA issuer must never wait behind eight ALU-busy epilogue warps.
#ifndef FIE_GEMM_ROLES_HIGH
#define FIE_GEMM_ROLES_HIGH 1
#endif
constexpr int W_EPI0 = FIE_GEMM_ROLES_HIGH ? 0 : 4;        // first of the 8 epilogue warps
constexpr int W_PROD = FIE_GEMM_ROLES_HIGH ? 8 : 0, W_MMA = W_PROD + 1, W_ALLOC = W_PROD + 2;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;   // 16 KiB
constexpr int MAX_STAGES = 12;
constexpr int SMEM_BUDGET = 192 * 1024;      // pipeline stages
// Halo mode (stride-1 3x3 convolutions whose output rows are >= 128 pixels wide): per 64-channel chunk the producer loads
// the three input rows h-1, h, h+1 of a 128-pixel output segment ONCE as 130-pixel slabs (130 x 128 B, padded to 17 KiB so
// every slab base stays 1024-byte aligned) and the 9 filter taps read them through shifted shared-memory descriptors
// (start address + kw * 128 B): a third of the L2 -> SM traffic of loading 9 shifted A tiles.
constexpr int HALO_PX = BLOCK_M + 2;
constexpr int HALO_SLAB_BYTES = 17 * 1024;
constexpr int HALO_SET_BYTES = 3 * HALO_SLAB_BYTES;
constexpr int HALO_A_BYTES = 2 * HALO_SET_BYTES;     // double-buffered slab sets; the B ring takes the rest of SMEM_BUDGET
constexpr int EPI_STAGE_BYTES = 8 * 1024;      // per-epilogue-warp bias staging (8 slots x 32 fp32)

struct GemmParams {
    CUtensorMap a_maps[4];
    CUtensorMap b_map;
    int mode;         // 0 = GEMM, 1 = CONV (one shifted A tile per tap), 2 = CONV halo (A slabs shared by the 9 taps),
                      // 3 = CONV im2col (one raster run of 128 output pixels per tap; a_maps are im2col maps)
    int num_kb;       // K blocks of 64
    int kb_per_tap;   // CONV: cin/64
    int kb_split;     // GEMM: k-blocks taken from a_maps[0]; the rest from a_maps[1]
    int8_t tap_map[12], tap_dh[12], tap_dw[12];
    int OH, OW;
    int up2, up_a, up_b;   // up2 = 1: rows are INPUT pixels (n,h,w) of a nearest-2x-upsampled conv phase; output pixel (2h+a, 2w+b)
    long long M;
    int N;            // accumulator columns (B rows)
    int block_n;
    int cg;           // 1 or 2 CTAs per tile
    int kps;          // 64-wide K blocks per pipeline stage (1 or 2)
    int mt;           // 128-row M sub-tiles per CTA (1 or 2)
    int dbg;          // debug/tuning: 1 = skip TMA loads, 2 = skip MMA issue, 4 = skip epilogue math/stores
    long long* trace; // debug: per-CTA wait-time accounting [grid][8] (see fie_gemm_trace), or NULL
    int num_m_blocks, num_n_blocks;   // m blocks of 128*cg rows
    int num_stages;
    int tmem_cols;
    // epilogue
    void* D;
    long long ldd;
    int n_store;      // number of valid output columns
    const float* col_bias;
    const float* row_bias;
    long long rows_per_group;
    long long ld_row_bias;
    const float* m_bias;
    const __half* residual;         // in the output's 16-bit type (fp16, or bf16 when out_bf16)
    long long ld_res;
    float scale;
    int act;
    int out_f32;
    int out_bf16;                   // 16-bit output (and residual) is bf16 (kernel variant OBF = 1)
    int ab_bf16;                    // A and B are bf16 (instruction-descriptor operand formats and TMA maps)
    unsigned long long* gn_stats;   // optional GroupNorm statistics of the output [images][groups][2], 2^-20 fixed point
    int gn_cpg, gn_groups;          // channels per group (divides 32), groups
    long long gn_rows;              // rows per image
    // LayerNorm folding (see fie_epilogue): statistics of the output rows / normalisation of the input rows
    unsigned long long* ln_out;     // [M][2] (sum, sum of squares of the fp16 outputs; 2^-20 fixed point) or NULL
    const unsigned long long* ln_in;  // [M][2] statistics of the A rows, or NULL
    float ln_eps;
    double ln_inv;                  // 1 / (2^20 * length of the normalised A rows)
    const float* row_scale;         // [M] optional per-row scale of the accumulator (exclusive with ln_in)
};

// Output row of accumulator row m (identity, or the strided scatter of one phase of the fused nearest-2x upsample).
__device__ __forceinline__ long long out_row(const GemmParams& p, long long m) {
    if (!p.up2) return m;
    const int pix = p.OH * p.OW;
    const int n = (int)(m / pix), rem = (int)(m - (long long)n * pix);
    const int h = rem / p.OW, w = rem - h * p.OW;
    return ((long long)n * 2 * p.OH + 2 * h + p.up_a) * (2 * p.OW) + 2 * w + p.up_b;
}

template <bool OBF>
__device__ __forceinline__ void store_chunk(const GemmParams& p, long long m, int n0, const float (&v)[32]) {
    // stores v[0..31] to output row m, columns n0..n0+31 (masked by n_store)
    if (p.out_f32) {
        float* d = reinterpret_cast<float*>(p.D) + out_row(p, m) * p.ldd + n0;
        if (n0 + 32 <= p.n_store && (p.ldd & 3) == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) reinterpret_cast<float4*>(d)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        } else {
            for (int i = 0; i < 32; ++i) if (n0 + i < p.n_store) d[i] = v[i];
        }
    } else {
        uint16_t* d = reinterpret_cast<uint16_t*>(p.D) + out_row(p, m) * p.ldd + n0;
        if (n0 + 32 <= p.n_store && (p.ldd & 7) == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                uint4 u;
                u.x = pack_h2<OBF>(v[8 * i], v[8 * i + 1]); u.y = pack_h2<OBF>(v[8 * i + 2], v[8 * i + 3]);
                u.z = pack_h2<OBF>(v[8 * i + 4], v[8 * i + 5]); u.w = pack_h2<OBF>(v[8 * i + 6], v[8 * i + 7]);
                reinterpret_cast<uint4*>(d)[i] = u;
            }
        } else {
            for (int i = 0; i < 32; ++i) if (n0 + i < p.n_store) d[i] = f_to_h<OBF>(v[i]);
        }
    }
}

// GroupNorm statistics of one 32 x 32 output chunk (thread = row, v = its 32 fp32 outputs): per-thread partial sums of the NG
// = 32 / cpg groups the chunk covers and a halving butterfly over the 32 rows of the warp (NG + log2 stages shuffles instead of
// 5 per value).  The warp keeps adding into per-chunk-slot registers across its tiles and only flushes them with 64-bit
// fixed-point atomics when the (image, tile column) changes: integer accumulation keeps the result independent of the order in
// which warps finish, and the number of atomics independent of the problem size.
template <int NG>
__device__ __forceinline__ void gn_stats_chunk(const float (&v)[32], bool row_ok, int lane, float& s_out, float& q_out) {
    constexpr int CPG = 32 / NG;
    float s[NG], q[NG];
#pragma unroll
    for (int j = 0; j < NG; ++j) {
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int i = 0; i < CPG; ++i) { const float x = row_ok ? v[j * CPG + i] : 0.f; a += x; b = fmaf(x, x, b); }
        s[j] = a; q[j] = b;
    }
    int n = NG, off = 16;
#pragma unroll
    for (; n > 1; n >>= 1, off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int j = 0; j < n / 2; ++j) {
            const float ss = upper ? s[j] : s[j + n / 2], sq = upper ? q[j] : q[j + n / 2];
            const float rs = __shfl_xor_sync(0xffffffffu, ss, off), rq = __shfl_xor_sync(0xffffffffu, sq, off);
            s[j] = (upper ? s[j + n / 2] : s[j]) + rs; q[j] = (upper ? q[j + n / 2] : q[j]) + rq;
        }
    }
#pragma unroll
    for (; off > 0; off >>= 1) { s[0] += __shfl_xor_sync(0xffffffffu, s[0], off); q[0] += __shfl_xor_sync(0xffffffffu, q[0], off); }
    s_out += s[0]; q_out += q[0];       // every lane of a group class now holds that group's total over the warp's 32 rows
}

// Out-of-line generic epilogue for one 32-column chunk of one accumulator row per thread: partial chunks at the N edge,
// fp32 output, unaligned leading dimensions.  Rare; kept out of the hot loop on purpose.
template <bool OBF>
__device__ __noinline__ void epi_slow_chunk(const GemmParams& p, uint32_t taddr, uint32_t taddr_gate, int ngate, long long m, bool row_ok,
                                            int nacc, int nout, float mb, const float* rb) {
    uint32_t r[32];
    float v[32];
    tmem_ld_32x32(taddr, r);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]) + mb;
    if (nout >= p.n_store && p.act != FIE_ACT_GEGLU) return;                      // chunk entirely beyond the stored columns
    if (p.col_bias) for (int i = 0; i < 32; ++i) if (nacc + i < p.N) v[i] += __ldg(p.col_bias + nacc + i);
    if (rb) for (int i = 0; i < 32; ++i) if (nacc + i < p.N) v[i] += __ldg(rb + nacc + i);
    if (p.act == FIE_ACT_GEGLU) {
        tmem_ld_32x32(taddr_gate, r);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            float gate = __uint_as_float(r[i]);
            if (p.col_bias && ngate + i < p.N) gate += __ldg(p.col_bias + ngate + i);
            v[i] *= gelu_erf_f(gate);
        }
    } else if (p.act == FIE_ACT_SILU) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = silu_f(v[i]);
    } else if (p.act == FIE_ACT_GELU) {
        for (int i = 0; i < 32; ++i) v[i] = gelu_erf_f(v[i]);
    } else if (p.act == FIE_ACT_QUICKGELU) {
        for (int i = 0; i < 32; ++i) v[i] = quick_gelu_f(v[i]);
    } else if (p.act == FIE_ACT_RELU) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.0f);
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] *= p.scale;
    if (row_ok && nout < p.n_store) {
        if (p.residual) {
            const uint16_t* rp = reinterpret_cast<const uint16_t*>(p.residual) + m * p.ld_res + nout;
            for (int i = 0; i < 32; ++i) if (nout + i < p.n_store) v[i] += h_to_f<OBF>(rp[i]);
        }
        if (!p.out_f32 && !p.up2 && nout == 0 && p.n_store <= 4 && p.ldd == 4 && (reinterpret_cast<uintptr_t>(p.D) & 7) == 0) {
            // <= 4 output channels in a 4-wide row (decoder conv_out: 3 of 4): one 8-byte store per pixel; the spare lane gets 0
            uint2 u; u.x = pack_h2<OBF>(v[0], p.n_store > 1 ? v[1] : 0.f); u.y = pack_h2<OBF>(p.n_store > 2 ? v[2] : 0.f, p.n_store > 3 ? v[3] : 0.f);
            *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(p.D) + m * 4) = u;
        } else store_chunk<OBF>(p, m, nout, v);
    }
}

// acc * rstd + bias: rstd is the epilogue thread's LayerNorm row scale, exactly 1 (-> acc + bias) when no LayerNorm is folded
#define FIE_LN_LIN(acc, b) fmaf(__uint_as_float(acc), ln_rstd, __uint_as_float(b))

// Debug accounting: clock cycles a role spends blocked on a barrier (only when a trace buffer is installed).
#define FIE_TIMED(acc, stmt) do { if (p.trace) { const long long t0_ = clock64(); stmt; (acc) += clock64() - t0_; } else { stmt; } } while (0)

// CG = 1: one CTA per tile (M = 128).  CG = 2: CTA pair (cta_group::2), tile M = 256, each CTA loads half of B.
// KPS = 64-wide K blocks per pipeline stage (per producer/consumer mbarrier handshake).
// MT = 128-row M sub-tiles per CTA that share every B tile (narrow-N problems: twice the MMA work per handshake).
// OBF = 1: 16-bit outputs and residuals are bf16 (the bf16 VAE); the operand format is a run-time field of the instruction descriptor.
template <int CG, int KPS, int MT, int GEGLU, int OBF>
__global__ void __launch_bounds__(384, 1) k_gemm_conv(const __grid_constant__ GemmParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // dynamic smem base is only guaranteed 16-byte aligned by the ABI; round up to 1024 for the 128B swizzle
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], tmem_full[2], tmem_empty[2], a_full[2], a_empty[2];
    __shared__ uint32_t tmem_base_slot;

    const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;
    uint8_t* epi_smem = smem + SMEM_BUDGET;        // [8 epilogue warps][8 bias slots][32 fp32]
    const int block_n = p.block_n;
    const int b_rows = block_n / CG;                                   // B rows held by this CTA
    const int b_sub_bytes = b_rows * BLOCK_K * 2;
    const int stage_bytes = KPS * (MT * A_STAGE_BYTES + b_sub_bytes);
    const int num_sb = (p.num_kb + KPS - 1) / KPS;                     // pipeline iterations per tile
    const int num_stages = p.num_stages;
    const int num_tiles = p.num_m_blocks * p.num_n_blocks;            // m blocks of 128*CG rows
    const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    const int first_tile = blockIdx.x / CG, tile_step = gridDim.x / CG;

    // Programmatic dependent launch: the whole (persistent, <= 1 CTA per SM) grid is resident from the start, so the next kernel
    // in the stream may begin launching right away; its CTAs land on SMs as this grid's CTAs retire and run their own prologue
    // (barrier init, TMEM allocation, descriptor prefetch) under this kernel's tail.  No-ops without the launch attribute.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (warp == W_PROD && lane == 0) {
        for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.a_maps[i]);
        tma_prefetch_desc(&p.b_map);
    }
    if (warp == W_MMA && lane == 0) {
        for (int s = 0; s < num_stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], 8 * CG); mbar_init(&a_full[b], 1); mbar_init(&a_empty[b], 1); }
        mbar_fence_init();
    }
    if (warp == W_ALLOC) { if (CG == 2) tmem_alloc_2sm(&tmem_base_slot, (uint32_t)p.tmem_cols); else tmem_alloc(&tmem_base_slot, (uint32_t)p.tmem_cols); }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    asm volatile("griddepcontrol.wait;" ::: "memory");      // everything below may read what the previous kernel wrote (and overwrite what it read)
    const uint32_t tmem_base = tmem_base_slot;
    long long tr_wait = 0, tr_wait2 = 0;
    const long long tr_start = p.trace ? clock64() : 0;

    // Register re-partition (384 threads x 168 at launch): the producer / MMA / allocator warpgroup keeps 56 registers per
    // thread, the two epilogue warpgroups get 224 so that the epilogue math has the ILP to stay off the critical path.
    if (warp >= W_PROD && warp < W_PROD + 4) {
#if FIE_GEMM_SETMAXNREG
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
#endif
    if (warp == W_PROD) {
        // ===================== TMA producer =====================
        const bool prod_lane = elect_one_sync();
        if (prod_lane && p.mode == 2) {
            // ---- halo convolution: slab sets (per 64-channel chunk) + a ring of per-tap B tiles ----
            int stage = 0; uint32_t phase = 0; int ab = 0; uint32_t aph = 0;
            uint8_t* smem_b = smem + HALO_A_BYTES;
            const int num_cc = p.kb_per_tap, tps = p.kps;
            for (int tile = first_tile; tile < num_tiles; tile += tile_step) {
                const int m_blk = tile / p.num_n_blocks, n_blk = tile % p.num_n_blocks;
                const long long m0 = ((long long)m_blk * CG + cta_rank) * BLOCK_M;
                const long long pix = (long long)p.OH * p.OW;
                const int n0i = (int)(m0 / pix), rem = (int)(m0 % pix), h0 = rem / p.OW, w0 = rem % p.OW;
                for (int cc = 0; cc < num_cc; ++cc) {
                    FIE_TIMED(tr_wait, mbar_wait(&a_empty[ab], aph ^ 1));
                    if (CG == 1 || leader) mbar_arrive_expect_tx(&a_full[ab], (uint32_t)(CG * 3 * HALO_PX * BLOCK_K * 2));
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        uint8_t* dst = smem + ab * HALO_SET_BYTES + r * HALO_SLAB_BYTES;
                        if (CG == 1) tma_load_4d(&p.a_maps[0], &a_full[ab], dst, cc * BLOCK_K, w0 - 1, h0 + r - 1, n0i);
                        else tma_load_4d_2sm(&p.a_maps[0], &a_full[ab], dst, cc * BLOCK_K, w0 - 1, h0 + r - 1, n0i);
                    }
                    ab ^= 1; if (ab == 0) aph ^= 1;
                    for (int tap0 = 0; tap0 < 9; tap0 += tps) {          // one ring stage = tps taps (a whole kernel row when it fits)
                        FIE_TIMED(tr_wait, mbar_wait(&empty_bar[stage], phase ^ 1));
                        if (CG == 1 || leader) mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(CG * tps * b_sub_bytes));
                        for (int t = 0; t < tps; ++t) {
                            const int kcol = ((tap0 + t) * num_cc + cc) * BLOCK_K;
                            uint8_t* dst = smem_b + (size_t)(stage * tps + t) * b_sub_bytes;
                            if (CG == 1) tma_load_2d(&p.b_map, &full_bar[stage], dst, kcol, n_blk * block_n);
                            else tma_load_2d_2sm(&p.b_map, &full_bar[stage], dst, kcol, n_blk * block_n + (int)cta_rank * b_rows);
                        }
                        if (++stage == num_stages) { stage = 0; phase ^= 1; }
                    }
                }
            }
            if (p.trace) { p.trace[blockIdx.x * 8 + 0] = tr_wait; p.trace[blockIdx.x * 8 + 1] = clock64() - tr_start; }
        } else if (prod_lane) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = first_tile; tile < num_tiles; tile += tile_step) {
                const int m_blk = tile / p.num_n_blocks, n_blk = tile % p.num_n_blocks;
                long long m0[MT]; int n0i[MT], h0[MT], w0[MT];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    m0[mt] = (((long long)m_blk * MT + mt) * CG + cta_rank) * BLOCK_M;
                    n0i[mt] = 0; h0[mt] = 0; w0[mt] = 0;
                    if (p.mode == 1 || p.mode == 3) {
                        const long long pix = (long long)p.OH * p.OW;
                        n0i[mt] = (int)(m0[mt] / pix);
                        const int rem = (int)(m0[mt] % pix);
                        h0[mt] = rem / p.OW; w0[mt] = rem % p.OW;
                    }
                }
                for (int sb = 0; sb < num_sb; ++sb) {
                    FIE_TIMED(tr_wait, mbar_wait(&empty_bar[stage], phase ^ 1));
                    uint8_t* sbase = smem + (size_t)stage * stage_bytes;
                    if (p.dbg & 1) {
                        if (CG == 1 || leader) mbar_arrive(&full_bar[stage]);
                    } else {
                        // the leader's barrier collects the bytes of both CTAs of a pair
                        if (CG == 1 || leader) mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(CG * stage_bytes));
#pragma unroll
                        for (int sub = 0; sub < KPS; ++sub) {
                            const int kb = sb * KPS + sub;                       // kb >= num_kb: coordinates fall outside -> zero fill
                            uint8_t* sbm = sbase + KPS * MT * A_STAGE_BYTES + sub * b_sub_bytes;
#pragma unroll
                            for (int mt = 0; mt < MT; ++mt) {
                                uint8_t* sa = sbase + (sub * MT + mt) * A_STAGE_BYTES;
                                if (p.mode == 0) {
                                    const bool first = kb < p.kb_split;
                                    const CUtensorMap* am = first ? &p.a_maps[0] : &p.a_maps[1];
                                    const int kc = (first ? kb : kb - p.kb_split) * BLOCK_K;
                                    if (CG == 1) tma_load_2d(am, &full_bar[stage], sa, kc, (int)m0[mt]); else tma_load_2d_2sm(am, &full_bar[stage], sa, kc, (int)m0[mt]);
                                } else if (p.mode == 3) {
                                    // the run starts at input pixel (x - 1, y - 1) of the bounding box; tap (dh, dw) reads it at (+dw+1, +dh+1).
                                    // Past the last K block the B tile is zero-filled, so any in-bounds A block adds nothing (tap 0, chunk 0).
                                    const bool pad_kb = kb >= p.num_kb;
                                    const int tap = pad_kb ? 0 : kb / p.kb_per_tap;
                                    const int c0 = pad_kb ? 0 : (kb - tap * p.kb_per_tap) * BLOCK_K;
                                    const CUtensorMap* am = &p.a_maps[p.tap_map[tap]];
                                    const uint16_t ow = (uint16_t)(p.tap_dw[tap] + 1), oh = (uint16_t)(p.tap_dh[tap] + 1);
                                    if (CG == 1) tma_load_im2col_4d(am, &full_bar[stage], sa, c0, w0[mt] - 1, h0[mt] - 1, n0i[mt], ow, oh);
                                    else tma_load_im2col_4d_2sm(am, &full_bar[stage], sa, c0, w0[mt] - 1, h0[mt] - 1, n0i[mt], ow, oh);
                                } else {
                                    int tap = kb / p.kb_per_tap;
                                    int c0 = (kb - tap * p.kb_per_tap) * BLOCK_K;
                                    if (kb >= p.num_kb) { tap = 0; c0 = p.kb_per_tap * BLOCK_K; }
                                    const CUtensorMap* am = &p.a_maps[p.tap_map[tap]];
                                    if (CG == 1) tma_load_4d(am, &full_bar[stage], sa, c0, w0[mt] + p.tap_dw[tap], h0[mt] + p.tap_dh[tap], n0i[mt]);
                                    else tma_load_4d_2sm(am, &full_bar[stage], sa, c0, w0[mt] + p.tap_dw[tap], h0[mt] + p.tap_dh[tap], n0i[mt]);
                                }
                            }
                            if (CG == 1) tma_load_2d(&p.b_map, &full_bar[stage], sbm, kb * BLOCK_K, n_blk * block_n);
                            else tma_load_2d_2sm(&p.b_map, &full_bar[stage], sbm, kb * BLOCK_K, n_blk * block_n + (int)cta_rank * b_rows);
                        }
                    }
                    if (++stage == num_stages) { stage = 0; phase ^= 1; }
                }
            }
            if (p.trace) { p.trace[blockIdx.x * 8 + 0] = tr_wait; p.trace[blockIdx.x * 8 + 1] = clock64() - tr_start; }
        }
    } else if (warp == W_MMA && leader) {
        // ===================== MMA issuer (leader CTA of the pair) =====================
        const uint32_t idesc = umma_idesc_f16(BLOCK_M * CG, block_n) | (p.ab_bf16 ? kIdescABBF16 : 0u);
        int stage = 0; uint32_t phase = 0; int it = 0;
        if (p.mode == 2) {
            int ab = 0; uint32_t aph = 0;
            const int num_cc = p.kb_per_tap, tps = p.kps;
            const uint32_t smem_a = smem_u32(smem), smem_b = smem_a + HALO_A_BYTES;
            for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++it) {
                const int buf = it & 1; const uint32_t acc_phase = (it >> 1) & 1;
                FIE_TIMED(tr_wait2, if (CG == 2) mbar_wait_cluster(&tmem_empty[buf], acc_phase ^ 1); else mbar_wait(&tmem_empty[buf], acc_phase ^ 1));
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(buf * block_n);
                for (int cc = 0; cc < num_cc; ++cc) {
                    FIE_TIMED(tr_wait, mbar_wait(&a_full[ab], aph));
                    for (int tap0 = 0; tap0 < 9; tap0 += tps) {
                        FIE_TIMED(tr_wait, mbar_wait(&full_bar[stage], phase));
                        tc_fence_after();
                        if (elect_one_sync()) {
                            for (int t = 0; t < tps; ++t) {
                                const int tap = tap0 + t, kh = tap / 3, kw = tap - 3 * kh;
                                const uint64_t bdesc = umma_desc_sw128(smem_b + (uint32_t)((stage * tps + t) * b_sub_bytes));
                                // rows kw .. kw+127 of slab kh: start address shifted by kw pixels (128 B each).  Measured on B200: the 128B
                                // swizzle is a function of the shared-memory ADDRESS bits, so the descriptor's base-offset field stays 0.
                                const uint64_t adesc = umma_desc_sw128(smem_a + (uint32_t)(ab * HALO_SET_BYTES + kh * HALO_SLAB_BYTES + kw * 128));
#pragma unroll
                                for (int k = 0; k < BLOCK_K / 16; ++k) {
                                    if (p.dbg & 2) continue;
                                    const uint32_t acc = (cc | tap | k) ? 1u : 0u;
                                    if (CG == 2) umma_f16_2sm(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, acc);
                                    else umma_f16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, acc);
                                }
                            }
                            const bool last_tap = tap0 + tps == 9, last = last_tap && cc == num_cc - 1;
                            if (CG == 2) { umma_commit_2sm(&empty_bar[stage]); if (last_tap) umma_commit_2sm(&a_empty[ab]); if (last) umma_commit_2sm(&tmem_full[buf]); }
                            else { umma_commit(&empty_bar[stage]); if (last_tap) umma_commit(&a_empty[ab]); if (last) umma_commit(&tmem_full[buf]); }
                        }
                        __syncwarp();
                        if (++stage == num_stages) { stage = 0; phase ^= 1; }
                    }
                    ab ^= 1; if (ab == 0) aph ^= 1;
                }
            }
        } else
        for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++it) {
            const int buf = it & 1; const uint32_t acc_phase = (it >> 1) & 1;
            FIE_TIMED(tr_wait2, if (CG == 2) mbar_wait_cluster(&tmem_empty[buf], acc_phase ^ 1); else mbar_wait(&tmem_empty[buf], acc_phase ^ 1));
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + (uint32_t)(buf * MT * block_n);
            for (int sb = 0; sb < num_sb; ++sb) {
                FIE_TIMED(tr_wait, mbar_wait(&full_bar[stage], phase));
                if (p.trace && it == 0 && sb == 0 && lane == 0) p.trace[blockIdx.x * 8 + 7] = clock64() - tr_start;   // prologue + first TMA round trip
                tc_fence_after();
                if (elect_one_sync()) {
                    const uint32_t sbase = smem_u32(smem + (size_t)stage * stage_bytes);
#pragma unroll
                    for (int sub = 0; sub < KPS; ++sub) {
                        const uint64_t bdesc = umma_desc_sw128(sbase + KPS * MT * A_STAGE_BYTES + sub * b_sub_bytes);
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) {
                            const uint64_t adesc = umma_desc_sw128(sbase + (sub * MT + mt) * A_STAGE_BYTES);
#pragma unroll
                            for (int k = 0; k < BLOCK_K / 16; ++k) {
                                if (p.dbg & 2) continue;
                                const uint32_t acc = (sb | sub | k) ? 1u : 0u;
                                if (CG == 2) umma_f16_2sm(tmem_d + mt * block_n, adesc + 2 * k, bdesc + 2 * k, idesc, acc);
                                else umma_f16(tmem_d + mt * block_n, adesc + 2 * k, bdesc + 2 * k, idesc, acc);
                            }
                        }
                    }
                    if (CG == 2) { umma_commit_2sm(&empty_bar[stage]); if (sb == num_sb - 1) umma_commit_2sm(&tmem_full[buf]); }
                    else { umma_commit(&empty_bar[stage]); if (sb == num_sb - 1) umma_commit(&tmem_full[buf]); }
                }
                __syncwarp();
                if (++stage == num_stages) { stage = 0; phase ^= 1; }
            }
        }
        if (p.trace && elect_one_sync()) { p.trace[blockIdx.x * 8 + 2] = tr_wait; p.trace[blockIdx.x * 8 + 3] = tr_wait2; p.trace[blockIdx.x * 8 + 4] = clock64() - tr_start; }
    }
    } else {
#if FIE_GEMM_SETMAXNREG
        asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
#endif
        // ===================== Epilogue: 8 warps, two per TMEM lane quadrant (even / odd 32-column chunks) =====================
        // Work item = one 32-row x 32-column chunk of the accumulator; a thread owns one row of it (TMEM lane == row), i.e.
        // 64 contiguous bytes of fp16 output, moved as two 256-bit global accesses (full 32-byte sectors, no shared-memory
        // transpose: the main loop already saturates the shared-memory bandwidth with TMA writes + MMA operand reads).
        // The hot path (fp16 output, full chunk, 32-byte aligned rows) is straight-line code; everything else goes through
        // the out-of-line epi_slow_chunk.
        const int ew = warp & 3;                       // TMEM lane quadrant accessible to this warp
        const int cpar = (warp - W_EPI0) >> 2;              // 0: even chunks, 1: odd chunks
        const uint32_t lane_addr = (uint32_t)(ew * 32) << 16;
        const int ncols_tile = GEGLU ? (block_n >> 1) : block_n;      // output columns per tile
        const int nchunks = ncols_tile / 32;
        const bool fast_cfg = (p.out_f32 ? ((p.ldd & 7) == 0 && !p.residual) : (p.ldd & 15) == 0) && (reinterpret_cast<uintptr_t>(p.D) & 31) == 0 &&
                              (!p.residual || ((p.ld_res & 15) == 0 && (reinterpret_cast<uintptr_t>(p.residual) & 31) == 0)) &&
                              (!p.row_bias || (p.rows_per_group & 31) == 0);
        const bool res_fast = fast_cfg && p.residual != nullptr;
        auto chunk_fast = [&](int n_blk_, int c_) -> bool {
            return fast_cfg && n_blk_ * ncols_tile + c_ * 32 + 32 <= p.n_store && n_blk_ * block_n + (GEGLU ? (block_n >> 1) : 0) + c_ * 32 + 32 <= p.N;
        };
        auto row_of = [&](int tile_, int mt_) -> long long {
            return (((long long)(tile_ / p.num_n_blocks) * MT + mt_) * CG + cta_rank) * BLOCK_M + ew * 32 + lane;
        };
        // Residual prefetch: this thread's 64 bytes of the NEXT item's residual block are requested before the current item
        // is processed (across tiles: before the wait on the accumulator), so the L2 latency is off the critical path.
        uint32_t pre0[8], pre1[8], prf0[8], prf1[8];     // residual of item +1 and of item +2
        auto issue_res = [&](int tile_, int mt_, int c_, uint32_t (&d0)[8], uint32_t (&d1)[8]) {
            if (tile_ >= num_tiles || c_ >= nchunks || !chunk_fast(tile_ % p.num_n_blocks, c_)) return;
            const long long m_ = row_of(tile_, mt_);
            if (m_ < p.M) {
                const __half* rp = p.residual + m_ * p.ld_res + (tile_ % p.num_n_blocks) * ncols_tile + c_ * 32;
                ldg256(rp, d0); ldg256(rp + 16, d1);
            }
        };
        auto next_item = [&](int& tile_, int& mt_, int& c_) {       // order in which this warp visits its chunks
            if (c_ + 2 < nchunks) c_ += 2;
            else if (mt_ + 1 < MT) { ++mt_; c_ = cpar; }
            else { tile_ += tile_step; mt_ = 0; c_ = cpar; }
        };
        // Bias staging.  With ~210 KB of shared memory the L1 is tiny, so every bias load is an L2 round trip; instead of paying
        // it per chunk, lane i fetches element i of each of this warp's chunks for the NEXT (tile, mt) group into registers
        // while the current group is processed, then parks them in the warp's private staging area, where the hot loop reads
        // them back as broadcast 128-bit shared loads.  Slots 0-3: value columns (col_bias + row_bias), 4-7: GEGLU gate columns.
        // Folded LayerNorm (p.ln_in): A holds the raw rows x and the rows of B = gamma (.) W are centred over K, so that
        // sum_k x_k B_nk = sum_k (x_k - mean) (gamma W)_nk and LN(x) W^T + b = rstd * acc + (b + W beta): the epilogue only scales
        // by this row's 1/sigma (a thread owns one row; its statistics are fetched with the next group's biases).
        const uint32_t bias_s = smem_u32(epi_smem) + (uint32_t)(warp - W_EPI0) * 1024u;
        float nb_col[4], nb_row[4], nb_gate[4];
        const bool ln_on = p.ln_in != nullptr, rs_on = p.row_scale != nullptr;
        float nl_rs = 1.0f;                                    // next group's row scale
        unsigned long long nl_s = 0, nl_q = 0;                 // next group's row statistics
        float ln_rstd = 1.0f;                                  // this group's 1/sigma (1 when no LayerNorm is folded)
        float lo_s = 0.0f, lo_q = 0.0f;                        // p.ln_out: this thread's partial row sums over its chunks
        auto bias_issue = [&](int tile_, int mt_) {
            if (!fast_cfg || tile_ >= num_tiles) return;
            const int n_blk_ = tile_ % p.num_n_blocks;
            const long long mw_ = row_of(tile_, mt_) - lane;
            const float* rbp = (p.row_bias && mw_ < p.M) ? p.row_bias + (mw_ / p.rows_per_group) * p.ld_row_bias : nullptr;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n_ = n_blk_ * block_n + (cpar + 2 * j) * 32 + lane;
                const bool in = cpar + 2 * j < nchunks && n_ < p.N;
                nb_col[j] = (p.col_bias && in) ? __ldg(p.col_bias + n_) : 0.0f;
                nb_row[j] = (rbp && in) ? __ldg(rbp + n_) : 0.0f;
                if (GEGLU) nb_gate[j] = (p.col_bias && in && n_ + (block_n >> 1) < p.N) ? __ldg(p.col_bias + n_ + (block_n >> 1)) : 0.0f;
            }
            if (ln_on) {
                const long long m_ = mw_ + lane;
                nl_s = nl_q = 0;
                if (m_ < p.M) { nl_s = __ldg(p.ln_in + 2 * m_); nl_q = __ldg(p.ln_in + 2 * m_ + 1); }
            }
            if (rs_on) { const long long m_ = mw_ + lane; nl_rs = m_ < p.M ? __ldg(p.row_scale + m_) : 1.0f; }
        };
        auto bias_commit = [&]() {
            if (!fast_cfg) return;
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(bias_s + j * 128 + lane * 4), "f"(nb_col[j] + nb_row[j]) : "memory");
                if (GEGLU) asm volatile("st.shared.f32 [%0], %1;" ::"r"(bias_s + (4 + j) * 128 + lane * 4), "f"(nb_gate[j]) : "memory");
            }
            if (ln_on) {                                          // biased variance in double: E[x^2] - mean^2 cancels
                const double mean = __ll2double_rn((long long)nl_s) * p.ln_inv;
                const double var = fma(-mean, mean, __ll2double_rn((long long)nl_q) * p.ln_inv);
                ln_rstd = rsqrtf(fmaxf((float)var, 0.0f) + p.ln_eps);
            }
            if (rs_on) ln_rstd = nl_rs;
            __syncwarp();
        };
        // GroupNorm statistics of the output (optional): per chunk slot, accumulated over this warp's tiles
        float gn_s[4] = {0.f, 0.f, 0.f, 0.f}, gn_q[4] = {0.f, 0.f, 0.f, 0.f};
        long long gn_key = -1;                                   // image * num_n_blocks + n_blk of the accumulated sums
        auto gn_flush = [&]() {
            if (gn_key < 0) return;
            const int ng = 32 / p.gn_cpg, stages = ng == 8 ? 3 : ng == 4 ? 2 : ng == 2 ? 1 : 0;
            if ((lane & ((32 >> stages) - 1)) == 0) {
                unsigned long long* st = p.gn_stats + (gn_key / p.num_n_blocks) * (2 * p.gn_groups);
                const int nb = (int)(gn_key % p.num_n_blocks);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (cpar + 2 * j >= nchunks) break;
                    // the last tile column may extend past N (N = 512 with 96-wide tiles): those chunks hold no output channels, and
                    // their (zero) sums would be added past the last group -- past the END of the statistics buffer for the last image
                    if (nb * ncols_tile + (cpar + 2 * j) * 32 >= p.n_store) break;
                    const int g = (nb * ncols_tile + (cpar + 2 * j) * 32) / p.gn_cpg + (stages ? (lane >> (5 - stages)) : 0);
                    atomicAdd(st + g * 2, (unsigned long long)__float2ll_rn(gn_s[j] * 1048576.0f));
                    atomicAdd(st + g * 2 + 1, (unsigned long long)__float2ll_rn(gn_q[j] * 1048576.0f));
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) { gn_s[j] = 0.f; gn_q[j] = 0.f; }
        };
        bias_issue(first_tile, 0);
        if (res_fast) {
            int t_ = first_tile, m_ = 0, c_ = cpar;
            issue_res(t_, m_, c_, pre0, pre1);
            next_item(t_, m_, c_);
            issue_res(t_, m_, c_, prf0, prf1);
        }
        int it = 0;
        for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++it) {
            const int buf = it & 1; const uint32_t acc_phase = (it >> 1) & 1;
            const int n_blk = tile % p.num_n_blocks;
            FIE_TIMED(tr_wait, mbar_wait(&tmem_full[buf], acc_phase));
            tc_fence_after();
#pragma unroll 1
            for (int mt = 0; mt < MT; ++mt) {
                const long long m = row_of(tile, mt);
                const bool row_ok = m < p.M;
                const uint32_t tacc = tmem_base + lane_addr + (uint32_t)((buf * MT + mt) * block_n);
                const float mb = (p.m_bias && row_ok) ? p.m_bias[m] : 0.0f;
                const float* rb = (p.row_bias && row_ok) ? p.row_bias + (m / p.rows_per_group) * p.ld_row_bias : nullptr;
                __half* orow = reinterpret_cast<__half*>(p.D) + out_row(p, row_ok ? m : 0) * p.ldd;
                bias_commit();                                         // this group's biases -> staging; then fetch the next group's
                if (mt + 1 < MT) bias_issue(tile, mt + 1); else bias_issue(tile + tile_step, 0);
#pragma unroll 1
                for (int c = cpar; c < ((p.dbg & 4) ? 0 : nchunks); c += 2) {
                    const int nacc = n_blk * block_n + c * 32;        // accumulator column (B row) of element 0
                    const int nout = n_blk * ncols_tile + c * 32;     // output column of element 0
                    uint32_t res0[8], res1[8];
                    if (res_fast) {                                   // advance the prefetch queue on EVERY item (fast or not)
#pragma unroll
                        for (int i = 0; i < 8; ++i) { res0[i] = pre0[i]; res1[i] = pre1[i]; pre0[i] = prf0[i]; pre1[i] = prf1[i]; }
                        int t_ = tile, m_ = mt, c_ = c;
                        next_item(t_, m_, c_); next_item(t_, m_, c_);
                        issue_res(t_, m_, c_, prf0, prf1);
                    }
                    if (!chunk_fast(n_blk, c)) {
                        epi_slow_chunk<OBF>(p, tacc + (uint32_t)(c * 32), GEGLU ? tacc + (uint32_t)((block_n >> 1) + c * 32) : 0u, GEGLU ? nacc + (block_n >> 1) : 0,
                                       m, row_ok, nacc, nout, mb, rb);
                        continue;
                    }
                    const uint32_t bslot = bias_s + (uint32_t)(((c - cpar) >> 1) * 128);
                    float v[32];
                    if (GEGLU) {
                        uint32_t r[32], g[32];
                        tmem_ld_32x32(tacc + (uint32_t)(c * 32), r);
                        tmem_ld_32x32(tacc + (uint32_t)((block_n >> 1) + c * 32), g);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const uint4 bv = lds128(bslot + i * 16), bg = lds128(bslot + 512 + i * 16);
                            v[4 * i] = FIE_LN_LIN(r[4 * i], bv.x) * gelu_erf_f(FIE_LN_LIN(g[4 * i], bg.x));
                            v[4 * i + 1] = FIE_LN_LIN(r[4 * i + 1], bv.y) * gelu_erf_f(FIE_LN_LIN(g[4 * i + 1], bg.y));
                            v[4 * i + 2] = FIE_LN_LIN(r[4 * i + 2], bv.z) * gelu_erf_f(FIE_LN_LIN(g[4 * i + 2], bg.z));
                            v[4 * i + 3] = FIE_LN_LIN(r[4 * i + 3], bv.w) * gelu_erf_f(FIE_LN_LIN(g[4 * i + 3], bg.w));
                        }
                    } else {
                        uint32_t r[32];
                        tmem_ld_32x32(tacc + (uint32_t)(c * 32), r);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const uint4 bv = lds128(bslot + i * 16);
                            v[4 * i] = FIE_LN_LIN(r[4 * i], bv.x); v[4 * i + 1] = FIE_LN_LIN(r[4 * i + 1], bv.y);
                            v[4 * i + 2] = FIE_LN_LIN(r[4 * i + 2], bv.z); v[4 * i + 3] = FIE_LN_LIN(r[4 * i + 3], bv.w);
                        }
                        if (p.act == FIE_ACT_SILU) {
#pragma unroll
                            for (int i = 0; i < 32; ++i) v[i] = silu_f(v[i]);
                        } else if (p.act == FIE_ACT_GELU) {
#pragma unroll
                            for (int i = 0; i < 32; ++i) v[i] = gelu_erf_f(v[i]);
                        } else if (p.act == FIE_ACT_QUICKGELU) {
#pragma unroll
                            for (int i = 0; i < 32; ++i) v[i] = quick_gelu_f(v[i]);
                        } else if (p.act == FIE_ACT_RELU) {
#pragma unroll
                            for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.0f);
                        }
                    }
                    if (p.m_bias) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] += mb;        // (GEGLU with a per-row bias is not a supported combination)
                    }
                    if (p.scale != 1.0f) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] *= p.scale;
                    }
                    if (res_fast && row_ok) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            float2 f = unpack_h2<OBF>(res0[i]); v[2 * i] += f.x; v[2 * i + 1] += f.y;
                            f = unpack_h2<OBF>(res1[i]); v[16 + 2 * i] += f.x; v[16 + 2 * i + 1] += f.y;
                        }
                    }
                    if (p.ln_out) {                                     // LayerNorm statistics of this row of the (fp16-rounded) output
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const float2 f = __half22float2(__floats2half2_rn(v[2 * i], v[2 * i + 1]));
                            lo_s += f.x + f.y; lo_q = fmaf(f.x, f.x, fmaf(f.y, f.y, lo_q));
                        }
                    }
                    // GroupNorm statistics of the (fp16-rounded) output for the consumer.  Only warps whose rows start below M: a warp of the
                    // last, partial tile that lies wholly past M would key image n, one block past the [n][groups][2] buffer.  (gn_rows is a
                    // multiple of 32 and divides M, so a warp is either wholly inside or wholly past M, and never spans two images.)
                    if (p.gn_stats && m - lane < p.M) {
                        const long long key = ((m - lane) / p.gn_rows) * p.num_n_blocks + n_blk;
                        if (key != gn_key) { gn_flush(); gn_key = key; }
                        float vr[32];
#pragma unroll
                        for (int i = 0; i < 16; ++i) { const float2 f = __half22float2(__floats2half2_rn(v[2 * i], v[2 * i + 1])); vr[2 * i] = f.x; vr[2 * i + 1] = f.y; }
                        const int slot = (c - cpar) >> 1;
                        float ds = 0.f, dq = 0.f;
                        if (p.gn_cpg == 4) gn_stats_chunk<8>(vr, row_ok, lane, ds, dq);
                        else if (p.gn_cpg == 8) gn_stats_chunk<4>(vr, row_ok, lane, ds, dq);
                        else if (p.gn_cpg == 16) gn_stats_chunk<2>(vr, row_ok, lane, ds, dq);
                        else gn_stats_chunk<1>(vr, row_ok, lane, ds, dq);
#pragma unroll
                        for (int j = 0; j < 4; ++j) if (j == slot) { gn_s[j] += ds; gn_q[j] += dq; }
                    }
                    if (p.out_f32) {
                        if (row_ok) {                                   // fp32 output (attention scores): 128 B per row and chunk
                            float* of = reinterpret_cast<float*>(p.D) + out_row(p, m) * p.ldd + nout;
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                uint32_t o[8];
#pragma unroll
                                for (int j = 0; j < 8; ++j) o[j] = __float_as_uint(v[8 * i + j]);
                                stg256(of + 8 * i, o);
                            }
                        }
                    } else if (row_ok) {
                        uint32_t o0[8], o1[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) { o0[i] = pack_h2<OBF>(v[2 * i], v[2 * i + 1]); o1[i] = pack_h2<OBF>(v[16 + 2 * i], v[16 + 2 * i + 1]); }
                        stg256(orow + nout, o0); stg256(orow + nout + 16, o1);
                    }
                }
                if (p.ln_out) {
                    if (row_ok) {
                        atomicAdd(p.ln_out + 2 * m, (unsigned long long)__float2ll_rn(lo_s * 1048576.0f));
                        atomicAdd(p.ln_out + 2 * m + 1, (unsigned long long)__float2ll_rn(lo_q * 1048576.0f));
                    }
                    lo_s = 0.0f; lo_q = 0.0f;
                }
            }   // mt
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (CG == 2) mbar_arrive_remote_relaxed(&tmem_empty[buf], 0); else mbar_arrive_relaxed(&tmem_empty[buf]); }
        }
        if (p.gn_stats) gn_flush();
        if (p.trace && warp == W_EPI0 && lane == 0) { p.trace[blockIdx.x * 8 + 5] = tr_wait; p.trace[blockIdx.x * 8 + 6] = clock64() - tr_start; }
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();   // the peer's MMAs read this CTA's shared memory until the very end
    if (warp == W_ALLOC) {
        tc_fence_after();
        if (CG == 2) tmem_dealloc_2sm(tmem_base, (uint32_t)p.tmem_cols); else tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
    }
}

// ------------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------------

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

int make_tmap_f16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box, bool bf16) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled not available (driver too old?)"); return FIE_ERR_CUDA; }
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) { set_error("TMA base pointer %p not 16-byte aligned", base); return FIE_ERR_INVALID; }
    cuuint64_t gd[5]; cuuint64_t gs[4]; cuuint32_t bx[5]; cuuint32_t es[5];
    for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; if (box[i] > 256 || box[i] == 0) { set_error("TMA box dim %d = %u out of range", i, box[i]); return FIE_ERR_INVALID; } }
    for (int i = 0; i + 1 < rank; ++i) { gs[i] = strides_bytes[i]; if (gs[i] & 15) { set_error("TMA stride %d = %llu not a multiple of 16 bytes", i, (unsigned long long)gs[i]); return FIE_ERR_INVALID; } }
    CUresult r = enc(out, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d dims %llu,%llu box %u,%u)", (int)r, rank,
                                       (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0), box[0], rank > 1 ? box[1] : 0); return FIE_ERR_CUDA; }
    return FIE_OK;
}

typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const int*,
                                     const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_tmap_im2col_f16(CUtensorMap* out, const void* base, const uint64_t* dims, const uint64_t* strides_bytes, const int* lower,
                         const int* upper, bool bf16) {
    static PFN_encodeIm2col enc = nullptr;
    if (!enc) {
        void* fp = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fp, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            enc = (PFN_encodeIm2col)fp;
    }
    if (!enc) { set_error("cuTensorMapEncodeIm2col not available (driver too old?)"); return FIE_ERR_CUDA; }
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) { set_error("TMA base pointer %p not 16-byte aligned", base); return FIE_ERR_INVALID; }
    cuuint64_t gd[4]; cuuint64_t gs[3]; const cuuint32_t es[4] = {1, 1, 1, 1};
    for (int i = 0; i < 4; ++i) gd[i] = dims[i];
    for (int i = 0; i < 3; ++i) { gs[i] = strides_bytes[i]; if (gs[i] & 15) { set_error("TMA stride %d = %llu not a multiple of 16 bytes", i, (unsigned long long)gs[i]); return FIE_ERR_INVALID; } }
    CUresult r = enc(out, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), gd, gs, lower, upper,
                     (cuuint32_t)BLOCK_K, (cuuint32_t)BLOCK_M, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeIm2col failed with CUresult %d (dims %llu,%llu,%llu,%llu)", (int)r, (unsigned long long)dims[0],
                                       (unsigned long long)dims[1], (unsigned long long)dims[2], (unsigned long long)dims[3]); return FIE_ERR_CUDA; }
    return FIE_OK;
}

static int num_sms() { return device_sm_count(); }

static int g_force_im2col = 0;      // test / measurement hook (fie_tune_conv_im2col): im2col mode on shapes the box also tiles

// The rectangular A box {64 ch, bw, bh, bn} of 128 output pixels for an OH x OW output, or false when no such box tiles it (the
// width is neither a multiple nor a divisor of 128, or the rows do not stack into whole boxes): those shapes run in im2col mode.
static bool box_tile(int OW, int OH, int* bw, int* bh, int* bn) {
    if (g_force_im2col) return false;
    if (OW >= BLOCK_M) { *bw = BLOCK_M; *bh = 1; *bn = 1; return (OW % BLOCK_M) == 0; }
    if ((BLOCK_M % OW) != 0) return false;
    *bw = OW; *bh = BLOCK_M / OW; *bn = 1;
    if (*bh <= OH) return (OH % *bh) == 0;
    if ((*bh % OH) != 0) return false;
    *bn = *bh / OH; *bh = OH;
    return true;
}

// Tile configuration.  Measured on B200 (scripts/gemm_bench.py, scripts/gemm_dbg.py): the producer/consumer mbarrier
// handshake costs ~300 ns per pipeline stage regardless of tile width, so the kernel runs 2 K-blocks per stage (KPS = 2)
// and prefers the CTA-pair form (cta_group::2: 256-row tiles, B split across the pair) with the widest accumulator that
// does not waste columns: time per tile and K-block ~ (290 + block_n).  Waves are quantised over 74 CTA pairs.
// fie_tune_gemm() can force the form for experiments.
static int g_force_cg = -1;
static int g_force_bn = 0;
static int g_dbg = 0;
static int g_force_kps = 0;
static int g_force_mt = 0;
static long long* g_trace = nullptr;
static int g_halo = -1;             // FIE_CONV_HALO=0 disables the halo convolution path
static int g_halo_max_cout = 640;   // wider outputs reuse each A tile enough for the per-tap form to win
static void pick_config(long long M, int N, bool geglu, int* cg_out, int* bn_out, int* mt_out, int max_mt = 2) {
    if (g_force_cg < 0) { const char* s = getenv("FIE_GEMM_CG"); g_force_cg = s ? atoi(s) : 0; }
    const int sms = num_sms();
    double best_cost = 1e30; int best_cg = 2, best_bn = 32, best_mt = 1;
    for (int cg = 2; cg >= 1; --cg) {
        if (g_force_cg && cg != g_force_cg) continue;
        if (!g_force_cg && cg == 1 && M > BLOCK_M) continue;          // single-CTA form only for one-tile-high problems
        for (int mt = 1; mt <= max_mt; ++mt) {
            if (g_force_mt && mt != g_force_mt && max_mt > 1) continue;
            if (!g_force_mt && mt == 2 && N > 128) continue;     // measured: two M sub-tiles only pay off for N <= 128
            const long long mblocks = (M + BLOCK_M * cg * mt - 1) / (BLOCK_M * cg * mt);
            const int slots = sms / cg;
            for (int bn = 32; bn <= 256 / mt; bn += 32) {       // 2 buffers x mt x bn TMEM columns <= 512
                if (geglu && bn != fie_geglu_block_n(N)) continue;   // GEGLU rows are pre-interleaved per tile by the host
                if (!geglu && g_force_bn && bn != g_force_bn) continue;
                const long long tiles = mblocks * ((N + bn - 1) / bn);
                const long long waves = (tiles + slots - 1) / slots;
                const double cost = (double)waves * (mt * bn + 290.0) * (cg == 1 ? 0.6 : 1.0);
                if (cost < best_cost - 1e-9 || (cost < best_cost + 1e-9 && mt * bn > best_mt * best_bn)) { best_cost = cost; best_cg = cg; best_bn = bn; best_mt = mt; }
            }
        }
    }
    *cg_out = best_cg; *bn_out = best_bn; *mt_out = best_mt;
}

static int out_dtype_of(const fie_epilogue* ep) { return (ep && ep->out_f32) ? FIE_DT_F32 : FIE_DT_F16; }

// Validation of the explicit output type of the *_bf16 entry points (before any CUDA call).
static int check_out_dtype(const char* fn, const fie_epilogue* ep, int out_dtype) {
    FIE_REQUIRE(out_dtype == FIE_DT_F16 || out_dtype == FIE_DT_BF16 || out_dtype == FIE_DT_F32, "%s: bad out_dtype %d", fn, out_dtype);
    FIE_REQUIRE(!(ep && ep->out_f32 && out_dtype != FIE_DT_F32), "%s: fie_epilogue.out_f32 needs out_dtype FIE_DT_F32", fn);
    return FIE_OK;
}

static int fill_epilogue(GemmParams& p, const fie_epilogue* ep, long long M, int N, void* D, long long ldd, int out_dtype) {
    static const fie_epilogue kDefault = {nullptr, nullptr, 1, 0, nullptr, nullptr, 0, 1.0f, FIE_ACT_NONE, 0, nullptr, 0, 0, nullptr, nullptr, 0.0f, 0, nullptr};
    if (!ep) ep = &kDefault;
    p.D = D; p.ldd = ldd;
    p.col_bias = ep->col_bias; p.row_bias = ep->row_bias; p.rows_per_group = ep->rows_per_group > 0 ? ep->rows_per_group : 1;
    p.ld_row_bias = ep->ld_row_bias > 0 ? ep->ld_row_bias : N;
    p.m_bias = ep->m_bias; p.residual = (const __half*)ep->residual; p.ld_res = ep->ld_res;
    p.scale = ep->scale; p.act = ep->act; p.out_f32 = out_dtype == FIE_DT_F32; p.out_bf16 = out_dtype == FIE_DT_BF16;
    FIE_REQUIRE(p.act >= 0 && p.act <= FIE_ACT_RELU, "epilogue: bad act %d", p.act);
    FIE_REQUIRE(!(p.out_bf16 && (ep->gn_stats || ep->ln_stats_out || p.act == FIE_ACT_GEGLU)),
                "epilogue: gn_stats, ln_stats_out and GEGLU need fp16 output (not supported with bf16 output)");
    FIE_REQUIRE(!(p.act == FIE_ACT_GEGLU && (N % 64)), "GEGLU needs N %% 64 == 0");
    FIE_REQUIRE(!(p.residual && p.ld_res <= 0), "epilogue: residual needs ld_res");
    p.gn_stats = (unsigned long long*)ep->gn_stats; p.gn_groups = ep->gn_groups; p.gn_rows = ep->gn_rows_per_image; p.gn_cpg = 0;
    if (p.gn_stats) {
        const int n_out = p.act == FIE_ACT_GEGLU ? N / 2 : N;
        FIE_REQUIRE(p.gn_groups > 0 && (n_out % p.gn_groups) == 0, "epilogue: gn_groups must divide the output channels");
        p.gn_cpg = n_out / p.gn_groups;
        FIE_REQUIRE(p.gn_cpg <= 32 && (32 % p.gn_cpg) == 0 && p.gn_cpg >= 4, "epilogue: fused GroupNorm statistics need channels/group in {4, 8, 16, 32} (got %d)", p.gn_cpg);
        FIE_REQUIRE(p.gn_rows > 0 && (p.gn_rows % 32) == 0 && (M % p.gn_rows) == 0,
                    "epilogue: gn_rows_per_image must be a positive multiple of 32 that divides the rows");
        FIE_REQUIRE(!p.out_f32 && (n_out % 32) == 0 && (ldd % 16) == 0 && (reinterpret_cast<uintptr_t>(D) & 31) == 0 &&
                    (!p.residual || ((p.ld_res % 16) == 0 && (reinterpret_cast<uintptr_t>(p.residual) & 31) == 0)) &&
                    (!p.row_bias || (p.rows_per_group % 32) == 0),
                    "epilogue: fused GroupNorm statistics need the fast epilogue path (fp16 output, N %% 32 == 0, 32-byte aligned rows)");
    }
    p.ln_out = (unsigned long long*)ep->ln_stats_out; p.ln_in = (const unsigned long long*)ep->ln_stats_in;
    p.ln_eps = ep->ln_eps; p.ln_inv = ep->ln_dim > 0 ? 1.0 / (1048576.0 * (double)ep->ln_dim) : 0.0;
    p.row_scale = ep->row_scale;
    FIE_REQUIRE(!(p.row_scale && p.ln_in), "epilogue: row_scale and ln_stats_in are exclusive");
    if (p.ln_out || p.ln_in || p.row_scale) {
        const int n_out = p.act == FIE_ACT_GEGLU ? N / 2 : N;
        FIE_REQUIRE(!p.out_f32 && (n_out % 32) == 0 && (N % 32) == 0 && (ldd % 16) == 0 && (reinterpret_cast<uintptr_t>(D) & 31) == 0 &&
                    (!p.residual || ((p.ld_res % 16) == 0 && (reinterpret_cast<uintptr_t>(p.residual) & 31) == 0)) &&
                    (!p.row_bias || (p.rows_per_group % 32) == 0),
                    "epilogue: folded LayerNorm / row_scale need the fast epilogue path (fp16 output, N %% 32 == 0, 32-byte aligned rows)");
        FIE_REQUIRE(!p.ln_in || (ep->ln_dim > 0 && p.ln_eps >= 0.0f && !p.row_bias && !p.m_bias), "epilogue: ln_stats_in needs ln_dim > 0, ln_eps >= 0 and no row / m bias");
        FIE_REQUIRE(!(p.ln_out && p.act == FIE_ACT_GEGLU), "epilogue: ln_stats_out is not supported with the GEGLU epilogue");
    }
    return FIE_OK;
}

static int launch(GemmParams& p, cudaStream_t stream) {
    const int cg = p.cg;
    p.dbg = g_dbg;
    p.trace = g_trace;
    const int mt = p.mt;
    int kps = (g_force_kps > 0) ? g_force_kps : (p.num_kb >= 4 ? 2 : 1);
    if (kps == 2 && SMEM_BUDGET / (2 * (mt * A_STAGE_BYTES + (p.block_n / cg) * BLOCK_K * 2)) < 2) kps = 1;
    int halo_tps = 1;                              // halo: ring stage = B tiles of 9 taps (narrow N), else 3 (one kernel row), else 1, as two stages fit
    if (p.mode == 2) {
        kps = 1;
        const int bsub = (p.block_n / cg) * BLOCK_K * 2;
        if (2 * 9 * bsub <= SMEM_BUDGET - HALO_A_BYTES) halo_tps = 9;          // one handshake per channel chunk: N <= 80 would be handshake-bound otherwise
        else if (2 * 3 * bsub <= SMEM_BUDGET - HALO_A_BYTES) halo_tps = 3;
        if (g_force_kps == 1) halo_tps = 1;
    }
    p.kps = p.mode == 2 ? halo_tps : kps;
    const int stage_bytes = p.mode == 2 ? halo_tps * (p.block_n / cg) * BLOCK_K * 2 : kps * (mt * A_STAGE_BYTES + (p.block_n / cg) * BLOCK_K * 2);
    int stages = (p.mode == 2 ? SMEM_BUDGET - HALO_A_BYTES : SMEM_BUDGET) / stage_bytes; if (stages > MAX_STAGES) stages = MAX_STAGES;
    if (stages < 2) stages = 2;
    p.num_stages = stages;
    int cols = 2 * mt * p.block_n, tc = 32; while (tc < cols) tc <<= 1;
    p.tmem_cols = tc;
    size_t smem = (size_t)SMEM_BUDGET + EPI_STAGE_BYTES + 1024;
    // (>113 KiB of dynamic smem: one CTA per SM, so a 512-column TMEM allocation can never deadlock)
    typedef void (*KernelFn)(GemmParams);
#define FIE_K(cg, kps, mt) {k_gemm_conv<cg, kps, mt, 0, 0>, k_gemm_conv<cg, kps, mt, 1, 0>, k_gemm_conv<cg, kps, mt, 0, 1>}
    static const KernelFn kernels[2][2][2][3] = {{{FIE_K(1, 1, 1), FIE_K(1, 1, 2)}, {FIE_K(1, 2, 1), FIE_K(1, 2, 2)}},
                                                 {{FIE_K(2, 1, 1), FIE_K(2, 1, 2)}, {FIE_K(2, 2, 1), FIE_K(2, 2, 2)}}};
#undef FIE_K
    static bool attr_set_dev[kMaxDevices] = {false};          // cudaFuncSetAttribute is per device
    bool& attr_set = attr_set_dev[current_device()];
    if (!attr_set) {
        for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) for (int c = 0; c < 2; ++c) for (int d = 0; d < 3; ++d) {
            cudaError_t e = cudaFuncSetAttribute(kernels[a][b][c][d], cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BUDGET + EPI_STAGE_BYTES + 1024);
            if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(k_gemm_conv): %s", cudaGetErrorString(e)); return FIE_ERR_CUDA; }
        }
        attr_set = true;
    }
    KernelFn fn = kernels[cg - 1][kps - 1][mt - 1][p.act == FIE_ACT_GEGLU ? 1 : (p.out_bf16 ? 2 : 0)];
    const int tiles = p.num_m_blocks * p.num_n_blocks;
    const int slots = num_sms() / cg;
    const int grid = cg * (tiles < slots ? tiles : slots);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(384); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    static int pdl = -1;                               // FIE_PDL=0: plain stream-ordered launches
    if (pdl < 0) { const char* e = getenv("FIE_PDL"); pdl = e ? atoi(e) : 1; }
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cg; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 2 : 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, fn, p);
    if (e != cudaSuccess) { set_error("cudaLaunchKernelEx(k_gemm_conv): %s", cudaGetErrorString(e)); cudaGetLastError(); return FIE_ERR_CUDA; }
    return check_launch("k_gemm_conv");
}

}  // namespace fie

using namespace fie;

extern "C" void fie_tune_conv_halo(int enable, int max_cout) { fie::g_halo = enable; if (max_cout > 0) fie::g_halo_max_cout = max_cout; }

extern "C" void fie_tune_conv_im2col(int force) { fie::g_force_im2col = force != 0; }

extern "C" void fie_tune_gemm(int force_cg, int force_block_n) { fie::g_force_cg = force_cg & 3; fie::g_force_kps = (force_cg >> 2) & 3; fie::g_dbg = (force_cg >> 4) & 15; fie::g_force_mt = (force_cg >> 8) & 3; fie::g_force_bn = force_block_n; }

// Debug: install (or clear, with NULL) a device buffer of 8 x int64 per CTA that the next GEMM launches fill with
// [0] producer cycles blocked on "empty", [1] producer total, [2] MMA issuer blocked on "full", [3] on the accumulator buffer,
// [4] issuer total, [5] epilogue warp 4 blocked on "accumulator full", [6] epilogue total.
extern "C" void fie_gemm_trace(long long* device_buf) { fie::g_trace = device_buf; }

extern "C" int fie_geglu_block_n(int N) { return (N % 256) == 0 ? 256 : ((N % 128) == 0 ? 128 : 64); }

static int gemm_impl(const char* fn, const void* A, long long lda, const void* A1, long long lda1, int k_split,
                     const void* B, void* D, long long ldd, long long M, int N, int K,
                     const fie_epilogue* ep, int ab_bf16, int out_dtype, void* stream) {
    FIE_REQUIRE(A && B && D, "%s: null pointer", fn);
    FIE_REQUIRE(M > 0 && N > 0 && K > 0, "%s: bad shape M=%lld N=%d K=%d", fn, M, N, K);
    FIE_REQUIRE(M < (1ll << 31), "%s: M too large", fn);
    FIE_REQUIRE((lda % 8) == 0 && (K % 8) == 0 && lda >= (A1 ? k_split : K), "%s: lda/K must be multiples of 8", fn);
    GemmParams p;
    memset(&p, 0, sizeof(p));
    int rc = fill_epilogue(p, ep, M, N, D, ldd, out_dtype);
    if (rc) return rc;
    const bool geglu = p.act == FIE_ACT_GEGLU;
    p.mode = 0; p.M = M; p.N = N; p.ab_bf16 = ab_bf16;
    pick_config(M, N, geglu, &p.cg, &p.block_n, &p.mt);
    p.num_m_blocks = (int)((M + BLOCK_M * p.cg * p.mt - 1) / (BLOCK_M * p.cg * p.mt));
    p.num_n_blocks = (N + p.block_n - 1) / p.block_n;
    p.num_kb = (K + BLOCK_K - 1) / BLOCK_K;
    p.kb_per_tap = p.num_kb; p.kb_split = p.num_kb;
    p.n_store = geglu ? N / 2 : N;
    uint64_t dims[2], strides[1]; uint32_t box[2];
    if (A1) {
        FIE_REQUIRE(k_split > 0 && k_split < K && (k_split % BLOCK_K) == 0 && (lda1 % 8) == 0 && lda1 >= K - k_split, "%s: bad two-source split", fn);
        p.kb_split = k_split / BLOCK_K;
        dims[0] = (uint64_t)k_split; dims[1] = (uint64_t)M; strides[0] = (uint64_t)lda * 2; box[0] = BLOCK_K; box[1] = BLOCK_M;
        if ((rc = make_tmap_f16(&p.a_maps[0], A, 2, dims, strides, box, ab_bf16 != 0))) return rc;
        dims[0] = (uint64_t)(K - k_split); strides[0] = (uint64_t)lda1 * 2;
        if ((rc = make_tmap_f16(&p.a_maps[1], A1, 2, dims, strides, box, ab_bf16 != 0))) return rc;
    } else {
        dims[0] = (uint64_t)K; dims[1] = (uint64_t)M; strides[0] = (uint64_t)lda * 2; box[0] = BLOCK_K; box[1] = BLOCK_M;
        if ((rc = make_tmap_f16(&p.a_maps[0], A, 2, dims, strides, box, ab_bf16 != 0))) return rc;
        p.a_maps[1] = p.a_maps[0];
    }
    p.a_maps[2] = p.a_maps[0]; p.a_maps[3] = p.a_maps[0];
    dims[0] = (uint64_t)K; dims[1] = (uint64_t)N; strides[0] = (uint64_t)K * 2; box[0] = BLOCK_K; box[1] = (uint32_t)(p.block_n / p.cg);
    if ((rc = make_tmap_f16(&p.b_map, B, 2, dims, strides, box, ab_bf16 != 0))) return rc;
    return launch(p, (cudaStream_t)stream);
}

static int conv3x3_impl(const char* fn, const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                        int cout_valid, int stride, int pad_mode, const fie_epilogue* ep, int ab_bf16, int out_dtype, void* stream) {
    FIE_REQUIRE(x && wgt && out, "%s: null pointer", fn);
    FIE_REQUIRE(n > 0 && h > 0 && w > 0 && cin > 0 && cout > 0, "%s: bad shape", fn);
    FIE_REQUIRE((cin % BLOCK_K) == 0, "%s: cin=%d must be a multiple of 64", fn, cin);
    FIE_REQUIRE((cout % 32) == 0, "%s: cout=%d (weight rows) must be a multiple of 32", fn, cout);
    FIE_REQUIRE(stride == 1 || stride == 2, "%s: stride must be 1 or 2", fn);
    FIE_REQUIRE(stride == 1 || ((h % 2) == 0 && (w % 2) == 0), "%s: stride 2 needs even h, w", fn);
    const int OH = h / stride, OW = w / stride;
    int bw = 0, bh = 0, bn = 0;
    const bool boxed = box_tile(OW, OH, &bw, &bh, &bn);
    GemmParams p;
    memset(&p, 0, sizeof(p));
    const long long M = (long long)n * OH * OW;
    int rc = fill_epilogue(p, ep, M, cout, out, ldd, out_dtype);
    if (rc) return rc;
    FIE_REQUIRE(p.act != FIE_ACT_GEGLU, "%s: GEGLU epilogue not supported for conv", fn);
    if (g_halo < 0) { const char* e = getenv("FIE_CONV_HALO"); g_halo = e ? atoi(e) : 1; }
    const bool halo = boxed && g_halo > 0 && stride == 1 && (OW % BLOCK_M) == 0 && cout <= g_halo_max_cout;
    p.mode = halo ? 2 : (boxed ? 1 : 3); p.M = M; p.N = cout; p.OH = OH; p.OW = OW; p.ab_bf16 = ab_bf16;
    pick_config(M, cout, false, &p.cg, &p.block_n, &p.mt, halo ? 1 : 2);
    p.num_m_blocks = (int)((M + BLOCK_M * p.cg * p.mt - 1) / (BLOCK_M * p.cg * p.mt));
    p.num_n_blocks = (cout + p.block_n - 1) / p.block_n;
    p.kb_per_tap = cin / BLOCK_K;
    p.num_kb = 9 * p.kb_per_tap;
    p.kb_split = p.num_kb;
    p.n_store = cout_valid > 0 ? cout_valid : cout;
    const uint32_t box[4] = {BLOCK_K, (uint32_t)(halo ? HALO_PX : bw), (uint32_t)(halo ? 1 : bh), (uint32_t)(halo ? 1 : bn)};
    static const int lower[2] = {-1, -1}, upper[2] = {-1, -1};    // im2col: one run position per output pixel of the view
    if (stride == 1) {
        const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)w, (uint64_t)h, (uint64_t)n};
        const uint64_t strides[3] = {(uint64_t)cin * 2, (uint64_t)w * cin * 2, (uint64_t)h * w * cin * 2};
        if ((rc = boxed ? make_tmap_f16(&p.a_maps[0], x, 4, dims, strides, box, ab_bf16 != 0)
                        : make_tmap_im2col_f16(&p.a_maps[0], x, dims, strides, lower, upper, ab_bf16 != 0))) return rc;
        p.a_maps[1] = p.a_maps[0]; p.a_maps[2] = p.a_maps[0]; p.a_maps[3] = p.a_maps[0];
        for (int t = 0; t < 9; ++t) { p.tap_map[t] = 0; p.tap_dh[t] = (int8_t)(t / 3 - 1); p.tap_dw[t] = (int8_t)(t % 3 - 1); }
    } else {
        // parity-split views: element (c, w2, h2, n) of view (hp, wp) is x[n, 2*h2+hp, 2*w2+wp, c]
        const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)(w / 2), (uint64_t)(h / 2), (uint64_t)n};
        const uint64_t strides[3] = {(uint64_t)cin * 4, (uint64_t)w * cin * 4, (uint64_t)h * w * cin * 2};
        for (int hp = 0; hp < 2; ++hp)
            for (int wp = 0; wp < 2; ++wp) {
                const uint8_t* base = (const uint8_t*)x + ((size_t)hp * w + wp) * cin * 2;
                if ((rc = boxed ? make_tmap_f16(&p.a_maps[hp * 2 + wp], base, 4, dims, strides, box, ab_bf16 != 0)
                                : make_tmap_im2col_f16(&p.a_maps[hp * 2 + wp], base, dims, strides, lower, upper, ab_bf16 != 0))) return rc;
            }
        // input row = 2*oh + k - pad:  pad 1: k=0 -> (parity 1, shift -1), k=1 -> (0, 0), k=2 -> (1, 0)
        //                              pad 0 (asymmetric (0,1) padding): k=0 -> (0, 0), k=1 -> (1, 0), k=2 -> (0, +1)
        static const int par1[3] = {1, 0, 1}, sh1[3] = {-1, 0, 0}, par0[3] = {0, 1, 0}, sh0[3] = {0, 0, 1};
        const int* par = pad_mode == 0 ? par1 : par0; const int* sh = pad_mode == 0 ? sh1 : sh0;
        for (int t = 0; t < 9; ++t) {
            const int kh = t / 3, kw = t % 3;
            p.tap_map[t] = (int8_t)(par[kh] * 2 + par[kw]); p.tap_dh[t] = (int8_t)sh[kh]; p.tap_dw[t] = (int8_t)sh[kw];
        }
    }
    const uint64_t bdims[2] = {(uint64_t)9 * cin, (uint64_t)cout};
    const uint64_t bstr[1] = {(uint64_t)9 * cin * 2};
    const uint32_t bbox[2] = {BLOCK_K, (uint32_t)(p.block_n / p.cg)};
    if ((rc = make_tmap_f16(&p.b_map, wgt, 2, bdims, bstr, bbox, ab_bf16 != 0))) return rc;
    return launch(p, (cudaStream_t)stream);
}

// Nearest-2x upsample fused into the following 3x3 convolution (diffusers Upsample2D: F.interpolate(scale 2, nearest) then
// conv3x3).  Output pixel (2i+a, 2j+b) only ever sees a 2x2 neighbourhood of the input, with the 3x3 taps that land on the
// same input pixel pre-summed by the host: four phase convolutions with 2x2 taps = 16/36 of the FLOPs and no upsampled
// tensor in HBM.  wgt: fp16 [4 phases (a*2+b)][cout][2][2][cin].
static int conv_up2x_impl(const char* fn, const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                          const fie_epilogue* ep, int ab_bf16, int out_dtype, void* stream) {
    FIE_REQUIRE(x && wgt && out, "%s: null pointer", fn);
    FIE_REQUIRE(n > 0 && h > 0 && w > 0 && cin > 0 && cout > 0, "%s: bad shape", fn);
    FIE_REQUIRE((cin % BLOCK_K) == 0 && (cout % 32) == 0, "%s: cin %% 64 and cout %% 32 required", fn);
    int bw = 0, bh = 0, bn = 0;
    const bool boxed = box_tile(w, h, &bw, &bh, &bn);
    const long long M = (long long)n * h * w;
    for (int ph = 0; ph < 4; ++ph) {
        GemmParams p;
        memset(&p, 0, sizeof(p));
        int rc = fill_epilogue(p, ep, M, cout, out, ldd, out_dtype);
        if (rc) return rc;
        FIE_REQUIRE(p.act != FIE_ACT_GEGLU && !p.residual && !p.out_f32, "%s: unsupported epilogue", fn);
        p.mode = boxed ? 1 : 3; p.M = M; p.N = cout; p.OH = h; p.OW = w; p.ab_bf16 = ab_bf16;
        p.up2 = 1; p.up_a = ph >> 1; p.up_b = ph & 1;
        pick_config(M, cout, false, &p.cg, &p.block_n, &p.mt);
        p.num_m_blocks = (int)((M + BLOCK_M * p.cg * p.mt - 1) / (BLOCK_M * p.cg * p.mt));
        p.num_n_blocks = (cout + p.block_n - 1) / p.block_n;
        p.kb_per_tap = cin / BLOCK_K;
        p.num_kb = 4 * p.kb_per_tap;
        p.kb_split = p.num_kb;
        p.n_store = cout;
        const uint32_t box[4] = {BLOCK_K, (uint32_t)bw, (uint32_t)bh, (uint32_t)bn};
        const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)w, (uint64_t)h, (uint64_t)n};
        const uint64_t strides[3] = {(uint64_t)cin * 2, (uint64_t)w * cin * 2, (uint64_t)h * w * cin * 2};
        static const int lower[2] = {-1, -1}, upper[2] = {-1, -1};
        if ((rc = boxed ? make_tmap_f16(&p.a_maps[0], x, 4, dims, strides, box, ab_bf16 != 0)
                        : make_tmap_im2col_f16(&p.a_maps[0], x, dims, strides, lower, upper, ab_bf16 != 0))) return rc;
        p.a_maps[1] = p.a_maps[0]; p.a_maps[2] = p.a_maps[0]; p.a_maps[3] = p.a_maps[0];
        for (int t = 0; t < 4; ++t) {   // tap (ty, tx): input row i + ty - 1 + a, column j + tx - 1 + b
            p.tap_map[t] = 0; p.tap_dh[t] = (int8_t)((t >> 1) - 1 + p.up_a); p.tap_dw[t] = (int8_t)((t & 1) - 1 + p.up_b);
        }
        const uint64_t bdims[2] = {(uint64_t)4 * cin, (uint64_t)cout};
        const uint64_t bstr[1] = {(uint64_t)4 * cin * 2};
        const uint32_t bbox[2] = {BLOCK_K, (uint32_t)(p.block_n / p.cg)};
        const uint8_t* wp = (const uint8_t*)wgt + (size_t)ph * cout * 4 * cin * 2;
        if ((rc = make_tmap_f16(&p.b_map, wp, 2, bdims, bstr, bbox, ab_bf16 != 0))) return rc;
        if ((rc = launch(p, (cudaStream_t)stream))) return rc;
    }
    return FIE_OK;
}

// 3x3 convolution of an image-like input with <= 8 channels (conv_in of the VAE encoder and of the ControlNet conditioning
// embedding at full resolution) on the tensor cores.  The input is stored zero-padded as xp[n][h+2][w+8][8] fp16 (real pixel
// (y, x) at (y+1, x+1); see fie_preprocess_u8_to_f16_pad8), so the 3 pixels x 8 channels one kernel row needs for output pixel x are
// 24 contiguous fp16 starting at padded pixel x.  The A operand is an OVERLAPPING TMA view: dimension 0 = 64 contiguous fp16
// (8 padded pixels, of which the first 3 carry non-zero weights), dimension 1 = start pixel with a 16-byte stride.  K = 3 kernel
// rows x 64, so the generic implicit-GEMM kernel runs unchanged with 3 "taps" of one K block each.
// wgt: fp16 [cout][3][2][64]: per kernel row a hi and a lo block (w = hi + lo to ~2^-22), element kw*8 + c = w[co][c][kh][kw].
static int conv3x3_c8_impl(const char* fn, const void* xp, const void* wgt, void* out, long long ldd, int n, int h, int w, int cout,
                           int cout_valid, const fie_epilogue* ep, int out_dtype, void* stream) {
    FIE_REQUIRE(xp && wgt && out, "%s: null pointer", fn);
    FIE_REQUIRE(n > 0 && h > 0 && w > 0 && cout > 0 && (cout % 32) == 0, "%s: bad shape (cout must be a multiple of 32)", fn);
    int bw = 0, bh = 0, bn = 0;
    const bool boxed = box_tile(w, h, &bw, &bh, &bn);
    GemmParams p;
    memset(&p, 0, sizeof(p));
    const long long M = (long long)n * h * w;
    int rc = fill_epilogue(p, ep, M, cout, out, ldd, out_dtype);
    if (rc) return rc;
    FIE_REQUIRE(p.act != FIE_ACT_GEGLU, "%s: GEGLU epilogue not supported for conv", fn);
    p.mode = boxed ? 1 : 3; p.M = M; p.N = cout; p.OH = h; p.OW = w;
    pick_config(M, cout, false, &p.cg, &p.block_n, &p.mt);
    p.num_m_blocks = (int)((M + BLOCK_M * p.cg * p.mt - 1) / (BLOCK_M * p.cg * p.mt));
    p.num_n_blocks = (cout + p.block_n - 1) / p.block_n;
    p.kb_per_tap = 1; p.num_kb = 6; p.kb_split = 6;     // 3 kernel rows x (hi, lo) weight parts, each one 64-wide K block on the same A window
    p.n_store = cout_valid > 0 ? cout_valid : cout;
    const uint32_t box[4] = {BLOCK_K, (uint32_t)bw, (uint32_t)bh, (uint32_t)bn};
    const uint64_t wp = (uint64_t)w + 8, hp = (uint64_t)h + 2;
    const uint64_t dims[4] = {BLOCK_K, (uint64_t)w, hp, (uint64_t)n};
    const uint64_t strides[3] = {16, wp * 16, hp * wp * 16};
    // im2col: the run walks the w start pixels of the h output rows (the view has h + 2 rows); the taps add the kernel row
    static const int lower[2] = {-1, -1}, upper[2] = {-1, -3};
    if ((rc = boxed ? make_tmap_f16(&p.a_maps[0], xp, 4, dims, strides, box) : make_tmap_im2col_f16(&p.a_maps[0], xp, dims, strides, lower, upper)))
        return rc;
    p.a_maps[1] = p.a_maps[0]; p.a_maps[2] = p.a_maps[0]; p.a_maps[3] = p.a_maps[0];
    for (int t = 0; t < 6; ++t) { p.tap_map[t] = 0; p.tap_dh[t] = (int8_t)(t >> 1); p.tap_dw[t] = 0; }   // padded row y + kh, padded pixel x
    const uint64_t bdims[2] = {(uint64_t)6 * BLOCK_K, (uint64_t)cout};
    const uint64_t bstr[1] = {(uint64_t)6 * BLOCK_K * 2};
    const uint32_t bbox[2] = {BLOCK_K, (uint32_t)(p.block_n / p.cg)};
    if ((rc = make_tmap_f16(&p.b_map, wgt, 2, bdims, bstr, bbox))) return rc;
    return launch(p, (cudaStream_t)stream);
}

extern "C" int fie_gemm_f16(const void* A, long long lda, const void* A1, long long lda1, int k_split, const void* B, void* D, long long ldd,
                            long long M, int N, int K, const fie_epilogue* ep, void* stream) {
    return gemm_impl("fie_gemm_f16", A, lda, A1, lda1, k_split, B, D, ldd, M, N, K, ep, 0, out_dtype_of(ep), stream);
}

extern "C" int fie_gemm_bf16(const void* A, long long lda, const void* A1, long long lda1, int k_split, const void* B, void* D, long long ldd,
                             long long M, int N, int K, const fie_epilogue* ep, int out_dtype, void* stream) {
    if (int rc = check_out_dtype("fie_gemm_bf16", ep, out_dtype)) return rc;
    return gemm_impl("fie_gemm_bf16", A, lda, A1, lda1, k_split, B, D, ldd, M, N, K, ep, 1, out_dtype, stream);
}

extern "C" int fie_conv3x3_f16(const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                               int cout_valid, int stride, int pad_mode, const fie_epilogue* ep, void* stream) {
    return conv3x3_impl("fie_conv3x3_f16", x, wgt, out, ldd, n, h, w, cin, cout, cout_valid, stride, pad_mode, ep, 0, out_dtype_of(ep), stream);
}

extern "C" int fie_conv3x3_bf16(const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                                int cout_valid, int stride, int pad_mode, const fie_epilogue* ep, int out_dtype, void* stream) {
    if (int rc = check_out_dtype("fie_conv3x3_bf16", ep, out_dtype)) return rc;
    return conv3x3_impl("fie_conv3x3_bf16", x, wgt, out, ldd, n, h, w, cin, cout, cout_valid, stride, pad_mode, ep, 1, out_dtype, stream);
}

extern "C" int fie_conv_up2x_f16(const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                                 const fie_epilogue* ep, void* stream) {
    return conv_up2x_impl("fie_conv_up2x_f16", x, wgt, out, ldd, n, h, w, cin, cout, ep, 0, out_dtype_of(ep), stream);
}

extern "C" int fie_conv_up2x_bf16(const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                                  const fie_epilogue* ep, int out_dtype, void* stream) {
    if (int rc = check_out_dtype("fie_conv_up2x_bf16", ep, out_dtype)) return rc;
    return conv_up2x_impl("fie_conv_up2x_bf16", x, wgt, out, ldd, n, h, w, cin, cout, ep, 1, out_dtype, stream);
}

extern "C" int fie_conv3x3_c8_f16(const void* xp, const void* wgt, void* out, long long ldd, int n, int h, int w, int cout,
                                  int cout_valid, const fie_epilogue* ep, void* stream) {
    return conv3x3_c8_impl("fie_conv3x3_c8_f16", xp, wgt, out, ldd, n, h, w, cout, cout_valid, ep, out_dtype_of(ep), stream);
}

extern "C" int fie_conv3x3_c8_bf16(const void* xp, const void* wgt, void* out, long long ldd, int n, int h, int w, int cout,
                                   int cout_valid, const fie_epilogue* ep, int out_dtype, void* stream) {
    if (int rc = check_out_dtype("fie_conv3x3_c8_bf16", ep, out_dtype)) return rc;
    return conv3x3_c8_impl("fie_conv3x3_c8_bf16", xp, wgt, out, ldd, n, h, w, cout, cout_valid, ep, out_dtype, stream);
}
