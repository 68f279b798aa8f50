// Flash-style attention for head_dim 64 on tcgen05 tensor cores (sm_100a).
// Replaces F.scaled_dot_product_attention (AttnProcessor2_0) for the UNet / ControlNet self- and cross-attention
// of the reference's edit path (diffusers call at reference src/pipeline.py:261-272).  No mask, scale 1/sqrt(d).
//
// One work item = TWO 128-row Q tiles of one (batch, head) sharing every K/V tile (3-stage TMA ring of 128-row tiles).
// Per Q tile q and K/V tile j:
//   S_q = Q_q K_j^T   tcgen05.mma 128x128x64 -> TMEM columns [128q, 128q+128)
//   softmax           one warpgroup per Q tile, one thread per row (TMEM lane == row: no cross-thread reductions),
//                     online max / sum with 4-way ILP; P_q written as packed fp16 back into TMEM (tcgen05.st, 64 columns):
//                     with d = 64 the Q K^T product alone reads shared memory at the SM's 128 B/clk, so a P tile that went
//                     through shared memory (32 KB written + 32 KB read per 128 x 128 tile) would make shared-memory
//                     bandwidth, not the tensor pipe or the exponentials, the limit
//   O_qj = P_q V_j    tcgen05.mma 128x64x128, A = P_q from TMEM, B = V consumed MN-major straight from its row-major TMA
//                     tile -> TMEM
//   TMEM columns: S_0 0-127, S_1 128-255, O_0 256-319, O_1 320-383, P_0 384-447, P_1 448-511
//   O_q accumulates in TMEM across K/V tiles; it is rescaled by exp2(m_old - m_new) (tcgen05.ld/st) only when the
//   running row max of a warp moved.
// The two warpgroups ping-pong: while one does its softmax the tensor core serves the other (FlashAttention-4 style).
// Warp roles (384 threads): w0 TMA producer, w1 MMA issuer, w2 TMEM allocator, w3 idle, w4-7 softmax(q=0), w8-11 softmax(q=1).
#include "tc_common.cuh"
#include <type_traits>

namespace fie {

constexpr int ATT_EMU = 2;     // exponentials per 8 evaluated without MUFU in the self-attention softmax

// 2^x for x <= 127 without the MUFU unit: x = n + f (add with round-down against 1.5 * 2^23 leaves n in the low mantissa bits),
// 2^f by a cubic on [0, 1) (relative error ~1e-4), exponent patched in with an integer add.  Inputs below -126 give ~1e-38.
__device__ __forceinline__ float ex2_emulated(float x) {
    x = fmaxf(x, -126.0f);
    float t;
    asm("add.rm.ftz.f32 %0, %1, %2;" : "=f"(t) : "f"(x), "f"(12582912.0f));
    const float f = x - (t - 12582912.0f);
    const float p = fmaf(fmaf(fmaf(0.0771190897f, f, 0.2275643945f), f, 0.6951461434f), f, 1.0f);
    return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}

// 2^x of a column pair without the MUFU unit (see ex2_emulated): x2 must already be clamped to >= -126.
__device__ __forceinline__ void ex2_emulated2(f32x2 x2, float& p0, float& p1) {
    const f32x2 magic = pack2(12582912.0f, 12582912.0f);
    const f32x2 t = fadd2_rm(x2, magic);
    const f32x2 f = fsub2(x2, fsub2(t, magic));
    f32x2 q = ffma2(pack2(0.0771190897f, 0.0771190897f), f, pack2(0.2275643945f, 0.2275643945f));
    q = ffma2(q, f, pack2(0.6951461434f, 0.6951461434f));
    q = ffma2(q, f, pack2(1.0f, 1.0f));
    float q0, q1, t0, t1;
    unpack2(q, q0, q1); unpack2(t, t0, t1);
    p0 = __int_as_float(__float_as_int(q0) + (__float_as_int(t0) << 23));
    p1 = __int_as_float(__float_as_int(q1) + (__float_as_int(t1) << 23));
}


// O row (64 fp32 accumulators of one thread = one query row) * 1/l -> 64 fp16 = 128 contiguous bytes of the output.
// 256-bit stores (one full 32-byte sector per instruction) when the row is 32-byte aligned, else 128-bit ones.
__device__ __forceinline__ void store_o_row(__half* orow, const uint32_t (&r)[64], float inv_l, bool wide) {
    if (wide) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            uint32_t o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int e = u * 16 + 2 * i;
                const __half2 h = __floats2half2_rn(__uint_as_float(r[e]) * inv_l, __uint_as_float(r[e + 1]) * inv_l);
                o[i] = *reinterpret_cast<const uint32_t*>(&h);
            }
            stg256(orow + u * 16, o);
        }
    } else {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            uint4 v; __half2* hh = reinterpret_cast<__half2*>(&v);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int e = u * 8 + 2 * i;
                hh[i] = __floats2half2_rn(__uint_as_float(r[e]) * inv_l, __uint_as_float(r[e + 1]) * inv_l);
            }
            *reinterpret_cast<uint4*>(orow + u * 8) = v;
        }
    }
}

constexpr int ATT_BM = 128, ATT_BN = 128, ATT_D = 64, ATT_QT = 2;
constexpr int ATT_TILE_BYTES = 128 * 64 * 2;                                   // 16 KiB (Q, K or V tile)

struct AttnParams {
    CUtensorMap q_map, k_map, v_map;
    __half* out;
    long long ldo;
    int nq, nkv;
    float scale_log2;
    int causal;       // (kv1 kernel only) key j is visible to query row i iff j <= i
};

// ------------------------------------------------------------------------------------------------
// Self-attention (nkv > 128), persistent.  With 1024 keys a CTA per (batch, head, 256-row query block) item would live for 8 K/V
// steps (~12 us of steady state) and pay ~5 us of set-up and drain around them: block scheduling, barrier init, the 512-column TMEM
// allocation, the first Q / K / V round trip, the O read-out and store.  Here <= 148 CTAs each walk a strided list of items with
// everything allocated once: the producer runs ahead across items (Q is double-buffered, the K/V ring simply continues), the MMA
// warp issues S = Q K^T for the FIRST tile of the next item as soon as the last tile of the current one has been consumed, and a
// softmax warpgroup goes from the epilogue of one item straight into scores that are already waiting in TMEM.
// Barrier parities follow GLOBAL counters (tiles processed by this CTA), not per-item ones.  No extra barrier protects O_q / P_q across
// items: a softmax warpgroup reads O_q of item n (epilogue) before it arrives on p_full for the first tile of item n + 1, and the MMA
// warp only overwrites O_q / reads P_q after that arrival.
// ------------------------------------------------------------------------------------------------
constexpr int ATTP_KV_STAGES = 3;                                                 // K/V ring depth (prefetch distance across items)
constexpr int ATTP_OFF_KV = 2 * ATT_QT * ATT_TILE_BYTES;                          // after Q[2 buffers][2 tiles]
constexpr int ATTP_OFF_BAR = ATTP_OFF_KV + ATTP_KV_STAGES * 2 * ATT_TILE_BYTES;
constexpr int ATTP_SMEM = ATTP_OFF_BAR + 256;

__global__ void __launch_bounds__(384, 1) k_attention_d64_p(const __grid_constant__ AttnParams p, int heads, int batch) {
    extern __shared__ __align__(1024) uint8_t smem[];
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // persistent grid (<= 1 CTA per SM): the next kernel may start launching (see gemm_conv.cu)
    uint8_t* sQ = smem;                                   // buffer u: Q tiles at u * 32K
    uint8_t* sKV = smem + ATTP_OFF_KV;                    // stage s: K at s*32K, V at s*32K + 16K
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ATTP_OFF_BAR);
    uint64_t* q_full = bars;                 // [2]
    uint64_t* q_empty = bars + 2;            // [2]
    uint64_t* kv_full = bars + 4;                          // [ATTP_KV_STAGES]
    uint64_t* kv_empty = kv_full + ATTP_KV_STAGES;         // [ATTP_KV_STAGES]
    uint64_t* s_full = kv_empty + ATTP_KV_STAGES;          // [2]
    uint64_t* p_full = s_full + 2;                         // [2]
    uint64_t* o_full = p_full + 2;                         // [2]
    uint64_t* s_free = o_full + 2;                         // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_free + 2);
    if ((smem_u32(smem) & 1023u) != 0) { if (threadIdx.x == 0) printf("fie: attention smem base misaligned\n"); __trap(); }

    const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;
    const int nqp = (p.nq + ATT_QT * ATT_BM - 1) / (ATT_QT * ATT_BM);
    const int items = batch * heads * nqp;
    const int n_tiles = (p.nkv + ATT_BN - 1) / ATT_BN;
    const int my_items = blockIdx.x < (unsigned)items ? (items - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;   // items blockIdx.x, + gridDim.x, ...

    if (threadIdx.x == 0) {
        for (int u = 0; u < 2; ++u) { mbar_init(&q_full[u], 1); mbar_init(&q_empty[u], 1); }
        for (int s = 0; s < ATTP_KV_STAGES; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1); }
        for (int q = 0; q < ATT_QT; ++q) { mbar_init(&s_full[q], 1); mbar_init(&p_full[q], 128); mbar_init(&o_full[q], 1); mbar_init(&s_free[q], 128); }
        mbar_fence_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.q_map); tma_prefetch_desc(&p.k_map); tma_prefetch_desc(&p.v_map); }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (elect_one_sync()) {
            int s = 0; uint32_t ph = 0;
            for (int n = 0; n < my_items; ++n) {
                const int it = (int)blockIdx.x + n * (int)gridDim.x;
                const int qp = it % nqp, head = (it / nqp) % heads, b = it / (nqp * heads);
                const int u = n & 1;
                mbar_wait(&q_empty[u], (uint32_t)(((n >> 1) & 1) ^ 1));
                mbar_arrive_expect_tx(&q_full[u], ATT_QT * ATT_TILE_BYTES);
                for (int q = 0; q < ATT_QT; ++q)
                    tma_load_3d(&p.q_map, &q_full[u], sQ + (u * ATT_QT + q) * ATT_TILE_BYTES, head * ATT_D, (qp * ATT_QT + q) * ATT_BM, b);
                for (int j = 0; j < n_tiles; ++j) {
                    mbar_wait(&kv_empty[s], ph ^ 1);
                    mbar_arrive_expect_tx(&kv_full[s], 2 * ATT_TILE_BYTES);
                    tma_load_3d(&p.k_map, &kv_full[s], sKV + s * 2 * ATT_TILE_BYTES, head * ATT_D, j * ATT_BN, b);
                    tma_load_3d(&p.v_map, &kv_full[s], sKV + s * 2 * ATT_TILE_BYTES + ATT_TILE_BYTES, head * ATT_D, j * ATT_BN, b);
                    if (++s == ATTP_KV_STAGES) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        const uint32_t idesc_qk = umma_idesc_f16(ATT_BM, ATT_BN, 0, 0);
        const uint32_t idesc_pv = umma_idesc_f16(ATT_BM, ATT_D, 0, 1);   // B (= V) is MN-major
        const uint32_t aQ = smem_u32(sQ), aKV = smem_u32(sKV);
        // S_q = Q_q(buffer u) K_s^T; `last` = this is the item's last Q K^T: its completion releases the Q buffer
        auto issue_qk = [&](int q, int s, int u, bool last) {
            if (elect_one_sync()) {
                const uint64_t ad = umma_desc_sw128(aQ + (u * ATT_QT + q) * ATT_TILE_BYTES), bd = umma_desc_sw128(aKV + s * 2 * ATT_TILE_BYTES);
#pragma unroll
                for (int k = 0; k < ATT_D / 16; ++k) umma_f16(tmem + q * 128, ad + 2 * k, bd + 2 * k, idesc_qk, k ? 1u : 0u);
                umma_commit(&s_full[q]);
                if (last && q == ATT_QT - 1) umma_commit(&q_empty[u]);
            }
            __syncwarp();
        };
        if (my_items > 0) {
            mbar_wait(&q_full[0], 0);
            mbar_wait(&kv_full[0], 0);
            tc_fence_after();
            issue_qk(0, 0, 0, n_tiles == 1);
            issue_qk(1, 0, 0, n_tiles == 1);
        }
        int s = 0; uint32_t ph = 0;                 // stage / phase of the current tile
        uint32_t g = 0;                             // tiles processed by this CTA: parity source of the per-tile barriers
        for (int n = 0; n < my_items; ++n) {
            for (int j = 0; j < n_tiles; ++j, ++g) {
                int sn = s + 1; uint32_t phn = ph; if (sn == ATTP_KV_STAGES) { sn = 0; phn ^= 1; }
                // S_q(j+1) = Q_q K_{j+1}^T is issued as soon as the softmax warps hold S_q(j) in registers, i.e. while they are
                // still exponentiating it: the next scores are ready when P_q(j) is, and the softmax never waits on the tensor pipe.
                const bool next_same = j + 1 < n_tiles, next_item = !next_same && n + 1 < my_items;
                if (next_same || next_item) {
                    const int un = next_same ? (n & 1) : ((n + 1) & 1);
                    if (next_item) mbar_wait(&q_full[un], (uint32_t)(((n + 1) >> 1) & 1));
                    mbar_wait(&kv_full[sn], phn);
                    const bool last_qk = next_same ? (j + 2 == n_tiles) : (n_tiles == 1);
                    for (int q = 0; q < ATT_QT; ++q) {
                        mbar_wait(&s_free[q], g & 1u);
                        tc_fence_after();
                        issue_qk(q, sn, un, last_qk);
                    }
                }
                for (int q = 0; q < ATT_QT; ++q) {
                    mbar_wait(&p_full[q], g & 1u);
                    tc_fence_after();
                    if (elect_one_sync()) {
                        const uint32_t aV = aKV + s * 2 * ATT_TILE_BYTES + ATT_TILE_BYTES;
#pragma unroll
                        for (int k = 0; k < ATT_BN / 16; ++k) {
                            const uint64_t bd = umma_desc_sw128(aV + k * 2048, 1024, 1024);
                            umma_f16_ts(tmem + 256 + q * 64, tmem + 384 + q * 64 + k * 8, bd, idesc_pv, (j | k) ? 1u : 0u);   // O restarts with every item
                        }
                        umma_commit(&o_full[q]);
                        if (q == ATT_QT - 1) umma_commit(&kv_empty[s]);
                    }
                    __syncwarp();
                }
                s = sn; ph = phn;
            }
        }
    } else if (warp >= 4) {
        // ===================== softmax / epilogue: warpgroup = Q tile, thread = row =====================
        const int q = (warp - 4) >> 2;
        const int wq = warp & 3;                          // TMEM lane quadrant of this warp
        const int row = wq * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(wq * 32) << 16;
        const uint32_t tS = tmem + q * 128 + lane_addr, tO = tmem + 256 + q * 64 + lane_addr, tP = tmem + 384 + q * 64 + lane_addr;
        const float sl2 = p.scale_log2;
        const bool wide_o = (p.ldo & 15) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 31) == 0;   // 32-byte aligned output rows
        // exp2 of one 64-column half against the reference max folded into mneg -> packed fp16 in pp (the A operand layout of
        // P V: two columns per 32-bit TMEM column); returns the row sum of the half.  FULL: no column masking.  WITH_MAX: also
        // folds the raw scores into the four running-max accumulators mx[] (one FMNMX3 per column pair), so that the maximum
        // search rides in the issue slots the MUFU-bound exponentials leave free.
        auto exp_cols = [&](const uint32_t* r, int col0, float mneg, int kv_left, auto full_c, auto max_c, auto nu_c, uint32_t* pp, float (&mx)[4]) -> float {
            constexpr bool FULL = decltype(full_c)::value;
            constexpr bool WITH_MAX = decltype(max_c)::value;
            constexpr int NU = decltype(nu_c)::value;           // units of 8 columns: 8 (a 64-column half) or 4
            f32x2 psa = 0ull, psb = 0ull;                       // four partial row sums as two packed accumulators (0 bits == +0.f pair)
            const f32x2 sl22 = pack2(sl2, sl2), mneg2 = pack2(mneg, mneg);
#pragma unroll
            for (int u = 0; u < NU; ++u) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int c = u * 8 + 2 * i;
                    // The MUFU unit (16 ex2 / clk / SM) and the issue slots are this kernel's limits: ATT_EMU of every 8
                    // exponentials run on the FMA / ALU pipes instead (Cody-Waite split + cubic, ~1e-4 relative: below the fp16
                    // rounding of P), as packed column pairs.
                    if (WITH_MAX) {
                        if (FULL) mx[i] = fmaxf(fmaxf(mx[i], __uint_as_float(r[c])), __uint_as_float(r[c + 1]));
                        else { if (col0 + c < kv_left) mx[i] = fmaxf(mx[i], __uint_as_float(r[c])); if (col0 + c + 1 < kv_left) mx[i] = fmaxf(mx[i], __uint_as_float(r[c + 1])); }
                    }
                    const f32x2 x2 = ffma2(pack2u(r[c], r[c + 1]), sl22, mneg2);
                    float x0, x1, p0, p1;
                    unpack2(x2, x0, x1);
                    if (2 * i >= 8 - ATT_EMU) ex2_emulated2(pack2(fmaxf(x0, -126.0f), fmaxf(x1, -126.0f)), p0, p1);
                    else { p0 = ex2_approx(x0); p1 = ex2_approx(x1); }
                    if (!FULL) { if (col0 + c >= kv_left) p0 = 0.f; if (col0 + c + 1 >= kv_left) p1 = 0.f; }
                    if (i & 1) psb = fadd2(psb, pack2(p0, p1)); else psa = fadd2(psa, pack2(p0, p1));
                    __half2 h = __floats2half2_rn(p0, p1);
                    pp[4 * u + i] = *reinterpret_cast<uint32_t*>(&h);
                }
            }
            float s0, s1;
            unpack2(fadd2(psa, psb), s0, s1);
            return s0 + s1;
        };
        auto half_max = [&](const uint32_t (&r)[64], int hf, int kv_left, bool full_tile, float (&mx)[4]) {
            if (full_tile) {
#pragma unroll
                for (int i = 0; i < 64; i += 8) {                      // 3-input max (FMNMX3): two columns per instruction
                    mx[0] = fmaxf(fmaxf(mx[0], __uint_as_float(r[i])), __uint_as_float(r[i + 1])); mx[1] = fmaxf(fmaxf(mx[1], __uint_as_float(r[i + 2])), __uint_as_float(r[i + 3]));
                    mx[2] = fmaxf(fmaxf(mx[2], __uint_as_float(r[i + 4])), __uint_as_float(r[i + 5])); mx[3] = fmaxf(fmaxf(mx[3], __uint_as_float(r[i + 6])), __uint_as_float(r[i + 7]));
                }
            } else {
#pragma unroll
                for (int i = 0; i < 64; ++i) if (hf * 64 + i < kv_left) mx[0] = fmaxf(mx[0], __uint_as_float(r[i]));
            }
        };
        const std::true_type yes{}; const std::false_type no{};
        const std::integral_constant<int, 8> n8{}; const std::integral_constant<int, 4> n4{};
        uint32_t g = 0;                                   // tiles processed: parity of s_full / o_full
        for (int n = 0; n < my_items; ++n) {
            const int it = (int)blockIdx.x + n * (int)gridDim.x;
            const int qp = it % nqp, head = (it / nqp) % heads, b = it / (nqp * heads);
            float m_run = -INFINITY, l_run = 0.f;
            for (int j = 0; j < n_tiles; ++j, ++g) {
                mbar_wait(&s_full[q], g & 1u);
                tc_fence_after();
                const int kv_left = p.nkv - j * ATT_BN;     // valid columns in this tile
                const bool full_tile = kv_left >= ATT_BN;
                // Optimistic single pass: the exponentials of the first half are taken against the CURRENT reference max while the
                // tile's row maximum is still being searched.  The reference only has to move when a row maximum outgrows it by more
                // than 2^8 in the exponent domain (P = exp2((s - m_run) * scale) <= 256 still fits fp16, and O / l stays exact because
                // both are accumulated against the same reference) -- after the first tile that is rare, and then the first half is
                // simply redone.
                float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
                uint32_t pp0[32];
                float psum = 0.f;
                {
                    uint32_t ra[64];
                    tmem_ld_32x64(tS, ra);
                    tmem_ld_wait();
                    if (j == 0) half_max(ra, 0, kv_left, full_tile, mx4);
                    else if (full_tile) psum = exp_cols(ra, 0, -m_run * sl2, kv_left, yes, yes, n8, pp0, mx4);
                    else psum = exp_cols(ra, 0, -m_run * sl2, kv_left, no, yes, n8, pp0, mx4);
                }
                uint32_t rb[64];
                tmem_ld_32x64(tS + 64, rb);
                tmem_ld_wait();
                half_max(rb, 1, kv_left, full_tile, mx4);
                const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
                const bool move = (j == 0) || ((mx - m_run) * sl2 > 8.0f);
                float alpha = 1.0f;
                if (j > 0) {                                // P_q and O_q are free once PV(q, previous tile) has completed
                    mbar_wait(&o_full[q], (g - 1) & 1u);
                    tc_fence_after();
                }
                if (__any_sync(0xffffffffu, move)) {
                    // the reference max of some row of this warp moves (always on the first tile): rescale O_q, which lives in TMEM,
                    // by exp2(m_old - m_new), and (re)do the first half against the new reference
                    if (move) { alpha = ex2_approx((m_run - fmaxf(mx, m_run)) * sl2); m_run = fmaxf(mx, m_run); }      // first tile: exp2(-inf) = 0
                    // (32 columns at a time: this rare path must not raise the register pressure of the common one)
                    if (j > 0) {
#pragma unroll 1
                        for (int hq = 0; hq < 2; ++hq) {
                            uint32_t ro[32];
                            tmem_ld_32x32(tO + (uint32_t)(hq * 32), ro);
                            tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 32; ++i) ro[i] = __float_as_uint(__uint_as_float(ro[i]) * alpha);
                            tmem_st_32x32(tO + (uint32_t)(hq * 32), ro);
                        }
                    }
                    float dummy[4];
                    psum = 0.f;
#pragma unroll
                    for (int hq = 0; hq < 2; ++hq) {
                        uint32_t rq[32];
                        tmem_ld_32x32(tS + (uint32_t)(hq * 32), rq);
                        tmem_ld_wait();
                        if (full_tile) psum += exp_cols(rq, hq * 32, -m_run * sl2, kv_left, yes, no, n4, pp0 + hq * 16, dummy);
                        else psum += exp_cols(rq, hq * 32, -m_run * sl2, kv_left, no, no, n4, pp0 + hq * 16, dummy);
                    }
                }
                tmem_st_32x32(tP, pp0);
                tc_fence_before();
                mbar_arrive(&s_free[q]);                      // S_q has been consumed: Q_q K_{j+1}^T may be issued now
                {
                    uint32_t pp1[32];
                    float dummy[4];
                    if (full_tile) psum += exp_cols(rb, 64, -m_run * sl2, kv_left, yes, no, n8, pp1, dummy);
                    else psum += exp_cols(rb, 64, -m_run * sl2, kv_left, no, no, n8, pp1, dummy);
                    tmem_st_32x32(tP + 32u, pp1);
                }
                l_run = l_run * alpha + psum;
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(&p_full[q]);
            }
            // ---- epilogue of this item: O_q / l -> global (g already counts the item's last tile) ----
            mbar_wait(&o_full[q], (g - 1) & 1u);
            tc_fence_after();
            const float inv_l = 1.0f / l_run;
            const int qrow = (qp * ATT_QT + q) * ATT_BM + row;
            __half* orow = p.out + ((long long)b * p.nq + qrow) * p.ldo + head * ATT_D;
            {
                uint32_t r[64];
                tmem_ld_32x64(tO, r);
                tmem_ld_wait();
                tc_fence_before();                          // the O_q read is complete before this thread's next p_full arrive lets the MMA warp overwrite it
                if (qrow < p.nq) store_o_row(orow, r, inv_l, wide_o);
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ------------------------------------------------------------------------------------------------
// Cross-attention form (nkv <= 128: the 77 prompt tokens): one K/V tile, so the work per (batch, head, 256 query rows) is a
// short latency chain (Q K^T -> softmax -> P V -> store) and one CTA per item would spend most of its life in set-up.
// Here 148 persistent CTAs each walk a contiguous range of items; the producer keeps the next item's Q / K / V in flight in a
// second shared-memory buffer, and TMEM allocation, barrier set-up and descriptor fetches are paid once per CTA.
// Same warp roles as k_attention_d64_p.  Barriers flip once per item (parity = item counter & 1).
// ------------------------------------------------------------------------------------------------
constexpr int ATT1_OFF_KV = 2 * ATT_QT * ATT_TILE_BYTES;                       // after Q[2 buffers][2 tiles]
constexpr int ATT1_OFF_P = ATT1_OFF_KV + 2 * 2 * ATT_TILE_BYTES;               // after K/V[2 buffers]
constexpr int ATT1_OFF_BAR = ATT1_OFF_P + ATT_QT * 32768;
constexpr int ATT1_SMEM = ATT1_OFF_BAR + 256;

__global__ void __launch_bounds__(384, 1) k_attention_d64_kv1(const __grid_constant__ AttnParams p, int heads, int batch) {
    extern __shared__ __align__(1024) uint8_t smem[];
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // persistent grid (<= 1 CTA per SM): the next kernel may start launching (see gemm_conv.cu)
    uint8_t* sQ = smem;                                   // buffer u: Q tiles at u * 32K
    uint8_t* sKV = smem + ATT1_OFF_KV;                    // buffer u: K at u * 32K, V at u * 32K + 16K
    uint8_t* sP = smem + ATT1_OFF_P;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ATT1_OFF_BAR);
    uint64_t* ld_full = bars;                // [2] Q + K + V of an item landed
    uint64_t* ld_empty = bars + 2;           // [2] both P V of the item completed: its buffer may be refilled
    uint64_t* s_full = bars + 4;             // [2]
    uint64_t* p_full = bars + 6;             // [2]
    uint64_t* o_full = bars + 8;             // [2]
    uint64_t* o_free = bars + 10;            // [2] S_q and O_q have been read: the next item may overwrite them
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
    if ((smem_u32(smem) & 1023u) != 0) { if (threadIdx.x == 0) printf("fie: attention smem base misaligned\n"); __trap(); }

    const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;
    const int nqp = (p.nq + ATT_QT * ATT_BM - 1) / (ATT_QT * ATT_BM);          // 256-row query blocks per (batch, head)
    const int items = batch * heads * nqp;
    const int per = (items + gridDim.x - 1) / gridDim.x;
    const int it0 = blockIdx.x * per, it1 = min(it0 + per, items);

    if (threadIdx.x == 0) {
        for (int u = 0; u < 2; ++u) {
            mbar_init(&ld_full[u], 1); mbar_init(&ld_empty[u], 1);
            mbar_init(&s_full[u], 1); mbar_init(&p_full[u], 128); mbar_init(&o_full[u], 1); mbar_init(&o_free[u], 128);
        }
        mbar_fence_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.q_map); tma_prefetch_desc(&p.k_map); tma_prefetch_desc(&p.v_map); }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    asm volatile("griddepcontrol.wait;" ::: "memory");      // programmatic dependent launch: the prologue above overlaps the previous kernel's tail
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (elect_one_sync()) {
            for (int it = it0, n = 0; it < it1; ++it, ++n) {
                const int u = n & 1; const uint32_t ph = (uint32_t)((n >> 1) & 1);
                const int qp = it % nqp, head = (it / nqp) % heads, b = it / (nqp * heads);
                mbar_wait(&ld_empty[u], ph ^ 1);
                mbar_arrive_expect_tx(&ld_full[u], (ATT_QT + 2) * ATT_TILE_BYTES);
                for (int q = 0; q < ATT_QT; ++q)
                    tma_load_3d(&p.q_map, &ld_full[u], sQ + (u * ATT_QT + q) * ATT_TILE_BYTES, head * ATT_D, (qp * ATT_QT + q) * ATT_BM, b);
                tma_load_3d(&p.k_map, &ld_full[u], sKV + u * 2 * ATT_TILE_BYTES, head * ATT_D, 0, b);
                tma_load_3d(&p.v_map, &ld_full[u], sKV + u * 2 * ATT_TILE_BYTES + ATT_TILE_BYTES, head * ATT_D, 0, b);
            }
        }
    } else if (warp == 1) {
        const uint32_t idesc_qk = umma_idesc_f16(ATT_BM, ATT_BN, 0, 0);
        const uint32_t idesc_pv = umma_idesc_f16(ATT_BM, ATT_D, 0, 1);   // B (= V) is MN-major
        const uint32_t aQ = smem_u32(sQ), aP = smem_u32(sP), aKV = smem_u32(sKV);
        for (int it = it0, n = 0; it < it1; ++it, ++n) {
            const int u = n & 1; const uint32_t ph = (uint32_t)((n >> 1) & 1), par = (uint32_t)(n & 1);
            mbar_wait(&ld_full[u], ph);
            for (int q = 0; q < ATT_QT; ++q) {
                if (n > 0) mbar_wait(&o_free[q], par ^ 1);             // previous item's S_q / O_q consumed
                tc_fence_after();
                if (elect_one_sync()) {
                    const uint64_t ad = umma_desc_sw128(aQ + (u * ATT_QT + q) * ATT_TILE_BYTES), bd = umma_desc_sw128(aKV + u * 2 * ATT_TILE_BYTES);
#pragma unroll
                    for (int k = 0; k < ATT_D / 16; ++k) umma_f16(tmem + q * 128, ad + 2 * k, bd + 2 * k, idesc_qk, k ? 1u : 0u);
                    umma_commit(&s_full[q]);
                }
                __syncwarp();
            }
            for (int q = 0; q < ATT_QT; ++q) {
                mbar_wait(&p_full[q], par);
                tc_fence_after();
                if (elect_one_sync()) {
                    const uint32_t aV = aKV + u * 2 * ATT_TILE_BYTES + ATT_TILE_BYTES;
#pragma unroll
                    for (int k = 0; k < ATT_BN / 16; ++k) {
                        if (k * 16 >= p.nkv) break;                       // P columns / V rows beyond nkv contribute nothing
                        const uint64_t ad = umma_desc_sw128(aP + q * 32768 + (k >> 2) * 16384 + (k & 3) * 32);
                        const uint64_t bd = umma_desc_sw128(aV + k * 2048, 1024, 1024);
                        umma_f16(tmem + 256 + q * 64, ad, bd, idesc_pv, k ? 1u : 0u);
                    }
                    umma_commit(&o_full[q]);
                    if (q == ATT_QT - 1) umma_commit(&ld_empty[u]);
                }
                __syncwarp();
            }
        }
    } else if (warp >= 4) {
        const int q = (warp - 4) >> 2;
        const int wq = warp & 3;
        const int row = wq * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(wq * 32) << 16;
        const uint32_t tS = tmem + q * 128 + lane_addr, tO = tmem + 256 + q * 64 + lane_addr;
        const float sl2 = p.scale_log2;
        const bool wide_o = (p.ldo & 15) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 31) == 0;   // 32-byte aligned output rows
        uint8_t* prow = sP + q * 32768 + row * 128;
        const int sw = row & 7;
        const int kv = p.nkv;                                 // <= 128 valid columns
        const int kv16 = (kv + 15) & ~15;
        for (int it = it0, n = 0; it < it1; ++it, ++n) {
            const uint32_t par = (uint32_t)(n & 1);
            const int qp = it % nqp, head = (it / nqp) % heads, b = it / (nqp * heads);
            mbar_wait(&s_full[q], par);
            tc_fence_after();
            uint32_t ra[64], rb[64];
            tmem_ld_32x64(tS, ra);
            tmem_ld_32x64(tS + 64, rb);
            tmem_ld_wait();
            const int kvr = p.causal ? min(kv, (qp * ATT_QT + q) * ATT_BM + row + 1) : kv;       // columns visible to this row
            float mx = -INFINITY;
#pragma unroll
            for (int i = 0; i < 64; ++i) { if (i < kvr) mx = fmaxf(mx, __uint_as_float(ra[i])); if (64 + i < kvr) mx = fmaxf(mx, __uint_as_float(rb[i])); }
            const float mneg = -mx * sl2;
            float l = 0.f;
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                uint8_t* base = prow + hf * 16384;
#pragma unroll
                for (int uu = 0; uu < 8; ++uu) {
                    if (hf * 64 + uu * 8 >= kv16) break;          // 16-column K blocks beyond nkv are never read by the P V MMAs
                    uint32_t pk[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int c = uu * 8 + 2 * i;
                        const float s0 = __uint_as_float(hf ? rb[c] : ra[c]), s1 = __uint_as_float(hf ? rb[c + 1] : ra[c + 1]);
                        float p0 = (hf * 64 + c < kvr) ? ex2_approx(fmaf(s0, sl2, mneg)) : 0.f;
                        float p1 = (hf * 64 + c + 1 < kvr) ? ex2_approx(fmaf(s1, sl2, mneg)) : 0.f;
                        l += p0 + p1;
                        __half2 h = __floats2half2_rn(p0, p1);
                        pk[i] = *reinterpret_cast<uint32_t*>(&h);
                    }
                    *reinterpret_cast<uint4*>(base + ((uu ^ sw) * 16)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
            fence_proxy_async_smem();
            tc_fence_before();
            mbar_arrive(&p_full[q]);
            mbar_wait(&o_full[q], par);
            tc_fence_after();
            uint32_t r[64];
            tmem_ld_32x64(tO, r);
            tmem_ld_wait();
            tc_fence_before();
            mbar_arrive(&o_free[q]);                              // S_q (read above) and O_q are in registers
            const float inv_l = 1.0f / l;
            const int qrow = (qp * ATT_QT + q) * ATT_BM + row;
            if (qrow < p.nq) store_o_row(p.out + ((long long)b * p.nq + qrow) * p.ldo + head * ATT_D, r, inv_l, wide_o);
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

}  // namespace fie
using namespace fie;

static int attention_d64(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                         void* out, long long ldo, int b, int heads, int nq, int nkv, float scale, int causal, void* stream) {
    FIE_REQUIRE(q && k && v && out, "fie_attention_d64_f16: null pointer");
    FIE_REQUIRE(b > 0 && heads > 0 && nq > 0 && nkv > 0 && b <= 65535 && heads <= 65535, "fie_attention_d64_f16: bad shape");
    FIE_REQUIRE((ldq % 8) == 0 && (ldk % 8) == 0 && (ldv % 8) == 0 && (ldo % 8) == 0, "fie_attention_d64_f16: leading dims must be multiples of 8");
    FIE_REQUIRE(ldq >= heads * 64 && ldk >= heads * 64 && ldv >= heads * 64 && ldo >= heads * 64, "fie_attention_d64_f16: leading dim < heads*64");
    AttnParams p;
    memset(&p, 0, sizeof(p));
    const uint32_t box[3] = {64, 128, 1};
    int rc;
    {
        const uint64_t dims[3] = {(uint64_t)heads * 64, (uint64_t)nq, (uint64_t)b};
        const uint64_t str[2] = {(uint64_t)ldq * 2, (uint64_t)nq * ldq * 2};
        if ((rc = make_tmap_f16(&p.q_map, q, 3, dims, str, box))) return rc;
    }
    {
        const uint64_t dims[3] = {(uint64_t)heads * 64, (uint64_t)nkv, (uint64_t)b};
        const uint64_t strk[2] = {(uint64_t)ldk * 2, (uint64_t)nkv * ldk * 2};
        const uint64_t strv[2] = {(uint64_t)ldv * 2, (uint64_t)nkv * ldv * 2};
        if ((rc = make_tmap_f16(&p.k_map, k, 3, dims, strk, box))) return rc;
        if ((rc = make_tmap_f16(&p.v_map, v, 3, dims, strv, box))) return rc;
    }
    p.out = (__half*)out; p.ldo = ldo; p.nq = nq; p.nkv = nkv;
    p.scale_log2 = scale * 1.4426950408889634f;
    p.causal = causal;
    FIE_REQUIRE(!causal || nkv <= ATT_BN, "fie_attention_d64_causal_f16: nkv must be <= 128");
    cudaLaunchAttribute pdl_attr[1];                      // programmatic dependent launch (see gemm_conv.cu)
    pdl_attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl_attr[0].val.programmaticStreamSerializationAllowed = 1;
    const long long items = (long long)b * heads * ((nq + ATT_QT * ATT_BM - 1) / (ATT_QT * ATT_BM));
    const int sms = device_sm_count();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(items < sms ? items : sms)); cfg.blockDim = dim3(384); cfg.stream = (cudaStream_t)stream;
    cfg.attrs = pdl_attr; cfg.numAttrs = 1;
    if (nkv <= ATT_BN) {
        // cross-attention: one K/V tile per item
        static bool attr1_dev[kMaxDevices] = {false};               // cudaFuncSetAttribute is per device
        bool& attr1 = attr1_dev[current_device()];
        if (!attr1) {
            cudaError_t e = cudaFuncSetAttribute(k_attention_d64_kv1, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT1_SMEM);
            if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(k_attention_d64_kv1): %s", cudaGetErrorString(e)); return FIE_ERR_CUDA; }
            attr1 = true;
        }
        cfg.dynamicSmemBytes = ATT1_SMEM;
        cudaError_t e = cudaLaunchKernelEx(&cfg, k_attention_d64_kv1, p, heads, b);
        if (e != cudaSuccess) { set_error("cudaLaunchKernelEx(k_attention_d64_kv1): %s", cudaGetErrorString(e)); cudaGetLastError(); return FIE_ERR_CUDA; }
        return check_launch("fie_attention_d64_f16");
    }
    static bool attrp_dev[kMaxDevices] = {false};
    bool& attrp = attrp_dev[current_device()];
    if (!attrp) {
        cudaError_t e = cudaFuncSetAttribute(k_attention_d64_p, cudaFuncAttributeMaxDynamicSharedMemorySize, ATTP_SMEM);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(k_attention_d64_p): %s", cudaGetErrorString(e)); return FIE_ERR_CUDA; }
        attrp = true;
    }
    cfg.dynamicSmemBytes = ATTP_SMEM;
    cudaError_t e = cudaLaunchKernelEx(&cfg, k_attention_d64_p, p, heads, b);
    if (e != cudaSuccess) { set_error("cudaLaunchKernelEx(k_attention_d64_p): %s", cudaGetErrorString(e)); cudaGetLastError(); return FIE_ERR_CUDA; }
    return check_launch("fie_attention_d64_f16");
}

extern "C" int fie_attention_d64_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                                     void* out, long long ldo, int b, int heads, int nq, int nkv, float scale, void* stream) {
    return attention_d64(q, ldq, k, ldk, v, ldv, out, ldo, b, heads, nq, nkv, scale, 0, stream);
}
extern "C" int fie_attention_d64_causal_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                                            void* out, long long ldo, int b, int heads, int nq, int nkv, float scale, void* stream) {
    return attention_d64(q, ldq, k, ldk, v, ldv, out, ldo, b, heads, nq, nkv, scale, 1, stream);
}
