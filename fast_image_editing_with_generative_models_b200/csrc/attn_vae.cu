// AutoencoderKL mid-block attention (1 head, d = C = 512, N = H*W = 16 384 tokens at 1024^2): one C-ABI call.
// Replaces diffusers Attention / AttnProcessor2_0 inside UNetMidBlock2D of the VAE (F.scaled_dot_product_attention over a
// [1, N, 512] sequence; reference call site src/pipeline.py:261-272 -> AutoencoderKL.encode / decode).
//
// Why this is NOT a one-kernel flash attention (measured / derived, DESIGN.md 3.3): with d = 512 the fp32 output tile O[128 x 512]
// alone is all 512 TMEM columns and the Q tile is 128 KB of shared memory.  Splitting O over a CTA pair (256 columns each) forces the
// Q K^T reduction over d to be split too, and the partial scores to be exchanged through distributed shared memory at 32 KB per
// 64-key tile and direction; operand re-reads (Q half: 64 KB per tile), the exchange and the staging copies add up to ~290 KB of
// shared-memory traffic per 1024 clk of MMA, i.e. a shared-memory-bound kernel at <= 45 % of the tensor pipe -- no better than three
// passes of the persistent GEMM kernel, which is what this entry point launches:
//   S  = scale * Q K^T     k_gemm_conv, fp32 accumulation in TMEM, fp16 (or fp32) scores for `chunk_rows` query rows at a time
//   P' = exp(S - rowmax)   k_softmax_rows_exp (fp16 scores: exp-only, 1/rowsum on the side) or k_softmax_rows (fp32 scores)
//   O  = diag(1/rowsum) P' V   k_gemm_conv against V^T (K-major B operand), normalisation applied in fp32 by the epilogue
// With 180 GB of HBM a whole image's score matrix (512 MiB as fp16) is materialised at once, so the P V product runs as 128 tiles
// (1.7 waves of the 74 CTA pairs) instead of 32 tiles per 4096-row chunk.
#include "fie_common.cuh"

extern "C" size_t fie_attn_vae_workspace_bytes(int ntok, int chunk_rows, int f32_scores) {
    if (ntok <= 0) return 0;
    if (chunk_rows <= 0 || chunk_rows > ntok) chunk_rows = ntok;
    const size_t scores = (size_t)chunk_rows * ntok * (f32_scores ? 4 : 2);
    const size_t probs = f32_scores ? (size_t)chunk_rows * ntok * 2 : 0;      // fp32 scores are not softmaxed in place
    return ((scores + 255) / 256) * 256 + ((probs + 255) / 256) * 256 + (size_t)chunk_rows * sizeof(float) + 256;
}

// q, k: fp16 [ntok, d] (row stride ldq / ldk); vt: fp16 [d, ntok] = V transposed; out: fp16 [ntok, d] (row stride ldo).
extern "C" int fie_attn_vae_d512_f16(const void* q, long long ldq, const void* k, long long ldk, const void* vt, void* out, long long ldo,
                                     int ntok, int d, float scale, int f32_scores, int chunk_rows, void* workspace, size_t workspace_bytes,
                                     void* stream) {
    using namespace fie;
    FIE_REQUIRE(q && k && vt && out && workspace, "fie_attn_vae_d512_f16: null pointer");
    FIE_REQUIRE(ntok > 0 && d > 0 && (d % 64) == 0 && (ntok % 8) == 0, "fie_attn_vae_d512_f16: d %% 64 and ntok %% 8 required (d=%d ntok=%d)", d, ntok);
    if (chunk_rows <= 0 || chunk_rows > ntok) chunk_rows = ntok;
    FIE_REQUIRE(workspace_bytes >= fie_attn_vae_workspace_bytes(ntok, chunk_rows, f32_scores), "fie_attn_vae_d512_f16: workspace too small");
    FIE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "fie_attn_vae_d512_f16: workspace must be 256-byte aligned");
    const bool exp_only = !f32_scores && (ntok % 4) == 0 && ntok <= 16384;     // limits of k_softmax_rows_exp (row kept in registers)
    uint8_t* ws = (uint8_t*)workspace;
    const size_t score_bytes = (((size_t)chunk_rows * ntok * (f32_scores ? 4 : 2)) + 255) / 256 * 256;
    void* scores = ws;
    void* probs = f32_scores ? (void*)(ws + score_bytes) : scores;
    float* inv = (float*)(ws + score_bytes + (f32_scores ? (((size_t)chunk_rows * ntok * 2) + 255) / 256 * 256 : 0));
    for (int r0 = 0; r0 < ntok; r0 += chunk_rows) {
        const int rows = ntok - r0 < chunk_rows ? ntok - r0 : chunk_rows;
        fie_epilogue e1 = {};
        e1.rows_per_group = 1; e1.scale = f32_scores ? 1.0f : scale; e1.out_f32 = f32_scores ? 1 : 0;
        int rc = fie_gemm_f16((const __half*)q + (size_t)r0 * ldq, ldq, nullptr, 0, 0, k, scores, ntok, rows, ntok, d, &e1, stream);
        if (rc) return rc;
        fie_epilogue e2 = {};
        e2.rows_per_group = 1; e2.scale = 1.0f;
        if (exp_only) {
            if ((rc = fie_softmax_rows_exp_f16(scores, ntok, probs, ntok, inv, rows, ntok, 1.0f, stream))) return rc;
            e2.row_scale = inv;
        } else if (f32_scores) {
            if ((rc = fie_softmax_rows_f32_to_f16(scores, ntok, probs, ntok, rows, ntok, scale, stream))) return rc;
        } else {
            if ((rc = fie_softmax_rows_f16(scores, ntok, probs, ntok, rows, ntok, 1.0f, stream))) return rc;
        }
        if ((rc = fie_gemm_f16(probs, ntok, nullptr, 0, 0, vt, (__half*)out + (size_t)r0 * ldo, ldo, rows, d, ntok, &e2, stream))) return rc;
    }
    return FIE_OK;
}

// bf16 twin (the bf16 VAE): the same three passes with bf16 operands; the logits always stay fp32 between the passes, and P is written
// as bf16 so that both operands of the P V product are bf16.
extern "C" int fie_attn_vae_d512_bf16(const void* q, long long ldq, const void* k, long long ldk, const void* vt, void* out, long long ldo,
                                      int ntok, int d, float scale, int chunk_rows, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace fie;
    FIE_REQUIRE(q && k && vt && out && workspace, "fie_attn_vae_d512_bf16: null pointer");
    FIE_REQUIRE(ntok > 0 && d > 0 && (d % 64) == 0 && (ntok % 8) == 0, "fie_attn_vae_d512_bf16: d %% 64 and ntok %% 8 required (d=%d ntok=%d)", d, ntok);
    if (chunk_rows <= 0 || chunk_rows > ntok) chunk_rows = ntok;
    FIE_REQUIRE(workspace_bytes >= fie_attn_vae_workspace_bytes(ntok, chunk_rows, 1), "fie_attn_vae_d512_bf16: workspace too small");
    FIE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "fie_attn_vae_d512_bf16: workspace must be 256-byte aligned");
    uint8_t* ws = (uint8_t*)workspace;
    void* scores = ws;
    void* probs = ws + (((size_t)chunk_rows * ntok * 4) + 255) / 256 * 256;
    for (int r0 = 0; r0 < ntok; r0 += chunk_rows) {
        const int rows = ntok - r0 < chunk_rows ? ntok - r0 : chunk_rows;
        fie_epilogue e1 = {};
        e1.rows_per_group = 1; e1.scale = 1.0f; e1.out_f32 = 1;
        int rc = fie_gemm_bf16((const uint16_t*)q + (size_t)r0 * ldq, ldq, nullptr, 0, 0, k, scores, ntok, rows, ntok, d, &e1, FIE_DT_F32, stream);
        if (rc) return rc;
        if ((rc = fie_softmax_rows_f32_to_bf16(scores, ntok, probs, ntok, rows, ntok, scale, stream))) return rc;
        fie_epilogue e2 = {};
        e2.rows_per_group = 1; e2.scale = 1.0f;
        if ((rc = fie_gemm_bf16(probs, ntok, nullptr, 0, 0, vt, (uint16_t*)out + (size_t)r0 * ldo, ldo, rows, d, ntok, &e2, FIE_DT_BF16, stream))) return rc;
    }
    return FIE_OK;
}
