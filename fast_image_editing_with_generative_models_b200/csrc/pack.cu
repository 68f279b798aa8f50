// Load-time weight transforms on the GPU (SURVEY 8(b) `fie_pack_weights_*`): the cold path of FastEditor.__init__
// (reference src/pipeline.py:45-181: from_pretrained + load_lora_weights) without a single ATen / cuBLAS kernel.
// Inputs are the fp32 master tensors under diffusers' parameter layouts (OIHW convolutions, [out, in] linears); outputs are the
// layouts the kernels in this library consume (DESIGN.md section 2).  All plain CUDA-core kernels: these run once per model load.
//
//   fie_pack_conv3x3_f16      [O,I,3,3] fp32 -> fp16 [Op][kh][kw][Ip] (K-major B operand of the implicit GEMM), zero padded
//   fie_pack_conv3x3_c8_f16   [O,I<=8,3,3] fp32 -> fp16 [Op][kh][hi|lo][8 px][8 ch] (tensor-core conv_in; w = hi + lo to ~2^-22)
//   fie_pack_conv_up2x_f16    [O,I,3,3] fp32 -> fp16 [4 phases][O][ty][tx][I]: the 2x2 phase filters of nearest-2x upsample + conv3x3
//   fie_pack_rows_f16         [N,K] fp32 -> fp16 [N,K] with an optional row permutation (GEGLU tile interleave) and bias gather
//   fie_fold_layernorm_f16    LayerNorm(gamma, beta) folded into the following Linear: W'' = centred(W * gamma) fp16, b'' = b + W beta
//   fie_fuse_lora_f32         W += scale * B A  (LCM-LoRA fuse, fp32; conv weights viewed as [O, I*k*k])
//   fie_pack_{conv3x3,conv_up2x,rows}_bf16: the same layouts with bf16 elements (the bf16 VAE)
#include "fie_common.cuh"

namespace fie {

// OBF: bf16 elements instead of fp16 (the bf16 VAE); same layouts.
template <bool OBF>
__global__ void __launch_bounds__(256) k_pack_conv3x3(const float* __restrict__ w, uint16_t* __restrict__ out, int O, int I, int Op, int Ip) {
    const long long total = (long long)Op * 9 * Ip;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e % Ip), t = (int)((e / Ip) % 9), o = (int)(e / ((long long)9 * Ip));
        float v = 0.f;
        if (o < O && i < I) v = w[(((long long)o * I + i) * 9) + t];          // OIHW: tap t = kh * 3 + kw
        out[e] = f_to_h<OBF>(v);
    }
}

__global__ void __launch_bounds__(256) k_pack_conv3x3_c8(const float* __restrict__ w, __half* __restrict__ out, int O, int I, int Op) {
    const long long total = (long long)Op * 3 * 2 * 64;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(e & 7), px = (int)((e >> 3) & 7), part = (int)((e >> 6) & 1), kh = (int)((e >> 7) % 3), o = (int)(e / 384);
        float v = 0.f;
        if (o < O && px < 3 && c < I) {
            const float x = w[(((long long)o * I + c) * 3 + kh) * 3 + px];    // pixel px of the window = kw
            const float hi = __half2float(__float2half_rn(x));
            v = part ? x - hi : x;                                            // fp16(x) | fp16(x - fp16(x))
        }
        out[e] = __float2half_rn(v);
    }
}

template <bool OBF>
__global__ void __launch_bounds__(256) k_pack_conv_up2x(const float* __restrict__ w, uint16_t* __restrict__ out, int O, int I) {
    // phase (a, b), tap (ty, tx): sum of the 3x3 taps that land on input pixel (i + ty - 1 + a, j + tx - 1 + b) of the 2x-upsampled conv.
    // a = 0: ty 0 <- kh {0}, ty 1 <- kh {1, 2};  a = 1: ty 0 <- kh {0, 1}, ty 1 <- kh {2}; identically for columns.
    const long long total = (long long)4 * O * 4 * I;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e % I), tap = (int)((e / I) & 3), o = (int)((e / ((long long)4 * I)) % O), ph = (int)(e / ((long long)4 * I * O));
        const int a = ph >> 1, b = ph & 1, ty = tap >> 1, tx = tap & 1;
        const int kh0 = a == 0 ? (ty == 0 ? 0 : 1) : (ty == 0 ? 0 : 2), kh1 = a == 0 ? (ty == 0 ? 0 : 2) : (ty == 0 ? 1 : 2);
        const int kw0 = b == 0 ? (tx == 0 ? 0 : 1) : (tx == 0 ? 0 : 2), kw1 = b == 0 ? (tx == 0 ? 0 : 2) : (tx == 0 ? 1 : 2);
        const float* wp = w + ((long long)o * I + i) * 9;
        // the same association as weights.pack_conv_up2x: rows are summed first (fp32), then columns
        float acc = 0.f;
        bool first_col = true;
        for (int kw = kw0; kw <= kw1; ++kw) {
            float r = wp[kh0 * 3 + kw];
            for (int kh = kh0 + 1; kh <= kh1; ++kh) r += wp[kh * 3 + kw];
            acc = first_col ? r : acc + r;
            first_col = false;
        }
        out[e] = f_to_h<OBF>(acc);
    }
}

template <bool OBF>
__global__ void __launch_bounds__(256) k_pack_rows(const float* __restrict__ w, const float* __restrict__ b, const int* __restrict__ perm,
                                                   uint16_t* __restrict__ out_w, float* __restrict__ out_b, int N, int K) {
    const long long total = (long long)N * K;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(e / K), k = (int)(e % K);
        const int src = perm ? perm[n] : n;
        out_w[e] = f_to_h<OBF>(w[(long long)src * K + k]);
        if (k == 0 && b && out_b) out_b[n] = b[src];
    }
}

// One CTA per output row n: W'[k] = W[n,k] * gamma[k]; mean over k; out = fp16(W' - mean); bias = b[n] + sum_k W[n,k] beta[k].
__global__ void __launch_bounds__(256) k_fold_layernorm(const float* __restrict__ w, const float* __restrict__ b, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, __half* __restrict__ out_w, float* __restrict__ out_b, int K) {
    __shared__ float red[2][8];
    const int n = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const float* row = w + (long long)n * K;
    float s = 0.f, d = 0.f;
    for (int k = tid; k < K; k += 256) { const float x = row[k]; s += x * gamma[k]; if (beta) d += x * beta[k]; }
    s = warp_sum(s); d = warp_sum(d);
    if (lane == 0) { red[0][wid] = s; red[1][wid] = d; }
    __syncthreads();
    float ts = 0.f, td = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { ts += red[0][i]; td += red[1][i]; }
    const float mean = ts / (float)K;
    for (int k = tid; k < K; k += 256) out_w[(long long)n * K + k] = __float2half_rn(row[k] * gamma[k] - mean);
    if (tid == 0) out_b[n] = (b ? b[n] : 0.f) + td;
}

// W[o, c] += scale * sum_r B[o, r] * A[r, c]   (fp32; 32 x 32 output tile per CTA, the rank dimension staged through shared memory)
__global__ void __launch_bounds__(256) k_fuse_lora(float* __restrict__ w, const float* __restrict__ A, const float* __restrict__ B, float scale,
                                                   int O, int R, long long C) {
    __shared__ float sB[32][33], sA[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;                   // 32 x 8 threads, 4 rows each
    const long long c0 = (long long)blockIdx.x * 32;
    const int o0 = blockIdx.y * 32;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int r0 = 0; r0 < R; r0 += 32) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int row = ty + 8 * j;
            const int o = o0 + row, r = r0 + tx;
            sB[row][tx] = (o < O && r < R) ? B[(long long)o * R + r] : 0.f;                 // B tile [o][r]
            const int rr = r0 + row; const long long c = c0 + tx;
            sA[row][tx] = (rr < R && c < C) ? A[(long long)rr * C + c] : 0.f;               // A tile [r][c]
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            const float a = sA[k][tx];
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[j] = fmaf(sB[ty + 8 * j][k], a, acc[j]);
        }
        __syncthreads();
    }
    const long long c = c0 + tx;
    if (c < C) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { const int o = o0 + ty + 8 * j; if (o < O) w[(long long)o * C + c] += scale * acc[j]; }
    }
}

static unsigned grid_for(long long total) {
    long long b = (total + 255) / 256;
    const long long cap = (long long)device_sm_count() * 16;
    return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace fie
using namespace fie;

extern "C" int fie_pack_conv3x3_f16(const float* w, void* out, int cout, int cin, int cout_pad, int cin_pad, void* stream) {
    FIE_REQUIRE(w && out && cout > 0 && cin > 0 && cout_pad >= cout && cin_pad >= cin, "fie_pack_conv3x3_f16: bad arguments");
    k_pack_conv3x3<false><<<grid_for((long long)cout_pad * 9 * cin_pad), 256, 0, (cudaStream_t)stream>>>(w, (uint16_t*)out, cout, cin, cout_pad, cin_pad);
    return check_launch("fie_pack_conv3x3_f16");
}

extern "C" int fie_pack_conv3x3_bf16(const float* w, void* out, int cout, int cin, int cout_pad, int cin_pad, void* stream) {
    FIE_REQUIRE(w && out && cout > 0 && cin > 0 && cout_pad >= cout && cin_pad >= cin, "fie_pack_conv3x3_bf16: bad arguments");
    k_pack_conv3x3<true><<<grid_for((long long)cout_pad * 9 * cin_pad), 256, 0, (cudaStream_t)stream>>>(w, (uint16_t*)out, cout, cin, cout_pad, cin_pad);
    return check_launch("fie_pack_conv3x3_bf16");
}

extern "C" int fie_pack_conv3x3_c8_f16(const float* w, void* out, int cout, int cin, int cout_pad, void* stream) {
    FIE_REQUIRE(w && out && cout > 0 && cin > 0 && cin <= 8 && cout_pad >= cout, "fie_pack_conv3x3_c8_f16: bad arguments (cin <= 8)");
    k_pack_conv3x3_c8<<<grid_for((long long)cout_pad * 384), 256, 0, (cudaStream_t)stream>>>(w, (__half*)out, cout, cin, cout_pad);
    return check_launch("fie_pack_conv3x3_c8_f16");
}

extern "C" int fie_pack_conv_up2x_f16(const float* w, void* out, int cout, int cin, void* stream) {
    FIE_REQUIRE(w && out && cout > 0 && cin > 0, "fie_pack_conv_up2x_f16: bad arguments");
    k_pack_conv_up2x<false><<<grid_for((long long)16 * cout * cin), 256, 0, (cudaStream_t)stream>>>(w, (uint16_t*)out, cout, cin);
    return check_launch("fie_pack_conv_up2x_f16");
}

extern "C" int fie_pack_conv_up2x_bf16(const float* w, void* out, int cout, int cin, void* stream) {
    FIE_REQUIRE(w && out && cout > 0 && cin > 0, "fie_pack_conv_up2x_bf16: bad arguments");
    k_pack_conv_up2x<true><<<grid_for((long long)16 * cout * cin), 256, 0, (cudaStream_t)stream>>>(w, (uint16_t*)out, cout, cin);
    return check_launch("fie_pack_conv_up2x_bf16");
}

extern "C" int fie_pack_rows_f16(const float* w, const float* bias, const int* perm, void* out_w, float* out_bias, int n, int k, void* stream) {
    FIE_REQUIRE(w && out_w && n > 0 && k > 0 && (!bias || out_bias), "fie_pack_rows_f16: bad arguments");
    k_pack_rows<false><<<grid_for((long long)n * k), 256, 0, (cudaStream_t)stream>>>(w, bias, perm, (uint16_t*)out_w, out_bias, n, k);
    return check_launch("fie_pack_rows_f16");
}

extern "C" int fie_pack_rows_bf16(const float* w, const float* bias, const int* perm, void* out_w, float* out_bias, int n, int k, void* stream) {
    FIE_REQUIRE(w && out_w && n > 0 && k > 0 && (!bias || out_bias), "fie_pack_rows_bf16: bad arguments");
    k_pack_rows<true><<<grid_for((long long)n * k), 256, 0, (cudaStream_t)stream>>>(w, bias, perm, (uint16_t*)out_w, out_bias, n, k);
    return check_launch("fie_pack_rows_bf16");
}

extern "C" int fie_fold_layernorm_f16(const float* w, const float* bias, const float* gamma, const float* beta, void* out_w, float* out_bias,
                                      int n, int k, void* stream) {
    FIE_REQUIRE(w && gamma && out_w && out_bias && n > 0 && k > 0, "fie_fold_layernorm_f16: bad arguments");
    k_fold_layernorm<<<n, 256, 0, (cudaStream_t)stream>>>(w, bias, gamma, beta, (__half*)out_w, out_bias, k);
    return check_launch("fie_fold_layernorm_f16");
}

extern "C" int fie_fuse_lora_f32(float* w, const float* lora_a, const float* lora_b, float scale, int cout, int rank, long long cols, void* stream) {
    FIE_REQUIRE(w && lora_a && lora_b && cout > 0 && rank > 0 && cols > 0, "fie_fuse_lora_f32: bad arguments");
    FIE_REQUIRE((cols + 31) / 32 <= 2147483647ll && (cout + 31) / 32 <= 65535, "fie_fuse_lora_f32: matrix too large");
    dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((cout + 31) / 32));
    k_fuse_lora<<<grid, 256, 0, (cudaStream_t)stream>>>(w, lora_a, lora_b, scale, cout, rank, cols);
    return check_launch("fie_fuse_lora_f32");
}
