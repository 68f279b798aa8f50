/* fie_b200 — C-ABI of the B200-native (sm_100a) hot path behind the reference's FastEditor.edit().
 *
 * The reference (vismaychuriwala/Fast-Image-Editing-with-Generative-Models) is pure Python: its edit path
 * (src/pipeline.py:212-274) runs cv2.Canny on the CPU (:205) and then hands everything to the diffusers
 * pipeline (:261-272), which dispatches torch ops (conv2d / linear / group_norm / layer_norm / SDPA ...) to
 * cuDNN / cuBLAS / ATen.  The reference has no FFI of its own; the entry points below are what a binding for
 * this path would bind: one per hot op, raw device pointers + explicit shapes + a cudaStream_t, no torch
 * types, no allocation inside (workspace is passed in), no global mutable state besides the error string.
 *
 * Conventions
 *   - all functions return FIE_OK (0) or a negative error code; fie_last_error() gives a message (thread-local)
 *   - all pointers are DEVICE pointers unless stated otherwise; `stream` is a cudaStream_t passed as void*
 *   - activations are NHWC / token-major fp16: an image tensor [N,H,W,C] is the matrix [N*H*W, C]
 *   - weights are pre-packed by the host (see INTEGRATION.md): conv [Cout][kh][kw][Cin] fp16, linear [out][in] fp16
 */
#ifndef FIE_B200_H
#define FIE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FIE_OK 0
#define FIE_ERR_INVALID (-1) /* bad argument / unsupported shape */
#define FIE_ERR_CUDA (-2)    /* CUDA runtime / launch error */

const char* fie_last_error(void);
int fie_version(void);
/* 1 if the current device is sm_100 (tcgen05/TMA kernels usable). */
int fie_device_supported(void);

/* ---- Canny: replaces cv2.cvtColor + cv2.Canny at reference src/pipeline.py:200,205 (and np.stack :208) ----
 * img:   uint8 [n,h,w,in_channels] (in_channels 3 = RGB, 1 = gray)
 * edges: uint8 [n,h,w,out_channels] (out_channels 1, or 3 = replicated), values 0/255
 * Integer only; bit-exact with OpenCV (aperture 3, L1 gradient, no blur). */
size_t fie_canny_workspace_bytes(int n, int h, int w);
int fie_canny_u8(const void* img, void* edges, int n, int h, int w, int in_channels, int out_channels,
                 int low, int high, void* workspace, size_t workspace_bytes, void* stream);
/* Per-image thresholds (EditEngine.edit_batch with a threshold per image, pipeline.py): thresholds int32 [n][2] = (low, high) of
 * image i in DEVICE memory, so that a CUDA graph replays with new values.  Each pair must be normalised on the host as
 * cv2.Canny reads it: floor, swap if low > high, clamp both to [0, 2040] (ops.canny_thresholds).  L1 Sobel magnitudes lie in
 * [0, 2040] and a pixel of magnitude 0 never survives NMS, so the clamp changes no result.  Same kernels as fie_canny_u8. */
int fie_canny_u8_per_image(const void* img, void* edges, int n, int h, int w, int in_channels, int out_channels,
                           const int* thresholds, void* workspace, size_t workspace_bytes, void* stream);

/* ---- optional Canny pre-stage (DEFAULT OFF in the path: the reference's cv2.Canny call, src/pipeline.py:205, has no blur;
 * BASELINE.json's north_star lists a Gaussian stage, so it exists as an opt-in: FastEditor.preprocess_image(..., gaussian_blur=True)) ----
 * fie_rgb_to_gray_u8:    uint8 [n,h,w,3] -> uint8 [n,h,w], == cv2.cvtColor(RGB2GRAY) (15-bit fixed point), src/pipeline.py:200
 * fie_gaussian_blur5_u8: uint8 [n,h,w,channels] (1 or 3) -> same shape, bit-exact with cv2.GaussianBlur(img, (5, 5), 0)
 *                        (integer kernel [1 4 6 4 1]^2 / 256, one rounding, BORDER_REFLECT_101); dst != src. */
int fie_rgb_to_gray_u8(const void* rgb, void* gray, int n, int h, int w, void* stream);
int fie_gaussian_blur5_u8(const void* src, void* dst, int n, int h, int w, int channels, void* stream);

/* ---- Baseline JPEG encode (SURVEY 8(f)-2): replaces `edited.save(output_path)` (PIL -> libjpeg) at reference run_batch.py:224 /
 * run_single_image.py:114 ----
 * rgb: uint8 [n,h,w,3] on the device -> n complete JPEG files (JFIF, baseline sequential, 4:2:0, Annex K Huffman tables, `quality` as in
 * libjpeg / Pillow; default 75), image i at out + i * out_stride with its byte length in out_sizes[i] (device int32).  BYTE-IDENTICAL to
 * Pillow's Image.save(f, "JPEG", quality=quality) for the same pixels.  Integer only.  out_stride >= fie_jpeg_max_bytes(h, w);
 * workspace: fie_jpeg_workspace_bytes(n, h, w), 256-byte aligned.  fie_jpeg_write_header writes the 623 header bytes (host memory). */
int    fie_jpeg_header_bytes(void);
int    fie_jpeg_write_header(unsigned char* dst, int h, int w, int quality);
size_t fie_jpeg_workspace_bytes(int n, int h, int w);
size_t fie_jpeg_max_bytes(int h, int w);
int    fie_jpeg_encode_u8(const void* rgb, int n, int h, int w, int quality, void* out, size_t out_stride, int* out_sizes,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- Lanczos resize: replaces image.resize((1024, 1024), Image.LANCZOS) at reference src/pipeline.py:251 (SURVEY 8(f)-2) ----
 * uint8 [n,h,w,3] -> uint8 [n,oh,ow,3], bit-identical to Pillow: a horizontal then a vertical fixed-point pass (a pass is skipped when
 * that size does not change).  bounds_* int32 [out,2] = (first input index, count), coeff_* int32 [out,ksize] = 2^22 fixed-point
 * weights, computed on the host in double precision as Pillow does (resize.py); tmp: uint8 [n,h,ow,3] scratch (both passes). */
int fie_resample_lanczos_u8(const void* in_u8, void* out_u8, void* tmp_u8, int n, int h, int w, int oh, int ow,
                            const int* bounds_x, const int* coeff_x, int ksize_x, const int* bounds_y, const int* coeff_y, int ksize_y,
                            void* stream);

/* ---- Evaluation metrics (SURVEY 8(f)-4): the non-GEMM stages of the reference's MetricsCalculator, src/metrics.py:150-381 ----
 * The networks themselves (CLIP ViT-B/16 towers, DINO ViT-B/8, SqueezeNet 1.1) run on fie_gemm_f16 / fie_layernorm_f16 /
 * fie_attention_d64_f16. */
/* torchmetrics StructuralSimilarityIndexMeasure(data_range=1.0), src/metrics.py:175-177,214-237: a, b uint8 [n,h,w,c] read as v/255;
 * Gaussian window kernel_size (odd, <= 11; default 11) / sigma (1.5), k1 0.01, k2 0.03, valid region only (what the reflect-pad +
 * crop of torchmetrics leaves).  out_sum double [n] = sum of the SSIM map over channels and valid pixels (mean = / (c (h-k+1) (w-k+1))).  Pixels are float32 v/255 as in
 * the reference; the local moments are accumulated in double (float32 moments carry ~1e-4 of cancellation noise in flat regions). */
int fie_ssim_u8(const void* a, const void* b, int n, int h, int w, int c, int kernel_size, double sigma, double k1, double k2,
                double* out_sum, void* stream);
/* exact sum of (a - b)^2 over per_image bytes of each image -> uint64 [n]: MSE = sum / (255^2 per_image), PSNR = -10 log10(MSE)
 * (PeakSignalNoiseRatio / MeanSquaredError at src/metrics.py:190-197,285-336) */
int fie_sqdiff_u8(const void* a, const void* b, int n, long long per_image, unsigned long long* out, void* stream);
/* torchvision transforms.Resize(size, antialias=True) + Normalize on a float image (DinoDistanceMetric._to_tensor, src/metrics.py:124-136):
 * in uint8 (read as v/255) or fp32 [n,h,w,3] -> fp32 [n,oh,ow,3] = (resampled - mean) / std.  Separable, horizontal then vertical;
 * bounds_* int32 [out,2] = (first input index, count), coeff_* fp32 [out,ksize] normalised weights (resize.py: aten's
 * _upsample_bilinear2d_aa tables); a pass whose size does not change is skipped.  tmp: fp32 [n,h,ow,3] when ow != w. */
int fie_resample_f32(const void* in, int in_is_u8, void* out_f32, void* tmp_f32, int n, int h, int w, int oh, int ow,
                     const int* bounds_x, const float* coeff_x, int ksize_x, const int* bounds_y, const float* coeff_y, int ksize_y,
                     const float* mean3, const float* std3, void* stream);
/* ViT patch embedding as a GEMM operand: in uint8 (v/255) or fp32 [n,h,w,3] -> fp16 [n (h/P) (w/P), P P 3], K order (py, px, c);
 * mean3/std3 (host pointers, both or neither) normalise on the way */
int fie_patchify_f16(const void* in, int in_is_u8, void* out, int n, int h, int w, int patch, const float* mean3, const float* std3, void* stream);
/* tokens [n, n_patches + 1, c] = (class token | patch rows [n, n_patches, c]) + position embeddings [n_patches + 1, c]; fp16, c % 8 == 0 */
int fie_vit_assemble_f16(const void* patches, const void* cls, const void* pos, void* out, int n, int n_patches, int c, void* stream);
/* out[r] = in[r] / max(|in[r]|, eps), fp16 rows (fp32 math): the cosine self-similarity of DINO keys (src/metrics.py:79-84) is then a GEMM */
int fie_l2norm_rows_f16(const void* in, long long ld_in, void* out, long long ld_out, long long rows, int c, float eps, void* stream);
/* out_sum[0] = sum over a rows x cols window of (a - b)^2, fp32 inputs, double accumulation (F.mse_loss of two similarity maps, :146) */
int fie_sqdiff_f32(const void* a, long long lda, const void* b, long long ldb, long long rows, int cols, double* out_sum, void* stream);
/* out[r] = <a[r], b[r]> / max(|a[r]| |b[r]|, eps), fp16 rows -> fp32 [rows]: CLIPScore = 100 max(cos, 0) (src/metrics.py:264-283) */
int fie_cosine_rows_f16(const void* a, long long lda, const void* b, long long ldb, float* out, long long rows, int c, float eps, void* stream);
/* LPIPS / SqueezeNet 1.1 (LearnedPerceptualImagePatchSimilarity(net_type='squeeze'), src/metrics.py:180-182,239-262).
 * im2col of a 3x3 convolution for fie_gemm_f16: in fp16 [n,h,w,ld_in] (first c channels) -> fp16 [n oh ow, kpad], K order (ky, kx, c),
 * columns >= 9c zero.  in_is_u8: the RGB network input, mapped to ((v/255*2-1) - shift3[c]) / scale3[c] (LPIPS ScalingLayer). */
int fie_im2col3x3_f16(const void* in, int in_is_u8, long long ld_in, void* out, int n, int h, int w, int c, int stride, int pad, int kpad,
                      const float* shift3, const float* scale3, void* stream);
/* MaxPool2d(3, stride 2, ceil_mode=True): fp16 [n,h,w,c] -> [n, ceil((h-3)/2)+1, ceil((w-3)/2)+1, c]; c % 8 == 0 */
int fie_maxpool3s2_ceil_f16(const void* in, void* out, int n, int h, int w, int c, void* stream);
/* one LPIPS layer: out_sum double [n] = sum over pixels of sum_c lin[c] (f0/(|f0|+1e-10) - f1/(|f1|+1e-10))^2; f0, f1 fp16 [n,hw,c] */
int fie_lpips_layer_f16(const void* f0, const void* f1, const float* lin, int n, long long hw, int c, double* out_sum, void* stream);

/* ---- Pre/post-processing: replaces VaeImageProcessor.preprocess/postprocess inside the diffusers call
 *      at reference src/pipeline.py:261-272 ---- */
/* uint8 [n,h,w,3] -> fp16 [n,h+2,w+8,8]: x/127.5-1 (normalize=1) or x/255, written into the zero-padded 8-channel layout read by
 * fie_conv3x3_c8_f16 (real pixel (y,x) at (y+1,x+1); borders and channels 3..7 are zero) */
int fie_preprocess_u8_to_f16_pad8(const void* img_u8, void* out_f16, int n, int h, int w, int normalize, void* stream);
/* fp16 [n,h,w,4] (latents) -> the same zero-padded layout fp16 [n,h+2,w+8,8] (channels 4..7 and borders zero) */
int fie_pad8_f16(const void* x4_f16, void* out_f16, int n, int h, int w, void* stream);
/* fp16 [n,h,w,ld] (first 3 channels) -> uint8 [n,h,w,3]: round(clamp(x/2+0.5,0,1)*255) */
int fie_postprocess_f16_to_u8(const void* x_f16, int ld, void* out_u8, int n, int h, int w, void* stream);

/* ---- Elementwise helpers ---- */
/* out = silu(a) (fp16, count elements, multiple of 8) */
int fie_silu_f16(const void* a, void* out, long long count, void* stream);
/* sinusoidal embedding (diffusers Timesteps, flip_sin_to_cos, shift 0): vals fp32 [count] (HOST pointer,
 * count <= 64) -> fp16 [count, dim] = cat(cos, sin) */
int fie_sincos_embedding(const float* host_vals, int count, int dim, void* out_f16, void* stream);
/* the same from DEVICE values fp32 [count] (no count limit): the per-row timesteps of the time embedding (engine._EncoderPart.time_rows,
 * read from the graph's parameter block).  Bit-identical to fie_sincos_embedding for the same floats. */
int fie_sincos_embedding_dev(const float* dev_vals, int count, int dim, void* out_f16, void* stream);
/* softmax over rows: fp32 [rows, cols] (ld_in) * scale -> fp16 [rows, cols] (ld_out) */
int fie_softmax_rows_f32_to_f16(const void* s_f32, long long ld_in, void* p_f16, long long ld_out,
                                long long rows, int cols, float scale, void* stream);
/* the same with fp16 scores (already scaled by the producing GEMM's epilogue when scale = 1); may run in place (p = s) */
int fie_softmax_rows_f16(const void* s_f16, long long ld_in, void* p_f16, long long ld_out,
                         long long rows, int cols, float scale, void* stream);
/* The same softmax without its division: p = exp(scale * (s - rowmax)) <= 1 as fp16 and inv_sum[row] = 1 / sum(p) (of the
 * fp16-rounded values); the P V GEMM applies inv_sum through fie_epilogue.row_scale.  cols % 4 == 0, cols <= 16384; in place allowed. */
int fie_softmax_rows_exp_f16(const void* s_f16, long long ld_in, void* p_f16, long long ld_out, float* inv_sum,
                             long long rows, int cols, float scale, void* stream);

/* ---- GroupNorm(+SiLU), NHWC fp16: replaces F.group_norm (+F.silu) in ResnetBlock2D / Transformer2DModel ----
 * x0: [n, hw, c0]; optional x1: [n, hw, c1] is the channel-concatenated second source (torch.cat of the skip
 * connection in the up blocks); out: [n, hw, c0+c1].  stats_ws: int64 [n, groups, 2] (sum, sum of squares in 2^-20 fixed
 * point: integer atomics make the statistics bit-reproducible).  stats_ready = 1: stats_ws was already filled by the producing
 * GEMM / convolution (fie_epilogue.gn_stats) and the statistics pass is skipped (single source only). */
int fie_groupnorm_f16(const void* x0, int c0, const void* x1, int c1, void* out, int n, long long hw, int groups,
                      const float* gamma, const float* beta, float eps, int fuse_silu, void* stats_ws, int stats_ready, void* stream);

/* ---- LayerNorm over the last dim, fp16 rows: replaces F.layer_norm in BasicTransformerBlock ---- */
int fie_layernorm_f16(const void* x, void* out, long long rows, int c, const float* gamma, const float* beta,
                      float eps, void* stream);

/* ---- Tensor-core GEMM / implicit-GEMM convolution (tcgen05 + TMEM + TMA) ----
 * D[M, N] = epilogue( A[M, K] * B[N, K]^T ), fp16 operands, fp32 accumulation in TMEM.
 * Replaces F.linear (cuBLASLt) and F.conv2d (cuDNN) in every diffusers module on the path. */
enum { FIE_ACT_NONE = 0, FIE_ACT_SILU = 1, FIE_ACT_GEGLU = 2, FIE_ACT_GELU = 3 /* exact erf GELU */, FIE_ACT_QUICKGELU = 4 /* x*sigmoid(1.702x), CLIP-L */,
       FIE_ACT_RELU = 5 /* max(x, 0): the SqueezeNet of the LPIPS metric */ };

typedef struct {
    /* epilogue: v = acc + col_bias[n] + row_bias[m / rows_per_group][n] (+ m_bias[m])
     *           v = act(v); v *= scale; v += residual[m, n]; store
     * GEGLU: v = (value + col_bias + row_bias) * gelu_erf(gate + col_bias of the gate column), then scale and residual. */
    const float* col_bias;   /* [N] or NULL */
    const float* row_bias;   /* [ceil(M / rows_per_group), >= N] or NULL (time-embedding broadcast) */
    long long rows_per_group;
    long long ld_row_bias;   /* row stride of row_bias in elements (0 = N) */
    const float* m_bias;     /* [M] per-output-row bias or NULL (used for transposed projections); added before act; not with GEGLU */
    const void* residual;    /* fp16 [M, ld_res] or NULL */
    long long ld_res;
    float scale;             /* applied before the residual add */
    int act;                 /* FIE_ACT_* ; GEGLU: B rows interleaved per tile (value half | gate half), N_out = N/2 */
    int out_f32;             /* 1: D is fp32, else fp16 */
    /* Optional GroupNorm statistics of the OUTPUT, accumulated by the epilogue so that the following fie_groupnorm_f16 can
     * skip its statistics pass (stats_ready = 1): int64 [images][gn_groups][2] (sum, sum of squares; 2^-20 fixed point),
     * zeroed by the caller.  Requires channels-per-group = N_out / gn_groups dividing 32, gn_rows_per_image % 32 == 0 and
     * dividing the rows (M = images * gn_rows_per_image; fie_conv_up2x_*: rows are input pixels), and a
     * launch that stays on the fast epilogue path (fp16 output, N_out % 32 == 0, 32-byte aligned rows); else FIE_ERR_INVALID. */
    void* gn_stats;          /* or NULL */
    int gn_groups;
    long long gn_rows_per_image;
    /* Folded LayerNorm (BasicTransformerBlock: x -> LN -> Linear).  Producer side: ln_stats_out = int64 [M][2] (sum, sum of
     * squares of every fp16 output row over ALL N columns, 2^-20 fixed point; zeroed by the caller) is accumulated while the
     * rows are written.  Consumer side: ln_stats_in (the statistics of the A rows, ln_dim = their length K) makes the GEMM
     * compute LN(A) W^T without a normalisation pass: B must hold gamma (.) W with every row centred over K (then
     * sum_k x_k B_nk = sum_k (x_k - mean) gamma_k W_nk), col_bias includes W beta, and v = rstd[m] * acc + bias (see
     * weights.fold_layernorm).  Both need the fast epilogue path (fp16 output, N % 32 == 0, 32-byte aligned rows). */
    void* ln_stats_out;
    const void* ln_stats_in;
    float ln_eps;
    int ln_dim;
    /* Optional per-row scale applied to the accumulator before the biases: v = row_scale[m] * acc + bias ... (softmax
     * normalisation of the VAE mid-block attention).  Exclusive with ln_stats_in; needs the fast epilogue path. */
    const float* row_scale;
} fie_epilogue;

/* Accumulator tile width used for a GEGLU projection with N = 8C weight rows.  The host packs those rows per tile as
 * [value rows j*h..(j+1)*h | gate rows 4C + j*h ..] with h = fie_geglu_block_n(N)/2 (bias likewise). */
int fie_geglu_block_n(int N);

/* Tuning / test hook: force the CTA-group form (0 = auto, 1, 2) and the accumulator width (0 = auto) of fie_gemm_f16 /
 * fie_conv3x3_f16.  Not needed in production. */
void fie_tune_gemm(int force_cg, int force_block_n);

/* Tuning / test hook: enable (1) / disable (0) the halo form of the stride-1 3x3 convolution (input rows loaded once per channel
 * chunk and shared by the 9 taps) and set the widest cout it is used for (0 = keep).  Not needed in production. */
void fie_tune_conv_halo(int enable, int max_cout);
/* Test / measurement hook: force (1) the im2col form of fie_conv3x3_*, fie_conv_up2x_* and fie_conv3x3_c8_* on shapes that the
 * rectangular-box form also tiles (0 = choose by shape, the default).  Not needed in production. */
void fie_tune_conv_im2col(int force);
/* GroupNorm: largest thread-block cluster the single-pass shared-memory kernel (k_gn_slab) may use; 0 = always the two-kernel path,
 * default 1 — see the measurement note in csrc/norm.cu.  Experiments / tests only. */
void fie_tune_groupnorm_slab(int max_cluster);

/* Debug hook: device buffer of 8 x int64 per CTA that subsequent GEMM/conv launches fill with per-role wait-cycle
 * accounting (see gemm_conv.cu); NULL switches it off.  Not needed in production. */
void fie_gemm_trace(long long* device_buf);

/* A: fp16 [M, K] with row stride lda (elements, multiple of 8); optional second source A1 supplies
 * K columns [k_split, K) (k_split multiple of 64) — a virtual torch.cat along K.
 * B: fp16 [N, K] row-major (ldb = K).  D: [M, N_out] row stride ldd. */
int fie_gemm_f16(const void* A, long long lda, const void* A1, long long lda1, int k_split,
                 const void* B, void* D, long long ldd, long long M, int N, int K,
                 const fie_epilogue* ep, void* stream);
/* fie_gemm_f16 with a per-row-group scale: group_scale fp32 [ceil(M / ep->rows_per_group)] in device memory multiplies the
 * value where ep->scale does (after the activation, before the residual add), row m using group_scale[m / rows_per_group];
 * ep->scale is then ignored.  NULL: exactly fie_gemm_f16.  The ControlNet zero convolutions (engine.ControlNet.merge_into): one
 * conditioning scale per image and CFG half, rows_per_group = h*w. */
int fie_gemm_f16_ex(const void* A, long long lda, const void* A1, long long lda1, int k_split,
                    const void* B, void* D, long long ldd, long long M, int N, int K,
                    const fie_epilogue* ep, const float* group_scale, void* stream);

/* 3x3 convolution as implicit GEMM, NHWC fp16.  x: [n,h,w,cin] (cin multiple of 64), wgt: [cout][3][3][cin],
 * out: [n,oh,ow,cout].  stride 1: pad 1.  stride 2: pad_mode 0 = symmetric pad 1 (UNet Downsample2D),
 * pad_mode 1 = F.pad(0,1,0,1) then pad 0 (VAE encoder Downsample2D).  cout_valid <= cout columns are stored
 * (weights may be zero-padded to a multiple of 32 output channels).
 * Shapes: any n, h, w (stride 2: even h, w).  An output width that is a multiple of 128, or a divisor of 128 whose rows stack into
 * whole 128-pixel boxes, loads the A operand as a rectangular TMA box (stride 1 with >= 128-pixel rows: the halo form); every other
 * shape (e.g. widths 152, 76, 38, 576, 288, 144 of the 1216x832 / 1152x896 SDXL buckets) loads 128 consecutive output pixels in
 * raster order with TMA im2col mode.  The choice depends on the shape only; fie_conv_up2x_* and fie_conv3x3_c8_* follow the same
 * rule with the input width. */
int fie_conv3x3_f16(const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                    int cout_valid, int stride, int pad_mode, const fie_epilogue* ep, void* stream);

/* Nearest-2x upsample fused with the following 3x3 convolution (diffusers Upsample2D).  x: [n,h,w,cin] -> out [n,2h,2w,cout], any n, h, w.
 * wgt: fp16 [4][cout][2][2][cin] phase weights (host pre-sums the 3x3 taps that hit the same input pixel, see weights.py). */
int fie_conv_up2x_f16(const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                      const fie_epilogue* ep, void* stream);

/* 3x3 convolution with tiny Cin (<= 4, NHWC fp16 with 4 channels), CUDA cores: conv_in of UNet/ControlNet/VAE.
 * wgt: fp32 [cout][3][3][4]; bias fp32 [cout]; out fp16 [n,h,w,ld_out] (channels >= cout are zero-filled up to ld_out). */
int fie_conv3x3_cin4_f16(const void* x, const float* wgt, const float* bias, void* out, int ld_out,
                         int n, int h, int w, int cout, int act, void* stream);

/* 3x3 convolution (pad 1) of an image-like input with <= 8 channels on the tensor cores: conv_in of the VAE encoder and of
 * the ControlNet conditioning embedding at full resolution.  xp: fp16 zero-padded [n,h+2,w+8,8] (fie_preprocess_u8_to_f16_pad8);
 * wgt: fp16 [cout][3][2][64]: per kernel row a hi block and a lo block (w = hi + lo keeps the fp32 weights to ~2^-22), element
 * kw*8 + c = w[co][c][kh][kw], zeros elsewhere; out: [n,h,w,cout_valid..] rows of ldd.  Any n, h, w (see fie_conv3x3_f16). */
int fie_conv3x3_c8_f16(const void* xp, const void* wgt, void* out, long long ldd, int n, int h, int w, int cout,
                       int cout_valid, const fie_epilogue* ep, void* stream);

/* ---- bf16 VAE (DESIGN.md 3.11): the same tensor-core kernels with bf16 operands, for VAE checkpoints whose activations leave the
 * fp16 range (config.json "force_upcast": true, e.g. the original SDXL VAE).  Operands and fie_epilogue are as for the fp16 entry
 * points above, with every fp16 activation and weight replaced by bf16; accumulation stays fp32.  out_dtype selects the output
 * (FIE_DT_F16, FIE_DT_BF16 or FIE_DT_F32; fie_epilogue.out_f32 may only be set together with FIE_DT_F32); a residual is read in
 * the output's type.  GroupNorm statistics in the producing epilogue (gn_stats), ln_stats_out and GEGLU need fp16 output and are
 * rejected with FIE_ERR_INVALID for bf16 output. ---- */
enum { FIE_DT_F16 = 0, FIE_DT_BF16 = 1, FIE_DT_F32 = 2 };
int fie_gemm_bf16(const void* A, long long lda, const void* A1, long long lda1, int k_split,
                  const void* B, void* D, long long ldd, long long M, int N, int K,
                  const fie_epilogue* ep, int out_dtype, void* stream);
/* fie_gemm_bf16 with group_scale as in fie_gemm_f16_ex */
int fie_gemm_bf16_ex(const void* A, long long lda, const void* A1, long long lda1, int k_split,
                     const void* B, void* D, long long ldd, long long M, int N, int K,
                     const fie_epilogue* ep, int out_dtype, const float* group_scale, void* stream);
int fie_conv3x3_bf16(const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                     int cout_valid, int stride, int pad_mode, const fie_epilogue* ep, int out_dtype, void* stream);
int fie_conv_up2x_bf16(const void* x, const void* wgt, void* out, long long ldd, int n, int h, int w, int cin, int cout,
                       const fie_epilogue* ep, int out_dtype, void* stream);
/* conv_in at image / latent resolution: the operands stay fp16 (pad8 input and hi/lo weights exactly as fie_conv3x3_c8_f16, whose
 * inputs are bounded: an image in [-1, 1] or latents / scaling_factor); only the output type is selectable. */
int fie_conv3x3_c8_bf16(const void* xp, const void* wgt, void* out, long long ldd, int n, int h, int w, int cout,
                        int cout_valid, const fie_epilogue* ep, int out_dtype, void* stream);
/* GroupNorm(+SiLU) of bf16 NHWC activations (x0, optional concatenated x1, out as fie_groupnorm_f16).  Range-safe and deterministic:
 * slabs that fit one CTA take the single-pass two-pass-variance kernel (the fie_groupnorm_f16 rule); otherwise per-chunk
 * (count, mean, M2) partials over a fixed row partition are merged in a fixed order with Chan's formula (no fixed point, no
 * floating-point atomics).  workspace: fie_groupnorm_bf16_workspace_bytes(n, hw, c0 + c1, groups) bytes, 256-byte aligned. */
size_t fie_groupnorm_bf16_workspace_bytes(int n, long long hw, int c, int groups);
int fie_groupnorm_bf16(const void* x0, int c0, const void* x1, int c1, void* out, int n, long long hw, int groups,
                       const float* gamma, const float* beta, float eps, int fuse_silu, void* workspace, size_t workspace_bytes, void* stream);
/* row softmax of fp32 scores * scale -> bf16 probabilities */
int fie_softmax_rows_f32_to_bf16(const void* s_f32, long long ld_in, void* p_bf16, long long ld_out,
                                 long long rows, int cols, float scale, void* stream);
/* fie_attn_vae_d512_f16 with bf16 q, k, vt and out; the logits always stay fp32 between the passes
 * (workspace: fie_attn_vae_workspace_bytes(ntok, chunk_rows, 1)). */
int fie_attn_vae_d512_bf16(const void* q, long long ldq, const void* k, long long ldk, const void* vt, void* out, long long ldo,
                           int ntok, int d, float scale, int chunk_rows, void* workspace, size_t workspace_bytes, void* stream);
/* bf16 twins of the load-time packers below (same layouts, bf16 elements) */
int fie_pack_conv3x3_bf16(const float* w, void* out, int cout, int cin, int cout_pad, int cin_pad, void* stream);
int fie_pack_conv_up2x_bf16(const float* w, void* out, int cout, int cin, void* stream);
int fie_pack_rows_bf16(const float* w, const float* bias, const int* perm, void* out_w, float* out_bias, int n, int k, void* stream);

/* ---- VAE mid-block attention: 1 head, d = C (512), ntok = H*W tokens (16 384 at 1024^2) — SURVEY 8(b) `fie_attn_vae_d512` ----
 * Replaces Attention / AttnProcessor2_0 of the AutoencoderKL UNetMidBlock2D.  q, k: fp16 [ntok, d]; vt: fp16 [d, ntok] (V transposed, so
 * that P V is a K-major GEMM); out: fp16 [ntok, d].  One call = softmax(scale q k^T) v for one image, computed as three passes of the
 * tcgen05 GEMM / row-softmax kernels over `chunk_rows` query rows at a time (<= 0: the whole image; csrc/attn_vae.cu explains why this is
 * not a single flash kernel at d = 512).  f32_scores = 1 keeps the logits in fp32 between the passes (safe for real checkpoints whose
 * logits reach the hundreds); 0 stores them as fp16 (half the traffic).  workspace: fie_attn_vae_workspace_bytes(...), 256-byte aligned. */
size_t fie_attn_vae_workspace_bytes(int ntok, int chunk_rows, int f32_scores);
int fie_attn_vae_d512_f16(const void* q, long long ldq, const void* k, long long ldk, const void* vt, void* out, long long ldo,
                          int ntok, int d, float scale, int f32_scores, int chunk_rows, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Load-time weight transforms (SURVEY 8(b) `fie_pack_weights_*`): the cold path of FastEditor.__init__ — what from_pretrained +
 * load_lora_weights prepare at reference src/pipeline.py:89-161 — on the GPU without library kernels.  fp32 master tensors in diffusers'
 * layouts in, the layouts of DESIGN.md section 2 out.
 *   fie_pack_conv3x3_f16     w [cout,cin,3,3] -> fp16 [cout_pad][3][3][cin_pad] (zero padded): B operand of fie_conv3x3_f16
 *   fie_pack_conv3x3_c8_f16  w [cout,cin<=8,3,3] -> fp16 [cout_pad][3][2][64]: hi / lo parts for fie_conv3x3_c8_f16
 *   fie_pack_conv_up2x_f16   w [cout,cin,3,3] -> fp16 [4][cout][2][2][cin]: phase filters for fie_conv_up2x_f16
 *   fie_pack_rows_f16        w [n,k] (+ bias [n]) -> fp16 [n,k] (+ fp32 bias) with an optional row permutation perm[n] (device int32)
 *   fie_fold_layernorm_f16   LayerNorm(gamma, beta over k) followed by Linear(w [n,k], bias) -> centred fp16 weights + fp32 bias for a GEMM
 *                            with fie_epilogue.ln_stats_in (bias / beta may be NULL)
 *   fie_fuse_lora_f32        w [cout, cols] += scale * lora_b [cout, rank] x lora_a [rank, cols], fp32 in place (LCM-LoRA fuse; a conv
 *                            weight is viewed as [cout, cin*k*k], its LoRA A as [rank, cin*k*k]) */
int fie_pack_conv3x3_f16(const float* w, void* out, int cout, int cin, int cout_pad, int cin_pad, void* stream);
int fie_pack_conv3x3_c8_f16(const float* w, void* out, int cout, int cin, int cout_pad, void* stream);
int fie_pack_conv_up2x_f16(const float* w, void* out, int cout, int cin, void* stream);
int fie_pack_rows_f16(const float* w, const float* bias, const int* perm, void* out_w, float* out_bias, int n, int k, void* stream);
int fie_fold_layernorm_f16(const float* w, const float* bias, const float* gamma, const float* beta, void* out_w, float* out_bias,
                           int n, int k, void* stream);
int fie_fuse_lora_f32(float* w, const float* lora_a, const float* lora_b, float scale, int cout, int rank, long long cols, void* stream);

/* ---- Flash attention, head_dim 64 (tcgen05): replaces F.scaled_dot_product_attention in AttnProcessor2_0 ----
 * q: fp16 rows [b*nq, ldq] (head h at columns h*64..), k/v: [b*nkv, ldk/ldv], out: [b*nq, ldo]. No mask. */
int fie_attention_d64_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                          void* out, long long ldo, int b, int heads, int nq, int nkv, float scale, void* stream);
/* the same with a causal mask (key j visible to query i iff j <= i): the CLIP text encoders of the prompt-encoding stage that
 * precedes the path (transformers CLIPTextModel inside the diffusers call).  nkv <= 128. */
int fie_attention_d64_causal_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                                 void* out, long long ldo, int b, int heads, int nq, int nkv, float scale, void* stream);
/* token + position embedding lookup (CLIPTextEmbeddings): ids int32 [rows] (row r is position r % seq_len),
 * tok fp16 [vocab, c], pos fp16 [seq_len, c] -> out fp16 [rows, c]; c multiple of 8 */
int fie_embed_tokens_f16(const int* ids, const void* tok, const void* pos, void* out, long long rows, int seq_len, int c, int vocab, void* stream);

/* ---- Scheduler / latent math: replaces DiagonalGaussianDistribution.sample, LCMScheduler.add_noise,
 *      the CFG combine and LCMScheduler.step inside the diffusers call ---- */
/* The latent state is carried in fp32 between the scheduler steps; each call also writes the fp16 copy the UNet / ControlNet read.
 * Every image of a batch has its own strength, step count and guidance (EditEngine.edit_batch, pipeline.py): the coefficients are
 * DEVICE arrays, so that one CUDA graph serves every setting; image i covers pixels [i px_per_img, (i+1) px_per_img).
 * moments fp16 [n,hw,ld_m] (mean = ch 0..3, logvar = ch 4..7), xi/noise fp16 [n,hw,4], coef fp32 [n][2] = (sqrt_a, sqrt_1ma):
 * z0 = (mean + exp(0.5*clamp(logvar,-30,20))*xi)*scaling; x = sqrt_a*z0 + sqrt_1ma*noise. Writes x as fp32 and fp16 [n,hw,4] */
int fie_vae_sample_add_noise_batched(const void* moments, int ld_m, const void* xi, const void* noise, float* x_out_f32, void* x_out_f16,
                                     long long count_px, long long px_per_img, float scaling, const float* coef, void* stream);
/* eps_u/eps_c fp16 [count_px, ld_e] (first 4 ch), x fp32 [count_px,4], noise fp16 or NULL (last step), coef fp32 [n][7] =
 * (g, sa, s1, c_skip, c_out, sap, s1p) = (guidance, sqrt_a, sqrt_1ma, c_skip, c_out, sqrt_a_prev, sqrt_1ma_prev):
 * eps = eps_u + g*(eps_c-eps_u); x0 = (x - s1*eps)/sa; den = c_out*x0 + c_skip*x; x' = sap*den + s1p*noise, or den when last
 * (fp32 and fp16 out) */
int fie_cfg_lcm_step_batched(const void* eps_u, const void* eps_c, int ld_e, const float* x_f32, const void* noise, float* x_out_f32,
                             void* x_out_f16, long long count_px, long long px_per_img, const float* coef, int last, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FIE_B200_H */
