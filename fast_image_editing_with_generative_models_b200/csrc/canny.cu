// Integer Canny edge detector, bit-exact with cv2.cvtColor(RGB2GRAY) + cv2.Canny(gray, low, high)
// (aperture 3, L1 gradient, no blur) as called by the reference at src/pipeline.py:200,205.
//
// Stages (all integer):
//   k_nms       RGB (-> gray on the fly, 15-bit fixed point) tile + 2-px halo staged in shared memory -> Sobel (replicate border), L1 magnitude
//               (0 outside the image), integer-tangent NMS, double threshold -> state {0,1 weak,2 strong}; then the connected components
//               of the candidates INSIDE the 64 x 32 tile by a lock-free union-find in shared memory (strong pixels get the smaller
//               label so they win the root); global memory receives depth-1 trees (parent = the tile-local root)
//   k_seams     global lock-free union-find (atomicMin on roots), but only over the pixel pairs that straddle a tile seam
//   k_finalize  edge = candidate whose root is a strong pixel -> 0/255 (optionally replicated x3)
//   (the global finds of k_seams and k_finalize halve the paths they walk: uf_find_halve)
//   (k_gray     RGB -> gray as a separate plane: only for the optional Gaussian pre-stage / fie_rgb_to_gray_u8)
// The hysteresis result is the unique closure of strong pixels through candidates, so the union-find
// formulation is bit-exact with OpenCV's stack-based flood fill without any host round trip.
#include "fie_common.cuh"

namespace fie {

static constexpr uint32_t kWeakBit = 1u << 30;
static constexpr uint32_t kIdxMask = kWeakBit - 1;
static constexpr int TG22 = 13573;

__global__ void __launch_bounds__(256) k_gray(const uint8_t* __restrict__ rgb, uint8_t* __restrict__ gray, long long npix4, long long npix) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i < npix4; i += (long long)gridDim.x * blockDim.x) {
        long long p = i * 4;
        if (p + 4 <= npix) {
            const uint32_t* s = reinterpret_cast<const uint32_t*>(rgb + p * 3);   // 12-byte aligned group
            uint32_t w0 = __ldg(s), w1 = __ldg(s + 1), w2 = __ldg(s + 2);
            uint32_t r0 = w0 & 255, g0 = (w0 >> 8) & 255, b0 = (w0 >> 16) & 255;
            uint32_t r1 = w0 >> 24, g1 = w1 & 255, b1 = (w1 >> 8) & 255;
            uint32_t r2 = (w1 >> 16) & 255, g2 = w1 >> 24, b2 = w2 & 255;
            uint32_t r3 = (w2 >> 8) & 255, g3 = (w2 >> 16) & 255, b3 = w2 >> 24;
            uint32_t y0 = (9798u * r0 + 19235u * g0 + 3735u * b0 + 16384u) >> 15;
            uint32_t y1 = (9798u * r1 + 19235u * g1 + 3735u * b1 + 16384u) >> 15;
            uint32_t y2 = (9798u * r2 + 19235u * g2 + 3735u * b2 + 16384u) >> 15;
            uint32_t y3 = (9798u * r3 + 19235u * g3 + 3735u * b3 + 16384u) >> 15;
            *reinterpret_cast<uint32_t*>(gray + p) = y0 | (y1 << 8) | (y2 << 16) | (y3 << 24);
        } else {
            for (long long q = p; q < npix; ++q) {
                uint32_t r = rgb[q * 3], g = rgb[q * 3 + 1], b = rgb[q * 3 + 2];
                gray[q] = (uint8_t)((9798u * r + 19235u * g + 3735u * b + 16384u) >> 15);
            }
        }
    }
}

constexpr int TW = 64, TH = 32;   // output tile per CTA (256 threads, 8 px each)

__device__ __forceinline__ uint32_t uf_find(const uint32_t* P, uint32_t idx) {
    uint32_t v = ((volatile const uint32_t*)P)[idx];
    while ((v & kIdxMask) != idx) { idx = v & kIdxMask; v = ((volatile const uint32_t*)P)[idx]; }
    return v;   // root's label value (strong roots have kWeakBit clear)
}
// The same with path halving for the GLOBAL forest: a visited node is re-pointed at its grandparent.  Every entry holds the label of its
// parent and links only ever go to smaller labels, so atomicMin keeps the forest valid under concurrent unions; the chains that
// k_finalize has to walk afterwards get shorter.
__device__ __forceinline__ uint32_t uf_find_halve(uint32_t* P, uint32_t idx) {
    uint32_t v = ((volatile uint32_t*)P)[idx];
    while ((v & kIdxMask) != idx) {
        const uint32_t p = v & kIdxMask;
        const uint32_t gv = ((volatile uint32_t*)P)[p];
        if ((gv & kIdxMask) != p) atomicMin(&P[idx], gv);
        idx = p; v = gv;
    }
    return v;
}
template <bool HALVE = false>
__device__ __forceinline__ void uf_union(uint32_t* P, uint32_t i, uint32_t j) {
    uint32_t a = HALVE ? uf_find_halve(P, i) : uf_find(P, i), b = HALVE ? uf_find_halve(P, j) : uf_find(P, j);
    while ((a & kIdxMask) != (b & kIdxMask)) {
        if (a > b) { uint32_t t = a; a = b; b = t; }
        uint32_t old = atomicMin(&P[b & kIdxMask], a);
        if (old == b) break;
        b = HALVE ? uf_find_halve(P, old & kIdxMask) : uf_find(P, old & kIdxMask);
        a = HALVE ? uf_find_halve(P, a & kIdxMask) : uf_find(P, a & kIdxMask);
    }
}

// Tile kernel: (RGB -> gray on the fly, IN_CH = 3) -> Sobel / L1 magnitude / integer-tangent NMS / double threshold, then the connected
// components of the candidates INSIDE the tile by a lock-free union-find in shared memory (strong pixels carry the smaller label, so a
// component's root is strong iff the component contains a strong pixel).  Global memory only sees the dense state byte and, for candidates,
// parent[pixel] = the global index of the tile-local root (+ weak bit): every tile-local component leaves as a depth-1 tree, and the global
// union-find (k_seams) only has to join components across tile seams.
// thr: per-image (low, high) in device memory, or NULL -> the by-value low, high (the same for every image).
template <int IN_CH>
__global__ void __launch_bounds__(256) k_nms(const uint8_t* __restrict__ src, uint8_t* __restrict__ state,
                                             uint32_t* __restrict__ parent, int H, int W, int low, int high, const int2* __restrict__ thr) {
    __shared__ uint8_t  sg[TH + 4][TW + 4 + 4];
    __shared__ int16_t  sdx[TH + 2][TW + 2], sdy[TH + 2][TW + 2], smg[TH + 2][TW + 2];
    __shared__ uint32_t slab[TH * TW];           // local union-find: label = local index | weak bit
    __shared__ uint8_t  sst[TH * TW];
    const int img = blockIdx.z;
    if (thr) { const int2 t = __ldg(thr + img); low = t.x; high = t.y; }
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const uint8_t* g = src + (size_t)img * H * W * IN_CH;
    const int tid = threadIdx.x;
    constexpr int RAW_W = ((TW + 4) * 3 + 3) / 4 + 2;               // 32-bit words that cover one tile row of RGB bytes at any alignment
    __shared__ uint32_t sraw[IN_CH == 3 ? TH + 4 : 1][IN_CH == 3 ? RAW_W : 1];
    const bool fast_rgb = IN_CH == 3 && (W & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 3) == 0;
    if (fast_rgb) {
        // coalesced 32-bit loads of the tile's RGB rows into shared memory, then the gray conversion reads bytes from there
        const long long row_bytes = (long long)W * 3;
        const long long a0 = ((long long)(x0 - 2) * 3) & ~3ll;       // first staged byte of a row (may be negative: left of the image)
        for (int i = tid; i < (TH + 4) * RAW_W; i += 256) {
            const int ly = i / RAW_W, wi = i - ly * RAW_W;
            const int y = min(max(y0 + ly - 2, 0), H - 1);           // BORDER_REPLICATE (rows)
            const long long off = a0 + 4ll * wi;
            sraw[ly][wi] = (off >= 0 && off + 4 <= row_bytes) ? __ldg(reinterpret_cast<const uint32_t*>(g + (size_t)y * row_bytes + off)) : 0u;
        }
        __syncthreads();
        for (int i = tid; i < (TH + 4) * (TW + 4); i += 256) {
            const int ly = i / (TW + 4), lx = i % (TW + 4);
            const int x = min(max(x0 + lx - 2, 0), W - 1);           // BORDER_REPLICATE (columns): always inside the staged window
            const uint8_t* p = reinterpret_cast<const uint8_t*>(sraw[ly]) + ((long long)x * 3 - a0);
            sg[ly][lx] = (uint8_t)((9798u * p[0] + 19235u * p[1] + 3735u * p[2] + 16384u) >> 15);   // cv2 RGB2GRAY
        }
    } else {
        for (int i = tid; i < (TH + 4) * (TW + 4); i += 256) {
            int ly = i / (TW + 4), lx = i % (TW + 4);
            int y = min(max(y0 + ly - 2, 0), H - 1), x = min(max(x0 + lx - 2, 0), W - 1);   // BORDER_REPLICATE
            const uint8_t* p = g + ((size_t)y * W + x) * IN_CH;
            if (IN_CH == 3) sg[ly][lx] = (uint8_t)((9798u * __ldg(p) + 19235u * __ldg(p + 1) + 3735u * __ldg(p + 2) + 16384u) >> 15);   // cv2 RGB2GRAY
            else sg[ly][lx] = __ldg(p);
        }
    }
    __syncthreads();
    for (int i = tid; i < (TH + 2) * (TW + 2); i += 256) {
        int ly = i / (TW + 2), lx = i % (TW + 2);
        int y = y0 + ly - 1, x = x0 + lx - 1;
        int dx = 0, dy = 0, m = 0;
        if (y >= 0 && y < H && x >= 0 && x < W) {
            // gray coordinates of (y,x) in sg are (ly+1, lx+1); at image borders the replicate clamp must be
            // relative to the pixel itself, which the clamped halo load already guarantees for in-image pixels.
            int a00 = sg[ly][lx], a01 = sg[ly][lx + 1], a02 = sg[ly][lx + 2];
            int a10 = sg[ly + 1][lx], a12 = sg[ly + 1][lx + 2];
            int a20 = sg[ly + 2][lx], a21 = sg[ly + 2][lx + 1], a22 = sg[ly + 2][lx + 2];
            dx = (a02 + 2 * a12 + a22) - (a00 + 2 * a10 + a20);
            dy = (a20 + 2 * a21 + a22) - (a00 + 2 * a01 + a02);
            m = abs(dx) + abs(dy);
        }
        sdx[ly][lx] = (int16_t)dx; sdy[ly][lx] = (int16_t)dy; smg[ly][lx] = (int16_t)m;   // m = 0 outside the image
    }
    __syncthreads();
    for (int i = tid; i < TH * TW; i += 256) {
        int ly = i / TW, lx = i % TW;
        int y = y0 + ly, x = x0 + lx;
        uint8_t s = 0;
        if (y < H && x < W) {
            int cy = ly + 1, cx = lx + 1;
            int m = smg[cy][cx];
            if (m > low) {
                int dx = sdx[cy][cx], dy = sdy[cy][cx];
                int ax = abs(dx), ay = abs(dy) << 15;          // <= 1020<<15 < 2^31
                int t22 = ax * TG22;                           // <= 1020*13573 < 2^31
                long long t67 = (long long)t22 + ((long long)ax << 16);
                bool keep;
                if (ay < t22) keep = m > smg[cy][cx - 1] && m >= smg[cy][cx + 1];
                else if ((long long)ay > t67) keep = m > smg[cy - 1][cx] && m >= smg[cy + 1][cx];
                else { int sg_ = ((dx ^ dy) < 0) ? -1 : 1; keep = m > smg[cy - 1][cx - sg_] && m > smg[cy + 1][cx + sg_]; }
                if (keep) s = (m > high) ? 2 : 1;
            }
        }
        sst[i] = s;
        slab[i] = (uint32_t)i | (s == 2 ? 0u : kWeakBit);
    }
    __syncthreads();
    // tile-local unions with the W, NW, N, NE neighbours (each 8-connected pair once)
    for (int i = tid; i < TH * TW; i += 256) {
        if (!sst[i]) continue;
        const int ly = i / TW, lx = i % TW;
        if (lx > 0 && sst[i - 1]) uf_union(slab, i, i - 1);
        if (ly > 0) {
            if (lx > 0 && sst[i - TW - 1]) uf_union(slab, i, i - TW - 1);
            if (sst[i - TW]) uf_union(slab, i, i - TW);
            if (lx < TW - 1 && sst[i - TW + 1]) uf_union(slab, i, i - TW + 1);
        }
    }
    __syncthreads();
    for (int i = tid; i < TH * TW; i += 256) {
        const int ly = i / TW, lx = i % TW;
        const int y = y0 + ly, x = x0 + lx;
        if (y >= H || x >= W) continue;
        const size_t o = (size_t)img * H * W + (size_t)y * W + x;
        const uint8_t s = sst[i];
        state[o] = s;
        if (s) {
            const uint32_t r = uf_find(slab, (uint32_t)i);            // root label: local index | weak bit of the whole local component
            const uint32_t rl = r & kIdxMask;
            parent[o] = (uint32_t)((y0 + (int)(rl / TW)) * W + x0 + (int)(rl % TW)) | (r & kWeakBit);
        }
    }
}

// ---- fast tile kernel for the pipeline's shape (RGB input, W % 64 == 0, H % 32 == 0, 4-byte aligned rows) -----------------------------
// Same arithmetic and the same outputs as k_nms<3>, with four pixels per task so that address arithmetic, loads and stores are paid per
// 32-bit word instead of per byte (k_nms spends ~250 thread instructions per pixel and is issue-bound; ncu profiles/r2p_canny.md):
//   A  gray: 36 rows x 18 groups of 4 px (columns x0-4 .. x0+67), three aligned 32-bit RGB words per group -> one packed gray word;
//      rows and the two out-of-image column groups are clamped (BORDER_REPLICATE)
//   B  Sobel on 2 x 16-bit lanes per register (sums are <= 1020, the differences are biased by 2048 so no borrow crosses a lane),
//      L1 magnitude and the NMS direction class of the pixel itself -> (mag << 2 | class) as 16 bits, 0 outside the image
//   C  NMS + double threshold on the tile's 32 x 16 groups; groups without a pixel above `low` (the common case) stop after one load
//   D  tile-local union-find over the candidates, E  packed state words and the depth-1 parents go to global memory (as k_nms).
constexpr int FG = (TW + 8) / 4;                       // 18 staged groups per row

__device__ __forceinline__ uint32_t gray4(uint32_t w0, uint32_t w1, uint32_t w2) {
    const uint32_t r0 = w0 & 255, g0 = (w0 >> 8) & 255, b0 = (w0 >> 16) & 255;
    const uint32_t r1 = w0 >> 24, g1 = w1 & 255, b1 = (w1 >> 8) & 255;
    const uint32_t r2 = (w1 >> 16) & 255, g2 = w1 >> 24, b2 = w2 & 255;
    const uint32_t r3 = (w2 >> 8) & 255, g3 = (w2 >> 16) & 255, b3 = w2 >> 24;
    const uint32_t y0 = (9798u * r0 + 19235u * g0 + 3735u * b0 + 16384u) >> 15;
    const uint32_t y1 = (9798u * r1 + 19235u * g1 + 3735u * b1 + 16384u) >> 15;
    const uint32_t y2 = (9798u * r2 + 19235u * g2 + 3735u * b2 + 16384u) >> 15;
    const uint32_t y3 = (9798u * r3 + 19235u * g3 + 3735u * b3 + 16384u) >> 15;
    return y0 | (y1 << 8) | (y2 << 16) | (y3 << 24);
}

// (mag << 2) | direction class of one pixel: 0 horizontal, 1 vertical, 2 diagonal with dx, dy of equal sign, 3 of opposite sign
__device__ __forceinline__ uint32_t mag_class(int dx, int dy) {
    const int ax = abs(dx), ayp = abs(dy);
    const int m = ax + ayp;
    const int ay = ayp << 15;                          // <= 1020 << 15 < 2^31
    const int t22 = ax * TG22;                         // <= 1020 * 13573
    const int t67 = t22 + (ax << 16);                  // <= 80.7e6 < 2^31
    const uint32_t cls = ay < t22 ? 0u : (ay > t67 ? 1u : (((dx ^ dy) < 0) ? 3u : 2u));
    return ((uint32_t)m << 2) | cls;
}

__global__ void __launch_bounds__(256, 6) k_nms_rgb_fast(const uint8_t* __restrict__ src, uint8_t* __restrict__ state,
                                                      uint32_t* __restrict__ parent, int H, int W, int low, int high, const int2* __restrict__ thr) {
    __shared__ uint32_t sgw[TH + 4][FG];               // gray, 4 px per word, image rows y0-2.., columns x0-4..
    __shared__ __align__(8) uint32_t smc[TH + 2][2 * FG];   // (mag << 2 | class), 2 px per word, image rows y0-1.., columns x0-4..
    __shared__ uint32_t slab[TH * TW];
    __shared__ __align__(4) uint8_t sst[TH * TW];
    const int img = blockIdx.z, x0 = blockIdx.x * TW, y0 = blockIdx.y * TH, tid = threadIdx.x;
    if (thr) { const int2 t = __ldg(thr + img); low = t.x; high = t.y; }
    const uint8_t* g = src + (size_t)img * H * W * 3;
    const size_t row_bytes = (size_t)W * 3;
    // A
    for (int t = tid; t < (TH + 4) * FG; t += 256) {
        const int ly = t / FG, gx = t - ly * FG;
        const int y = min(max(y0 + ly - 2, 0), H - 1);
        const int xg = x0 - 4 + 4 * gx;
        uint32_t w;
        if (xg >= 0 && xg < W) {
            const uint32_t* p = reinterpret_cast<const uint32_t*>(g + (size_t)y * row_bytes + (size_t)xg * 3);
            w = gray4(__ldg(p), __ldg(p + 1), __ldg(p + 2));
        } else {
            const uint8_t* p = g + (size_t)y * row_bytes + (size_t)(xg < 0 ? 0 : W - 1) * 3;
            w = ((9798u * p[0] + 19235u * p[1] + 3735u * p[2] + 16384u) >> 15) * 0x01010101u;
        }
        sgw[ly][gx] = w;
    }
    __syncthreads();
    // B
    const bool border = blockIdx.x == 0 || blockIdx.x == gridDim.x - 1 || blockIdx.y == 0 || blockIdx.y == gridDim.y - 1;
    for (int t = tid; t < (TH + 2) * FG; t += 256) {
        const int ly = t / FG, gx = t - ly * FG;
        const int gl = max(gx - 1, 0), gr = min(gx + 1, FG - 1);
        uint32_t L[3], C[3], R[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const uint32_t wl = sgw[ly + r][gl], wc = sgw[ly + r][gx], wr = sgw[ly + r][gr];
            L[r] = __byte_perm(wl, wc, 0x6543);        // columns c-1 .. c+2
            C[r] = wc;                                 // columns c   .. c+3
            R[r] = __byte_perm(wc, wr, 0x4321);        // columns c+1 .. c+4
        }
        uint32_t out[2];
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
            const uint32_t sel = hf ? 0x4342u : 0x4140u;                       // bytes (2, 3) or (0, 1) -> two 16-bit lanes
            const uint32_t Lt = __byte_perm(L[0], 0, sel), Lm = __byte_perm(L[1], 0, sel), Lb = __byte_perm(L[2], 0, sel);
            const uint32_t Ct = __byte_perm(C[0], 0, sel), Cb = __byte_perm(C[2], 0, sel);
            const uint32_t Rt = __byte_perm(R[0], 0, sel), Rm = __byte_perm(R[1], 0, sel), Rb = __byte_perm(R[2], 0, sel);
            const uint32_t DX = (Rt + 2 * Rm + Rb) + 0x08000800u - (Lt + 2 * Lm + Lb);
            const uint32_t DY = (Lb + 2 * Cb + Rb) + 0x08000800u - (Lt + 2 * Ct + Rt);
            const uint32_t a = mag_class((int)(DX & 0xFFFFu) - 2048, (int)(DY & 0xFFFFu) - 2048);
            const uint32_t b = mag_class((int)(DX >> 16) - 2048, (int)(DY >> 16) - 2048);
            out[hf] = a | (b << 16);
        }
        if (border) {                                   // magnitude 0 outside the image
            const int y = y0 - 1 + ly, xg = x0 - 4 + 4 * gx;
            if (y < 0 || y >= H) { out[0] = 0; out[1] = 0; }
            else {
                if (xg < 0 || xg >= W) out[0] &= 0xFFFF0000u;
                if (xg + 1 < 0 || xg + 1 >= W) out[0] &= 0x0000FFFFu;
                if (xg + 2 < 0 || xg + 2 >= W) out[1] &= 0xFFFF0000u;
                if (xg + 3 < 0 || xg + 3 >= W) out[1] &= 0x0000FFFFu;
            }
        }
        *reinterpret_cast<uint2*>(&smc[ly][2 * gx]) = make_uint2(out[0], out[1]);
    }
    __syncthreads();
    // C
    const uint32_t lowc = (uint32_t)low << 2 | 3u;      // (mag << 2 | class) > lowc  <=>  mag > low
    for (int t = tid; t < TH * (TW / 4); t += 256) {
        const int ly = t >> 4, gq = t & 15;             // tile row, group of 4 tile pixels; staged column of pixel 0 = 4 + 4 gq
        const uint2 c = *reinterpret_cast<const uint2*>(&smc[ly + 1][2 + 2 * gq]);
        uint32_t sw = 0;
        if ((c.x & 0xFFFFu) > lowc || (c.x >> 16) > lowc || (c.y & 0xFFFFu) > lowc || (c.y >> 16) > lowc) {
            int m[3][6];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const uint32_t wl = smc[ly + r][1 + 2 * gq], wr = smc[ly + r][4 + 2 * gq];
                const uint2 wc = r == 1 ? c : *reinterpret_cast<const uint2*>(&smc[ly + r][2 + 2 * gq]);
                m[r][0] = (int)(wl >> 18);
                m[r][1] = (int)((wc.x & 0xFFFFu) >> 2); m[r][2] = (int)(wc.x >> 18);
                m[r][3] = (int)((wc.y & 0xFFFFu) >> 2); m[r][4] = (int)(wc.y >> 18);
                m[r][5] = (int)((wr & 0xFFFFu) >> 2);
            }
            const uint32_t cls4[4] = {c.x & 3u, (c.x >> 16) & 3u, c.y & 3u, (c.y >> 16) & 3u};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int mm = m[1][k + 1];
                uint32_t st = 0;
                if (mm > low) {
                    bool keep;
                    if (cls4[k] == 0) keep = mm > m[1][k] && mm >= m[1][k + 2];
                    else if (cls4[k] == 1) keep = mm > m[0][k + 1] && mm >= m[2][k + 1];
                    else if (cls4[k] == 2) keep = mm > m[0][k] && mm > m[2][k + 2];
                    else keep = mm > m[0][k + 2] && mm > m[2][k];
                    if (keep) st = mm > high ? 2u : 1u;
                }
                if (st) slab[4 * t + k] = (uint32_t)(4 * t + k) | (st == 2 ? 0u : kWeakBit);
                sw |= st << (8 * k);
            }
        }
        reinterpret_cast<uint32_t*>(sst)[t] = sw;
    }
    __syncthreads();
    // D: unions with the W, NW, N, NE neighbours (each 8-connected pair once)
    for (int t = tid; t < TH * (TW / 4); t += 256) {
        const uint32_t sw = reinterpret_cast<const uint32_t*>(sst)[t];
        if (!sw) continue;
        const int ly = t >> 4;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!((sw >> (8 * k)) & 0xFFu)) continue;
            const int i = 4 * t + k, lx = i & (TW - 1);
            if (lx > 0 && sst[i - 1]) uf_union(slab, i, i - 1);
            if (ly > 0) {
                if (lx > 0 && sst[i - TW - 1]) uf_union(slab, i, i - TW - 1);
                if (sst[i - TW]) uf_union(slab, i, i - TW);
                if (lx < TW - 1 && sst[i - TW + 1]) uf_union(slab, i, i - TW + 1);
            }
        }
    }
    __syncthreads();
    // E
    for (int t = tid; t < TH * (TW / 4); t += 256) {
        const int ly = t >> 4, gq = t & 15;
        const size_t o = (size_t)img * H * W + (size_t)(y0 + ly) * W + x0 + 4 * gq;
        const uint32_t sw = reinterpret_cast<const uint32_t*>(sst)[t];
        *reinterpret_cast<uint32_t*>(state + o) = sw;
        if (!sw) continue;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!((sw >> (8 * k)) & 0xFFu)) continue;
            const uint32_t r = uf_find(slab, (uint32_t)(4 * t + k));
            const uint32_t rl = r & kIdxMask;
            parent[o + k] = (uint32_t)((y0 + (int)(rl / TW)) * W + x0 + (int)(rl % TW)) | (r & kWeakBit);
        }
    }
}

// Joins the tile-local components across the tile seams (global lock-free union-find on the per-image parent array): one thread per
// pixel on the left side of a vertical seam or the upper side of a horizontal seam, united with its up-to-three candidate neighbours on
// the other side.  Every 8-connected pair that straddles a seam is covered exactly once.
__global__ void __launch_bounds__(256) k_seams(const uint8_t* __restrict__ state, uint32_t* __restrict__ parent, int H, int W) {
    const int img = blockIdx.y;
    const int nvs = (W - 1) / TW, nhs = (H - 1) / TH;               // vertical / horizontal seams inside the image
    const long long nv = (long long)nvs * H, nh = (long long)nhs * W;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nv + nh) return;
    const uint8_t* s = state + (size_t)img * H * W;
    uint32_t* P = parent + (size_t)img * H * W;
    if (t < nv) {
        const int k = (int)(t / H) + 1, y = (int)(t % H);
        const int x = k * TW - 1;                                   // left pixel; neighbours at column x + 1
        if (!s[(size_t)y * W + x]) return;
        const uint32_t me = (uint32_t)(y * W + x);
        for (int d = -1; d <= 1; ++d) {
            const int yy = y + d;
            if (yy >= 0 && yy < H && s[(size_t)yy * W + x + 1]) uf_union<true>(P, me, (uint32_t)(yy * W + x + 1));
        }
    } else {
        const long long u = t - nv;
        const int k = (int)(u / W) + 1, x = (int)(u % W);
        const int y = k * TH - 1;                                   // upper pixel; neighbours in row y + 1
        if (!s[(size_t)y * W + x]) return;
        const uint32_t me = (uint32_t)(y * W + x);
        for (int d = -1; d <= 1; ++d) {
            const int xx = x + d;
            if (xx >= 0 && xx < W && s[(size_t)(y + 1) * W + xx]) uf_union<true>(P, me, (uint32_t)((y + 1) * W + xx));
        }
    }
}

// 4 pixels per thread when the row width allows it: one 32-bit state load, one (1 channel) or three (3 channels) 32-bit stores.
__global__ void __launch_bounds__(256) k_finalize(const uint8_t* __restrict__ state, uint32_t* parent,
                                                  uint8_t* __restrict__ out, int H, int W, int out_channels) {
    const int img = blockIdx.z;
    uint32_t* P = parent + (size_t)img * H * W;                    // (written too: path halving while the roots are looked up)
    if ((W & 3) == 0 && ((reinterpret_cast<uintptr_t>(state) | reinterpret_cast<uintptr_t>(out)) & 3) == 0) {
        const int x = (blockIdx.x * 64 + (threadIdx.x & 63)) * 4, y = blockIdx.y * 4 + (threadIdx.x >> 6);
        if (x >= W || y >= H) return;
        const size_t o = (size_t)img * H * W + (size_t)y * W + x;
        const uint32_t st = *reinterpret_cast<const uint32_t*>(state + o);
        uint32_t e = 0;                                             // 4 edge bytes
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if ((st >> (8 * k)) & 0xFFu) { const uint32_t r = uf_find_halve(P, (uint32_t)(y * W + x + k)); if (!(r & kWeakBit)) e |= 0xFFu << (8 * k); }
        if (out_channels == 1) *reinterpret_cast<uint32_t*>(out + o) = e;
        else {
            // bytes e0 e0 e0 e1 | e1 e1 e2 e2 | e2 e3 e3 e3
            const uint32_t e0 = e & 0xFFu, e1 = (e >> 8) & 0xFFu, e2 = (e >> 16) & 0xFFu, e3 = e >> 24;
            uint32_t* d = reinterpret_cast<uint32_t*>(out + o * 3);
            d[0] = e0 | (e0 << 8) | (e0 << 16) | (e1 << 24);
            d[1] = e1 | (e1 << 8) | (e2 << 16) | (e2 << 24);
            d[2] = e2 | (e3 << 8) | (e3 << 16) | (e3 << 24);
        }
        return;
    }
    const int x = blockIdx.x * 64 + (threadIdx.x & 63), y = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (x >= W || y >= H) return;
    const size_t o = (size_t)img * H * W + (size_t)y * W + x;
    uint8_t v = 0;
    if (state[o]) { uint32_t r = uf_find_halve(P, y * W + x); v = (r & kWeakBit) ? 0 : 255; }
    if (out_channels == 1) out[o] = v;
    else { out[o * 3] = v; out[o * 3 + 1] = v; out[o * 3 + 2] = v; }
}

// ---- optional integer Gaussian pre-stage (DEFAULT OFF: the reference calls cv2.Canny without a blur, src/pipeline.py:205) ----
// Bit-exact with cv2.GaussianBlur(img, (5, 5), 0) on uint8: OpenCV's fixed-point path uses the exact kernel [1 4 6 4 1] / 16 per
// axis in 8.8 / 16.16 fixed point with one final rounding, which equals (sum_ij w_i w_j p_ij + 128) >> 8 with integer weights
// (sum 256); border BORDER_REFLECT_101.  Horizontal pass into shared memory (16-bit), vertical pass out; C interleaved channels.
constexpr int GW = 128, GH = 16;
__device__ __forceinline__ int reflect101(int p, int len) {
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}
template <int C>
__global__ void __launch_bounds__(256) k_gauss5(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int H, int W) {
    __shared__ uint8_t  sp[GH + 4][(GW + 4) * C];
    __shared__ uint16_t sh[GH + 4][GW * C];
    const int img = blockIdx.z, x0 = blockIdx.x * GW, y0 = blockIdx.y * GH, tid = threadIdx.x;
    const uint8_t* s = src + (size_t)img * H * W * C;
    for (int i = tid; i < (GH + 4) * (GW + 4); i += 256) {
        const int ly = i / (GW + 4), lx = i % (GW + 4);
        const int y = reflect101(y0 + ly - 2, H), x = reflect101(x0 + lx - 2, W);
#pragma unroll
        for (int c = 0; c < C; ++c) sp[ly][lx * C + c] = __ldg(s + ((size_t)y * W + x) * C + c);
    }
    __syncthreads();
    for (int i = tid; i < (GH + 4) * GW * C; i += 256) {
        const int ly = i / (GW * C), e = i % (GW * C);
        sh[ly][e] = (uint16_t)(sp[ly][e] + 4 * sp[ly][e + C] + 6 * sp[ly][e + 2 * C] + 4 * sp[ly][e + 3 * C] + sp[ly][e + 4 * C]);
    }
    __syncthreads();
    for (int i = tid; i < GH * GW * C; i += 256) {
        const int ly = i / (GW * C), e = i % (GW * C);
        const int y = y0 + ly, x = x0 + e / C;
        if (y >= H || x >= W) continue;
        const int v = sh[ly][e] + 4 * sh[ly + 1][e] + 6 * sh[ly + 2][e] + 4 * sh[ly + 3][e] + sh[ly + 4][e];
        dst[((size_t)img * H + y) * W * C + (size_t)x0 * C + e] = (uint8_t)((v + 128) >> 8);
    }
}

}  // namespace fie

extern "C" int fie_gaussian_blur5_u8(const void* src, void* dst, int n, int h, int w, int channels, void* stream_) {
    using namespace fie;
    FIE_REQUIRE(n >= 0 && h > 0 && w > 0 && n <= 65535, "fie_gaussian_blur5_u8: bad shape n=%d h=%d w=%d", n, h, w);
    FIE_REQUIRE(channels == 1 || channels == 3, "fie_gaussian_blur5_u8: channels must be 1 or 3");
    if (n == 0) return FIE_OK;
    FIE_REQUIRE(src && dst && src != dst, "fie_gaussian_blur5_u8: null pointer or in-place call");
    dim3 grid(ceil_div(w, GW), ceil_div(h, GH), n);
    if (channels == 1) k_gauss5<1><<<grid, 256, 0, (cudaStream_t)stream_>>>((const uint8_t*)src, (uint8_t*)dst, h, w);
    else k_gauss5<3><<<grid, 256, 0, (cudaStream_t)stream_>>>((const uint8_t*)src, (uint8_t*)dst, h, w);
    return check_launch("fie_gaussian_blur5_u8");
}

extern "C" int fie_rgb_to_gray_u8(const void* rgb, void* gray, int n, int h, int w, void* stream_) {
    using namespace fie;
    FIE_REQUIRE(n >= 0 && h > 0 && w > 0, "fie_rgb_to_gray_u8: bad shape");
    if (n == 0) return FIE_OK;
    FIE_REQUIRE(rgb && gray, "fie_rgb_to_gray_u8: null pointer");
    FIE_REQUIRE((reinterpret_cast<uintptr_t>(rgb) & 3) == 0 && (reinterpret_cast<uintptr_t>(gray) & 3) == 0, "fie_rgb_to_gray_u8: pointers must be 4-byte aligned");
    const size_t px = (size_t)n * h * w;
    const long long n4 = (long long)((px + 3) / 4);
    int blocks = (int)((n4 + 255) / 256); if (blocks > device_sm_count() * 16) blocks = device_sm_count() * 16;
    k_gray<<<blocks, 256, 0, (cudaStream_t)stream_>>>((const uint8_t*)rgb, (uint8_t*)gray, n4, (long long)px);
    return check_launch("fie_rgb_to_gray_u8");
}

extern "C" size_t fie_canny_workspace_bytes(int n, int h, int w) {
    size_t px = (size_t)n * h * w;
    // gray u8 + state u8 (each rounded to 256 B) + parent u32
    return ((px + 255) / 256) * 256 * 2 + px * 4;
}

// thr == NULL: (low, high) for every image.  Otherwise the per-image pairs in device memory, which the caller has normalised
// (swap if low > high, clamp to [0, 2040]); low = 0, high = 2040 then stand for them in the kernel choice.
static int canny_impl(const char* fn, const void* img, void* edges, int n, int h, int w, int in_channels, int out_channels,
                      int low, int high, const int2* thr, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    using namespace fie;
    FIE_REQUIRE(n >= 0 && h > 0 && w > 0, "%s: bad shape n=%d h=%d w=%d", fn, n, h, w);
    FIE_REQUIRE(in_channels == 1 || in_channels == 3, "%s: in_channels must be 1 or 3", fn);
    FIE_REQUIRE(out_channels == 1 || out_channels == 3, "%s: out_channels must be 1 or 3", fn);
    FIE_REQUIRE((long long)h * w < (1ll << 30), "%s: image too large", fn);
    FIE_REQUIRE(n <= 65535, "%s: batch too large", fn);
    if (n == 0) return FIE_OK;
    FIE_REQUIRE(img && edges && workspace, "%s: null pointer", fn);
    FIE_REQUIRE(workspace_bytes >= fie_canny_workspace_bytes(n, h, w), "%s: workspace too small", fn);
    if (low > high) { int t = low; low = high; high = t; }
    size_t px = (size_t)n * h * w, pxr = ((px + 255) / 256) * 256;
    uint8_t* gray = (uint8_t*)workspace;
    uint8_t* state = gray + pxr;
    uint32_t* parent = (uint32_t*)(state + pxr);
    (void)gray;                                   // (the gray plane is no longer materialised: k_nms<3> converts on the fly)
    dim3 g1(ceil_div(w, TW), ceil_div(h, TH), n);
    const bool fast_tile = in_channels == 3 && (w % TW) == 0 && (h % TH) == 0 && low >= 0 && high < 8192 &&
                           ((reinterpret_cast<uintptr_t>(img) | reinterpret_cast<uintptr_t>(state)) & 3) == 0;
    if (fast_tile) k_nms_rgb_fast<<<g1, 256, 0, stream>>>((const uint8_t*)img, state, parent, h, w, low, high, thr);
    else if (in_channels == 3) k_nms<3><<<g1, 256, 0, stream>>>((const uint8_t*)img, state, parent, h, w, low, high, thr);
    else k_nms<1><<<g1, 256, 0, stream>>>((const uint8_t*)img, state, parent, h, w, low, high, thr);
    const long long seam_px = (long long)((w - 1) / TW) * h + (long long)((h - 1) / TH) * w;
    if (seam_px > 0) k_seams<<<dim3((unsigned)((seam_px + 255) / 256), n), 256, 0, stream>>>(state, parent, h, w);
    const bool fin4 = (w & 3) == 0 && ((reinterpret_cast<uintptr_t>(state) | reinterpret_cast<uintptr_t>(edges)) & 3) == 0;
    dim3 g2(ceil_div(fin4 ? w / 4 : w, 64), ceil_div(h, 4), n);
    // (measured on B200: 16-pixel / 128-bit and shared-memory-staged variants of this kernel are not faster -- its time is the latency of
    //  the root chains that k_seams leaves behind, paid by every warp that holds a candidate, not the store pattern)
    k_finalize<<<g2, 256, 0, stream>>>(state, parent, (uint8_t*)edges, h, w, out_channels);
    return check_launch(fn);
}

extern "C" int fie_canny_u8(const void* img, void* edges, int n, int h, int w, int in_channels, int out_channels,
                            int low, int high, void* workspace, size_t workspace_bytes, void* stream) {
    return canny_impl("fie_canny_u8", img, edges, n, h, w, in_channels, out_channels, low, high, nullptr, workspace, workspace_bytes,
                      (cudaStream_t)stream);
}

extern "C" int fie_canny_u8_per_image(const void* img, void* edges, int n, int h, int w, int in_channels, int out_channels,
                                      const int* thresholds, void* workspace, size_t workspace_bytes, void* stream) {
    FIE_REQUIRE(thresholds || n == 0, "fie_canny_u8_per_image: null thresholds");
    return canny_impl("fie_canny_u8_per_image", img, edges, n, h, w, in_channels, out_channels, 0, 2040, (const int2*)thresholds, workspace,
                      workspace_bytes, (cudaStream_t)stream);
}
