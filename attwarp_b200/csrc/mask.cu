// mask.cu -- the mask post-processing between stage 1 and stage 2b of the driver flow (SURVEY 8(f) N2).
//
// Replaces, on the device, the mask half of blend_mask
// ("Attention Guided Warping/attention_extraction/llava.py:207-256", called at AGW/main.py:361 and
// AGW/main_batched.py:268):
//   revise_mask: normalize(min) -> z-score x coe -> sigmoid -> clamp -> k x k box filter (replicate pad)
//   ToPILImage : float -> uint8 by truncation of v * 255
//   PIL resize(image.size, LANCZOS) of the mode-'L' mask
// The resize restates Pillow's 8-bit two-pass resampler (src/libImaging/Resample.c) exactly:
// per output coordinate a window of taps with weights normalised in double and rounded to 22-bit
// fixed point (computed once per (in, out) size pair on the host, with the C library's sin like Pillow),
// int32 accumulation from 1 << 21, clip to uint8 after the horizontal pass and after the vertical pass.
// Everything here is a few hundred KB per batch: one CTA per image (revise) / per tile of output rows
// (resize, the horizontal pass of the token rows recomputed per CTA into shared memory).
#include <math.h>
#include <stdlib.h>

#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "common.cuh"

namespace aw {
namespace {

constexpr int kMaskThreads = 256;
constexpr int kPrecisionBits = 32 - 8 - 2;      // Resample.c PRECISION_BITS
constexpr int kResizeRows = 32;                 // output rows per CTA

// ---- revise_mask + ToPILImage ---------------------------------------------------------------------
__global__ void __launch_bounds__(kMaskThreads)
revise_mask_kernel(const float* __restrict__ tok, int gh, int gw, int ksize, float coe,
                   float* __restrict__ revised, uint8_t* __restrict__ mask_u8) {
    extern __shared__ float sm_f[];
    __shared__ float red[32];
    __shared__ double redd[32];
    const int G = gh * gw;
    float* m = sm_f;                    // G
    const float* src = tok + (int64_t)blockIdx.x * G;
    float mn = INFINITY, mx = -INFINITY;
    for (int i = threadIdx.x; i < G; i += blockDim.x) {
        const float v = src[i];
        m[i] = v;
        mn = fminf(mn, v);
        mx = fmaxf(mx, v);
    }
    mx = block_max(mx, red);
    mn = -block_max(-mn, red);
    const float range = mx - mn;
    float part = 0.f;
    for (int i = threadIdx.x; i < G; i += blockDim.x) {          // normalize(mat, "min")
        const float v = (m[i] - mn) / range;
        m[i] = v;
        part += v;
    }
    const float mean = block_sum(part, red) / (float)G;
    double sq = 0.0;
    for (int i = threadIdx.x; i < G; i += blockDim.x) {          // enhance: centre, unbiased std
        const float v = m[i] - mean;
        m[i] = v;
        sq += (double)v * (double)v;
    }
    const float sd = (float)sqrt(block_sum(sq, redd) / (double)(G - 1));
    for (int i = threadIdx.x; i < G; i += blockDim.x) {
        const float z = m[i] / sd * coe;
        const float s = 1.0f / (1.0f + expf(-z));
        m[i] = fminf(fmaxf(s, 0.f), 1.f);
    }
    __syncthreads();
    const int pad = (ksize - 1) / 2;
    const float w = 1.0f / (float)(ksize * ksize);
    for (int i = threadIdx.x; i < G; i += blockDim.x) {          // box filter, replicate padding
        const int y = i / gw, x = i - y * gw;
        float acc = 0.f;
        for (int dy = -pad; dy <= pad; ++dy)
            for (int dx = -pad; dx <= pad; ++dx)
                acc = fadd_nofma(acc, fmul_nofma(w, m[clampi(y + dy, 0, gh - 1) * gw + clampi(x + dx, 0, gw - 1)]));
        if (revised != nullptr) revised[(int64_t)blockIdx.x * G + i] = acc;
        if (mask_u8 != nullptr) mask_u8[(int64_t)blockIdx.x * G + i] = (uint8_t)(int)fmul_nofma(acc, 255.0f);   // .mul(255).byte()
    }
}

// ---- Pillow LANCZOS resize of mode-'L' images -------------------------------------------------------
// tables: bounds [out] = {first tap, taps}, weights [out][ks]
__global__ void __launch_bounds__(kMaskThreads)
resize_lanczos_u8_kernel(const uint8_t* __restrict__ src, int h, int w, int Ho, int Wo,
                         const int2* __restrict__ bx, const int* __restrict__ kx, int ksx,
                         const int2* __restrict__ by, const int* __restrict__ ky, int ksy,
                         uint8_t* __restrict__ dst) {
    extern __shared__ uint8_t sm_b[];
    uint8_t* in = sm_b;                          // h * w        source image
    uint8_t* tmp = sm_b + ((h * w + 15) & ~15);  // rows * Wo    horizontal pass of the rows this tile taps
    const int b = blockIdx.y;
    const int y0 = blockIdx.x * kResizeRows, y1 = min(y0 + kResizeRows, Ho);
    // source rows tapped by the output rows [y0, y1): windows move monotonically with y
    const int r0 = Ho != h ? by[y0].x : y0;
    const int r1 = Ho != h ? by[y1 - 1].x + by[y1 - 1].y : y1;
    const uint8_t* img = src + (int64_t)b * h * w;
    for (int i = threadIdx.x; i < (r1 - r0) * w; i += blockDim.x) in[i] = img[r0 * w + i];
    __syncthreads();
    for (int i = threadIdx.x; i < (r1 - r0) * Wo; i += blockDim.x) {     // horizontal pass
        const int r = i / Wo, x = i - r * Wo;
        if (Wo != w) {
            const int2 bd = bx[x];
            const int* k = kx + (int64_t)x * ksx;
            int acc = 1 << (kPrecisionBits - 1);
            for (int t = 0; t < bd.y; ++t) acc += (int)in[r * w + bd.x + t] * k[t];
            tmp[i] = (uint8_t)clampi(acc >> kPrecisionBits, 0, 255);
        } else {
            tmp[i] = in[i];
        }
    }
    __syncthreads();
    uint8_t* out = dst + (int64_t)b * Ho * Wo;
    for (int i = threadIdx.x; i < (y1 - y0) * Wo; i += blockDim.x) {     // vertical pass
        const int yy = i / Wo, x = i - yy * Wo;
        const int y = y0 + yy;
        if (Ho != h) {
            const int2 bd = by[y];
            const int* k = ky + (int64_t)y * ksy;
            int acc = 1 << (kPrecisionBits - 1);
            for (int t = 0; t < bd.y; ++t) acc += (int)tmp[(bd.x - r0 + t) * Wo + x] * k[t];
            out[(int64_t)y * Wo + x] = (uint8_t)clampi(acc >> kPrecisionBits, 0, 255);
        } else {
            out[(int64_t)y * Wo + x] = tmp[yy * Wo + x];
        }
    }
}

// ---- the up-scaling case (a token-grid mask to image size: <= 8 taps per axis) ----------------------
// Same arithmetic, organised for throughput: the CTA owns a tile of output rows of one image, computes the
// horizontal pass of the (few) source rows the tile taps into shared memory once, then every thread owns
// FOUR adjacent output columns and walks down its share of the tile's rows with the tapped rows of the
// horizontal pass held in registers as a sliding window (the window moves one source row every Ho / h
// output rows); an output row is 8 x 4 IMAD with coefficients broadcast from shared memory, clip, one
// 32-bit store.  Zero-padded coefficient rows make every output row an 8-tap row.
// Pillow's window has 2 ceil(support) + 1 taps, always odd: an up-scaling has 7 per axis, never 8, so only the TAPS = 7
// instances below are compiled.
constexpr int kUpTaps = 8;        // coefficient rows in shared memory are padded to 8
__device__ __forceinline__ void unpack4(uint32_t w, int* v) {
    v[0] = (int)(w & 0xffu); v[1] = (int)((w >> 8) & 0xffu); v[2] = (int)((w >> 16) & 0xffu); v[3] = (int)(w >> 24);
}
__device__ __forceinline__ uint32_t clip8(int acc) { return (uint32_t)clampi(acc >> kPrecisionBits, 0, 255); }

//
// MARG (SURVEY 8(f) N2, the fusion of llava.py:243-255 with new_method.py:215-216): the mask is not written at all;
// the kernel leaves the marginal sums of its bytes instead, in the partial layout of profiles.cu (P2b) -- column
// sums per (tile, row group) chunk in colpart[b][chunk][Wo], whole row sums in rowpart[b][0][Ho], each with the
// + 1e-9 per element of new_method.py:212 added as count x 1e-9 -- for maps_from_partials_kernel to finish.  All
// sums are exact integers (<= 255 x 65535), whatever the order the threads add them in.
// Measured (profiles/r03d_row_kernels.txt), for THIS kernel (resize_lanczos_up_mma_kernel below replaced it wherever
// its geometry fits, and there the fusion does save time): this saves the B x H x W buffer, not time -- the resize is bound by the
// fma pipe, so the write it skips was free, and the sums cost about what the separate marginals kernel does
// (256 x 336^2: 53.5 us fused vs 52.5 us in two steps; 64 x 1344^2: 188 vs 167 us).
constexpr int kUpMaxThreads = 512;
template <int TAPS, bool MARG>     // taps per axis actually used (7 for pure up-scaling)
__global__ void __launch_bounds__(kUpMaxThreads)
resize_lanczos_up_kernel(const uint8_t* __restrict__ src, int h, int w, int Ho, int Wo,
                         const int2* __restrict__ bx, const int* __restrict__ kx, int ksx,
                         const int2* __restrict__ by, const int* __restrict__ ky, int ksy,
                         int rows_per_tile, int n_rowgroups, uint8_t* __restrict__ dst,
                         double* __restrict__ colpart, double* __restrict__ rowpart) {
    extern __shared__ __align__(16) uint8_t sm_b[];
    const int Wp = (Wo + 3) & ~3;                        // pitch of the horizontal pass
    const int b = blockIdx.y;
    const int y0 = blockIdx.x * rows_per_tile, y1 = min(y0 + rows_per_tile, Ho);
    const int r0 = by[y0].x;
    const int nr = by[y1 - 1].x + by[y1 - 1].y - r0;     // source rows the tile taps: [r0, r0 + nr)
    int4* coef = reinterpret_cast<int4*>(sm_b);          // [rows_per_tile][2] int4: 8 coefficients per output row
    int* ymin = reinterpret_cast<int*>(sm_b + (size_t)rows_per_tile * 32);      // [rows_per_tile], relative to r0
    uint8_t* in = sm_b + (size_t)rows_per_tile * 36;                            // [nr][w]
    uint8_t* tmp = in + (((size_t)h * w + 15) & ~(size_t)15);                   // [nr][Wp]
    const uint8_t* img = src + ((int64_t)b * h + r0) * w;
    for (int i = threadIdx.x; i < nr * w; i += blockDim.x) in[i] = img[i];
    // MARG: the row sums of the tile are added up in shared memory
    int* rsum = reinterpret_cast<int*>(tmp + (((size_t)h * Wp + 15) & ~(size_t)15));   // [rows_per_tile], MARG only
    if (MARG)
        for (int i = threadIdx.x; i < y1 - y0; i += blockDim.x) rsum[i] = 0;
    for (int i = threadIdx.x; i < (y1 - y0) * kUpTaps; i += blockDim.x) {
        const int yy = i >> 3, t = i & 7;
        reinterpret_cast<int*>(coef)[i] = t < ksy ? __ldg(ky + (int64_t)(y0 + yy) * ksy + t) : 0;
        if (t == 0) ymin[yy] = by[y0 + yy].x - r0;
    }
    __syncthreads();
    for (int x = threadIdx.x; x < Wp; x += blockDim.x) {                      // horizontal pass, column x
        int k[TAPS], c0 = 0;
        if (x < Wo) c0 = bx[x].x;
#pragma unroll
        for (int t = 0; t < TAPS; ++t) k[t] = (x < Wo && t < ksx) ? __ldg(kx + (int64_t)x * ksx + t) : 0;
        for (int r = 0; r < nr; ++r) {
            int acc = 1 << (kPrecisionBits - 1);
#pragma unroll
            for (int t = 0; t < TAPS; ++t) acc += (int)in[r * w + min(c0 + t, w - 1)] * k[t];
            tmp[r * Wp + x] = (uint8_t)clip8(acc);
        }
    }
    __syncthreads();
    // vertical pass: thread = (row group, column group of 4)
    const int n_cg = Wp >> 2;
    const int rg = threadIdx.x / n_cg;
    // MARG: the lanes of this warp that work on the same row group (they add their row sums up with one REDUX)
    const unsigned peers = MARG ? __match_any_sync(0xffffffffu, rg) : 0u;
    if (!MARG && rg >= n_rowgroups) return;
    const int cg = threadIdx.x - rg * n_cg;
    const int rows = y1 - y0;
    const bool live = rg < n_rowgroups;
    const int ya = live ? (int)(((int64_t)rows * rg) / n_rowgroups) : 0;
    const int yb = live ? (int)(((int64_t)rows * (rg + 1)) / n_rowgroups) : 0;
    const bool vec = (Wo & 3) == 0 && (reinterpret_cast<uintptr_t>(dst) & 3) == 0;
    uint8_t* out = dst + ((int64_t)b * Ho + y0) * Wo;
    uint32_t csum[4] = {0u, 0u, 0u, 0u};
    {
        const int g = cg;               // one column group per thread (the launcher sizes the CTA so)
        int win[TAPS][4];
        int base = -1000;
        for (int yy = ya; yy < yb; ++yy) {
            const int ym = ymin[yy];
            if (ym != base) {
                if (ym == base + 1) {
#pragma unroll
                    for (int t = 0; t < TAPS - 1; ++t)
#pragma unroll
                        for (int q = 0; q < 4; ++q) win[t][q] = win[t + 1][q];
                    unpack4(*reinterpret_cast<const uint32_t*>(tmp + min(ym + TAPS - 1, nr - 1) * Wp + 4 * g), win[TAPS - 1]);
                } else {
#pragma unroll
                    for (int t = 0; t < TAPS; ++t)
                        unpack4(*reinterpret_cast<const uint32_t*>(tmp + min(ym + t, nr - 1) * Wp + 4 * g), win[t]);
                }
                base = ym;
            }
            const int4 ca = coef[2 * yy], cb = coef[2 * yy + 1];
            const int c[kUpTaps] = {ca.x, ca.y, ca.z, ca.w, cb.x, cb.y, cb.z, cb.w};
            int acc[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[q] = 1 << (kPrecisionBits - 1);
#pragma unroll
            for (int t = 0; t < TAPS; ++t)
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[q] += win[t][q] * c[t];
            // clip8 x 4 + pack: cvt.pack saturates two int32 to uint8 and packs them under the previous pair
            uint32_t hi2, o;
            asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(hi2) : "r"(acc[3] >> kPrecisionBits), "r"(acc[2] >> kPrecisionBits), "r"(0));
            asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(o) : "r"(acc[1] >> kPrecisionBits), "r"(acc[0] >> kPrecisionBits), "r"(hi2));
            if (MARG) {
                // columns >= Wo of the last group are zero (zero horizontal coefficients), so they add nothing
                csum[0] += o & 0xffu; csum[1] += (o >> 8) & 0xffu; csum[2] += (o >> 16) & 0xffu; csum[3] += o >> 24;
                const uint32_t part = __reduce_add_sync(peers, __dp4a(o, 0x01010101u, 0u));
                if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&rsum[yy], (int)part);
                continue;
            }
            uint8_t* p = out + (int64_t)yy * Wo + 4 * g;
            if (vec) {
                *reinterpret_cast<uint32_t*>(p) = o;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (4 * g + q < Wo) p[q] = (uint8_t)(o >> (8 * q));
            }
        }
    }
    if (MARG) {
        const int n_chunks = gridDim.x * n_rowgroups;
        if (live) {
            double* cp = colpart + ((int64_t)b * n_chunks + blockIdx.x * n_rowgroups + rg) * Wo;
            const double base = (double)(yb - ya) * kBaseAttention;
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (4 * cg + q < Wo) cp[4 * cg + q] = (double)csum[q] + base;
        }
        __syncthreads();
        const double row_base = (double)Wo * kBaseAttention;
        for (int i = threadIdx.x; i < rows; i += blockDim.x)
            rowpart[(int64_t)b * Ho + y0 + i] = (double)rsum[i] + row_base;
    }
}

// ---- the up-scaling case on the tensor cores -------------------------------------------------------------------
// The vertical pass of an up-scaling IS a matrix product: out[y][x] = clip8((sum_k Wv[y][k] tmp[k][x] + 2^21) >> 22)
// with Wv the [Ho x h] band matrix of 22-bit coefficients and tmp the [h x Wo] horizontal pass -- and the kernel above
// spends 7 IMAD per output byte on it (bound by the fma pipe at a fifth of the HBM rate).  Integer MMA is exact, so
// the product can go to the tensor cores bit for bit: a coefficient (|w| < 2^23) is split into three bytes
// w = b0 + 2^8 b1 + 2^16 b2 (b0, b1 unsigned, b2 signed), three mma.sync.m16n8k16 (s8 x u8, u8 x u8, u8 x u8) give
// exact int32 partial products (< 2^21 each), chained through the accumulator as ((A2 B << 8) + A1 B << 8) + 2^21 +
// A0 B: Pillow's int32 accumulator (two's-complement wrap-around of the shifted parts cancels, the true sum fits;
// tests/test_mask_path.py::test_byte_plane_horner_equals_the_int32_accumulator checks the arithmetic on the host).
// K = 16 source rows: a tile of output rows taps at
// most 16 of them (the launcher sizes the tiles so), all relative to the tile's first tapped row.
//   CTA  = (tile of output rows) x (up to 8 strips of 64 columns), one warp per strip;
//   tmpT [column][16] bytes: the horizontal pass of the tile's source rows, transposed, so that a B fragment
//        (4 consecutive source rows of one column) is one aligned 32-bit shared load; a warp keeps its 8 B fragments
//        (64 columns) in registers for the whole tile;
//   Apl  [3][row][16] bytes: the byte planes of the coefficient band (copied from the table get_planes built once per
//        (h, Ho, rows per tile)), an A fragment is two 32-bit loads per plane;
//   the 8 column tiles of a strip interleave their columns (tile j holds columns 16 c + 2 j, + 1 of the strip) so
//   that a thread ends up with 16 ADJACENT output bytes of rows g and g + 8: two 128-bit stores per 16 x 64 block.
// Measured (profiles/r06h_row_kernels.txt, r06i ncu): 176 warp instructions per 16 x 64 block (24 IMMA, 62 shift-adds
// of the Horner combination, 32 shifts, 16 saturating packs) instead of ~10 per byte; revise + resize 64 x 24^2 ->
// 1344^2 127 -> 52 us, 256 x 24^2 -> 336^2 37 -> 27 us; with MARG the fused mask -> maps path 188 -> 73 us
// (profiles/r08e_row_kernels.txt).  Issue slots 58 % busy, tensor pipe 44 %, DRAM 13 %: still not its output stream.
constexpr int kMmaK = 16, kMmaStrip = 64, kMmaMaxWarps = 8;
__device__ __forceinline__ void mma_u8u8(int (&d)[4], const uint32_t (&a)[2], uint32_t b) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                 : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(b));
}
__device__ __forceinline__ void mma_s8u8(int (&d)[4], const uint32_t (&a)[2], uint32_t b) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.s32.s8.u8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                 : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(b));
}
// MARG (the fusion of llava.py:243-255 with new_method.py:215-216, as resize_lanczos_up_kernel<., true>): the mask is
// not written; column sums go to colpart [b][row tile][Wo], row sums to rowpart [b][x CTA][Ho] (exact integers).
// One CTA's tile: output rows [y0, y0 + rows_per_tile) x columns [x_base, x_base + 64 n_warps) of one image.  img: the
// image's [h][w] mask; planes: the tile's byte planes; out_img: the image's [Ho][Wo] mask (!MARG); cp: the column
// partials of the tile's chunk (indexed by column), rp: the row partials of the CTA's columns (indexed by y - y0).
// Warps from n_warps on (a ragged CTA is sized for the widest image) only take part in the horizontal pass.
template <bool MARG>
__device__ __forceinline__ void lanczos_up_mma_tile(const uint8_t* __restrict__ img, int w, int Ho, int Wo,
                                                    const int2* __restrict__ bx, const int* __restrict__ kx, int ksx,
                                                    const int2* __restrict__ by, const uint8_t* __restrict__ planes,
                                                    int rows_per_tile, int n_warps, int x_base, int y0,
                                                    uint8_t* __restrict__ out_img, double* __restrict__ cp,
                                                    double* __restrict__ rp) {
    extern __shared__ __align__(16) uint8_t sm_b[];
    const int cols_cta = n_warps * kMmaStrip;
    const int y1 = min(y0 + rows_per_tile, Ho);
    const int r0 = by[y0].x;
    const int nr = by[y1 - 1].x + by[y1 - 1].y - r0;     // source rows the tile taps: [r0, r0 + nr), nr <= 16
    uint8_t* tmpT = sm_b;                                              // [cols_cta][16]
    uint8_t* apl = tmpT + (size_t)cols_cta * kMmaK;                    // [3][rows_per_tile][16]
    int* rsum = reinterpret_cast<int*>(apl + (size_t)3 * rows_per_tile * kMmaK);   // [rows_per_tile] (MARG)
    uint8_t* in = reinterpret_cast<uint8_t*>(rsum + rows_per_tile);    // [nr][w]
    const uint8_t* src = img + (int64_t)r0 * w;
    for (int i = threadIdx.x; i < nr * w; i += blockDim.x) in[i] = src[i];
    {   // the coefficient band of this tile, byte planes (get_planes built them once)
        const uint4* pl = reinterpret_cast<const uint4*>(planes);
        for (int i = threadIdx.x; i < 3 * rows_per_tile; i += blockDim.x) reinterpret_cast<uint4*>(apl)[i] = __ldg(pl + i);
    }
    if (MARG)
        for (int i = threadIdx.x; i < rows_per_tile; i += blockDim.x) rsum[i] = 0;
    __syncthreads();
    for (int xl = threadIdx.x; xl < cols_cta; xl += blockDim.x) {          // horizontal pass, column x, transposed
        const int x = x_base + xl;
        uint32_t packed[4] = {0u, 0u, 0u, 0u};
        if (x < Wo) {
            int k[kUpTaps];
            const int c0 = bx[x].x;
#pragma unroll
            for (int t = 0; t < kUpTaps; ++t) k[t] = t < ksx ? __ldg(kx + (int64_t)x * ksx + t) : 0;
#pragma unroll
            for (int r = 0; r < kMmaK; ++r) {            // (unrolled: packed[] stays in registers)
                if (r < nr) {
                    int acc = 1 << (kPrecisionBits - 1);
#pragma unroll
                    for (int t = 0; t < kUpTaps; ++t) acc += (int)in[r * w + min(c0 + t, w - 1)] * k[t];
                    packed[r >> 2] |= clip8(acc) << (8 * (r & 3));
                }
            }
        }
        *reinterpret_cast<uint4*>(tmpT + (size_t)xl * kMmaK) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
    }
    __syncthreads();
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    const int xs = x_base + wid * kMmaStrip;             // the warp's strip of 64 columns
    const bool strip = wid < n_warps && xs < Wo;
    if (!MARG && !strip) return;
    if (strip) {
    uint32_t bf[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int xl = wid * kMmaStrip + 16 * (g >> 1) + 2 * j + (g & 1);
        bf[j] = *reinterpret_cast<const uint32_t*>(tmpT + (size_t)xl * kMmaK + 4 * tig);
    }
    const bool store_ok = xs + 16 * tig < Wo;            // Wo is a multiple of 16: whole 16-byte groups
    uint8_t* out = MARG ? nullptr : out_img + (int64_t)y0 * Wo + xs + 16 * tig;
    // MARG: column sums of the thread's 16 columns over its rows, two columns per register (16-bit lanes:
    // <= 2 rows x 32 blocks x 255); csum[2 m] = columns 4 m, 4 m + 2, csum[2 m + 1] = columns 4 m + 1, 4 m + 3
    uint32_t csum[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    for (int m0 = 0; m0 < y1 - y0; m0 += 16) {
        uint32_t a[3][2];
#pragma unroll
        for (int p = 0; p < 3; ++p) {
            a[p][0] = *reinterpret_cast<const uint32_t*>(apl + ((size_t)p * rows_per_tile + m0 + g) * kMmaK + 4 * tig);
            a[p][1] = *reinterpret_cast<const uint32_t*>(apl + ((size_t)p * rows_per_tile + m0 + g + 8) * kMmaK + 4 * tig);
        }
        uint32_t lo[4], hi[4];                           // 16 bytes of row m0 + g, of row m0 + g + 8
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            int v[2][4];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                // Horner over the byte planes: ((A2 B) 2^8 + A1 B) 2^8 + A0 B + 2^21, the accumulator chained through
                // the three MMAs (int32 wrap-around as in the flat sum)
                int d[4] = {0, 0, 0, 0};
                mma_s8u8(d, a[2], bf[2 * jj + q]);
#pragma unroll
                for (int i = 0; i < 4; ++i) d[i] = (int)((uint32_t)d[i] << 8);
                mma_u8u8(d, a[1], bf[2 * jj + q]);
#pragma unroll
                for (int i = 0; i < 4; ++i) d[i] = (int)(((uint32_t)d[i] << 8) + (1u << (kPrecisionBits - 1)));
                mma_u8u8(d, a[0], bf[2 * jj + q]);
#pragma unroll
                for (int i = 0; i < 4; ++i) v[q][i] = d[i] >> kPrecisionBits;
            }
            // cvt.pack saturates two int32 to uint8 and packs them under the previous pair: bytes 4 jj .. 4 jj + 3
            uint32_t t;
            asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(v[1][1]), "r"(v[1][0]), "r"(0));
            asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(lo[jj]) : "r"(v[0][1]), "r"(v[0][0]), "r"(t));
            asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(v[1][3]), "r"(v[1][2]), "r"(0));
            asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(hi[jj]) : "r"(v[0][3]), "r"(v[0][2]), "r"(t));
        }
        if (MARG) {
            // rows past the tile's end have zero coefficients: their bytes are 0 and add nothing
            uint32_t rlo = 0u, rhi = 0u;
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                rlo = __dp4a(lo[m], 0x01010101u, rlo);
                rhi = __dp4a(hi[m], 0x01010101u, rhi);
                csum[2 * m] += (lo[m] & 0x00ff00ffu) + (hi[m] & 0x00ff00ffu);
                csum[2 * m + 1] += ((lo[m] >> 8) & 0x00ff00ffu) + ((hi[m] >> 8) & 0x00ff00ffu);
            }
            rlo += __shfl_xor_sync(0xffffffffu, rlo, 1);
            rhi += __shfl_xor_sync(0xffffffffu, rhi, 1);
            rlo += __shfl_xor_sync(0xffffffffu, rlo, 2);
            rhi += __shfl_xor_sync(0xffffffffu, rhi, 2);
            if (tig == 0) {
                atomicAdd(&rsum[m0 + g], (int)rlo);
                atomicAdd(&rsum[m0 + g + 8], (int)rhi);
            }
        } else if (store_ok) {
            if (m0 + g < y1 - y0)
                *reinterpret_cast<uint4*>(out + (int64_t)(m0 + g) * Wo) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            if (m0 + g + 8 < y1 - y0)
                *reinterpret_cast<uint4*>(out + (int64_t)(m0 + g + 8) * Wo) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        }
    }
    if (MARG) {
        // column sums: add up the 8 row groups g (lanes 4 apart hold the same columns), then lanes g == 0 write their
        // 16 columns of this tile's chunk; the + 1e-9 per element of new_method.py:212 is added as count x 1e-9
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            uint32_t lo16 = csum[m] & 0xffffu, hi16 = csum[m] >> 16;
#pragma unroll
            for (int d = 4; d < 32; d <<= 1) {
                lo16 += __shfl_xor_sync(0xffffffffu, lo16, d);
                hi16 += __shfl_xor_sync(0xffffffffu, hi16, d);
            }
            if (g == 0) {
                const double base = (double)(y1 - y0) * kBaseAttention;
                const int c = xs + 16 * tig + 4 * (m >> 1) + (m & 1);       // and c + 2
                if (c < Wo) cp[c] = (double)lo16 + base;
                if (c + 2 < Wo) cp[c + 2] = (double)hi16 + base;
            }
        }
    }
    }   // strip
    if (MARG) {
        // the row sums of the CTA's columns: one partial per column range
        __syncthreads();
        const int cols = min(cols_cta, Wo - x_base);
        const double row_base = (double)cols * kBaseAttention;
        for (int i = threadIdx.x; i < y1 - y0; i += blockDim.x) rp[i] = (double)rsum[i] + row_base;
    }
}

template <bool MARG>
__global__ void __launch_bounds__(kMmaMaxWarps * 32)
resize_lanczos_up_mma_kernel(const uint8_t* __restrict__ src, int h, int w, int Ho, int Wo,
                             const int2* __restrict__ bx, const int* __restrict__ kx, int ksx,
                             const int2* __restrict__ by, const uint8_t* __restrict__ planes, int rows_per_tile,
                             uint8_t* __restrict__ dst, double* __restrict__ colpart, double* __restrict__ rowpart) {
    const int b = blockIdx.z, y0 = blockIdx.y * rows_per_tile, n_warps = blockDim.x >> 5;
    lanczos_up_mma_tile<MARG>(src + (int64_t)b * h * w, w, Ho, Wo, bx, kx, ksx, by,
                              planes + (size_t)blockIdx.y * 3 * rows_per_tile * kMmaK, rows_per_tile, n_warps,
                              blockIdx.x * n_warps * kMmaStrip, y0, MARG ? nullptr : dst + (int64_t)b * Ho * Wo,
                              MARG ? colpart + ((int64_t)b * gridDim.y + blockIdx.y) * Wo : nullptr,
                              MARG ? rowpart + ((int64_t)b * gridDim.x + blockIdx.x) * Ho + y0 : nullptr);
}

// The marginals variant over a ragged list of masks (attwarp_warp_ragged_from_mask) in one launch: CTA = item
// (image, row tile << 8 | column CTA) of a host-built table.  Every image keeps the tiles, column CTAs and coefficient
// planes a call on it alone uses (lanczos_ragged_geometry) and writes its partials where its RaggedAtt says, in the
// layout the ragged finish kernel reads: [row tiles][W] column and [column CTAs][H] row partials.  So its partials, and
// its maps, are those of attwarp_maps_from_mask on that image alone, whatever the rest of the list.
__global__ void __launch_bounds__(kMmaMaxWarps * 32)
resize_lanczos_up_mma_ragged_kernel(const int2* __restrict__ items, const RaggedAtt* __restrict__ atts,
                                    const RaggedLanczos* __restrict__ lz, int w, double* __restrict__ part) {
    const int2 it = items[blockIdx.x];
    const RaggedAtt& a = atts[it.x];
    const RaggedLanczos& l = lz[it.x];
    const int tile = it.y >> 8, xc = it.y & 255, rows = a.chunk_rows, y0 = tile * rows;
    lanczos_up_mma_tile<true>(static_cast<const uint8_t*>(a.att), w, a.H, a.W, l.bx, l.kx, l.ksx, l.by,
                              l.planes + (size_t)tile * 3 * rows * kMmaK, rows, l.warps, xc * a.tile_cols, y0, nullptr,
                              part + a.colpart + (int64_t)tile * a.W, part + a.rowpart + (int64_t)xc * a.H + y0);
}

// ---- coefficient tables (Resample.c precompute_coeffs + normalize_coeffs_8bpc, Lanczos, support 3) ----
double sinc_filter(double x) {
    if (x == 0.0) return 1.0;
    x = x * M_PI;
    return sin(x) / x;
}
double lanczos_filter(double x) { return (-3.0 <= x && x < 3.0) ? sinc_filter(x) * sinc_filter(x / 3.0) : 0.0; }

struct CoeffTable {
    int2* bounds = nullptr;     // device
    int* weights = nullptr;     // device
    int ksize = 0;
};

// Resample.c precompute_coeffs + normalize_coeffs_8bpc on the host: bounds [out] = {first tap, taps}, kk [out][ksize]
static int compute_table(int in_size, int out_size, std::vector<int2>& bounds, std::vector<int>& kk) {
    const double scale = (double)in_size / (double)out_size;
    const double fscale = scale < 1.0 ? 1.0 : scale;
    const double support = 3.0 * fscale;
    const int ksize = (int)ceil(support) * 2 + 1;
    bounds.assign((size_t)out_size, make_int2(0, 0));
    kk.assign((size_t)out_size * ksize, 0);
    std::vector<double> w((size_t)ksize);
    const double ss = 1.0 / fscale;
    for (int xx = 0; xx < out_size; ++xx) {
        const double center = (xx + 0.5) * scale;
        int xmin = (int)(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = (int)(center + support + 0.5);
        if (xmax > in_size) xmax = in_size;
        xmax -= xmin;
        double ww = 0.0;
        for (int x = 0; x < xmax; ++x) {
            w[(size_t)x] = lanczos_filter((x + xmin - center + 0.5) * ss);
            ww += w[(size_t)x];
        }
        for (int x = 0; x < xmax; ++x) {
            const double v = ww != 0.0 ? w[(size_t)x] / ww : w[(size_t)x];
            kk[(size_t)xx * ksize + x] = v < 0 ? (int)(-0.5 + v * (1 << kPrecisionBits)) : (int)(0.5 + v * (1 << kPrecisionBits));
        }
        bounds[(size_t)xx] = make_int2(xmin, xmax);
    }
    return ksize;
}

int build_table(int in_size, int out_size, CoeffTable* t) {
    std::vector<int2> bounds;
    std::vector<int> kk;
    const int ksize = compute_table(in_size, out_size, bounds, kk);
    AW_CUDA(cudaMalloc(&t->bounds, sizeof(int2) * (size_t)out_size));
    AW_CUDA(cudaMalloc(&t->weights, sizeof(int) * kk.size()));
    AW_CUDA(cudaMemcpy(t->bounds, bounds.data(), sizeof(int2) * (size_t)out_size, cudaMemcpyHostToDevice));
    AW_CUDA(cudaMemcpy(t->weights, kk.data(), sizeof(int) * kk.size(), cudaMemcpyHostToDevice));
    t->ksize = ksize;
    return ATTWARP_OK;
}

// Tables are constants of (device, in, out): built once (synchronous upload) and kept for the life of the
// process, so later calls on any stream only read them.
int get_table(int in_size, int out_size, CoeffTable* out) {
    static std::mutex mu;
    static std::map<std::pair<int, std::pair<int, int>>, CoeffTable> cache;
    int dev = 0;
    AW_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    const auto key = std::make_pair(dev, std::make_pair(in_size, out_size));
    auto it = cache.find(key);
    if (it == cache.end()) {
        CoeffTable t;
        const int rc = build_table(in_size, out_size, &t);
        if (rc != ATTWARP_OK) return rc;
        it = cache.emplace(key, t).first;
    }
    *out = it->second;
    return ATTWARP_OK;
}

// The byte planes of the vertical coefficient band for the tensor-core kernel, per tile of `rows` output rows:
// [tile][plane][row][16] bytes, k relative to the tile's first tapped source row.  Constants of (device, h, Ho, rows),
// built once like the tables (the CTAs used to rebuild their slice from the int32 table: a sixth of the kernel's
// instructions).
int get_planes(int h, int Ho, int rows, const uint8_t** out) {
    static std::mutex mu;
    static std::map<std::pair<std::pair<int, int>, std::pair<int, int>>, uint8_t*> cache;
    int dev = 0;
    AW_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    const auto key = std::make_pair(std::make_pair(dev, h), std::make_pair(Ho, rows));
    auto it = cache.find(key);
    if (it == cache.end()) {
        std::vector<int2> bounds;
        std::vector<int> kk;
        const int ksize = compute_table(h, Ho, bounds, kk);
        const int n_tiles = (Ho + rows - 1) / rows;
        std::vector<uint8_t> planes((size_t)n_tiles * 3 * rows * kMmaK, 0);
        for (int t = 0; t < n_tiles; ++t) {
            const int y0 = t * rows, r0 = bounds[(size_t)y0].x;
            for (int yy = 0; yy < rows && y0 + yy < Ho; ++yy) {
                const int2 bd = bounds[(size_t)(y0 + yy)];
                for (int tap = 0; tap < bd.y; ++tap) {
                    const int k = bd.x - r0 + tap;
                    if (k < 0 || k >= kMmaK) return fail(ATTWARP_ERR_UNSUPPORTED, "lanczos planes: a tile of %d rows taps more than %d source rows", rows, kMmaK);
                    const int wv = kk[(size_t)(y0 + yy) * ksize + tap];
                    for (int p = 0; p < 3; ++p)
                        planes[(((size_t)t * 3 + p) * rows + yy) * kMmaK + k] = (uint8_t)((wv >> (8 * p)) & 0xff);
                }
            }
        }
        uint8_t* d = nullptr;
        AW_CUDA(cudaMalloc(&d, planes.size()));
        AW_CUDA(cudaMemcpy(d, planes.data(), planes.size(), cudaMemcpyHostToDevice));
        it = cache.emplace(key, d).first;
    }
    *out = it->second;
    return ATTWARP_OK;
}

}  // namespace

int launch_revise_mask(const float* tok, int B, int gh, int gw, int ksize, float coe, float* revised,
                       uint8_t* mask_u8, cudaStream_t st) {
    const size_t smem = sizeof(float) * (size_t)gh * gw;
    if (smem > 160 * 1024) return fail(ATTWARP_ERR_UNSUPPORTED, "revise_mask: token grid %dx%d too large", gh, gw);
    if (smem > 48 * 1024)
        AW_CUDA(cudaFuncSetAttribute(revise_mask_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    revise_mask_kernel<<<B, kMaskThreads, smem, st>>>(tok, gh, gw, ksize, coe, revised, mask_u8);
    return check_launch("revise_mask_kernel");
}

// Launch geometry of the up-scaling kernel: tiles of `rows` output rows (enough CTAs to fill the GPU, as tall as
// possible: the horizontal pass is redone per tile), n_rg row groups of Wp / 4 threads each.
struct UpGeometry { bool ok; int n_tiles, rows, n_rg, threads; size_t smem; };
static UpGeometry up_geometry(int B, int h, int w, int Ho, int Wo) {
    UpGeometry g{};
    const int Wp = (Wo + 3) & ~3, n_cg = Wp / 4;
    if (n_cg > kUpMaxThreads) return g;
    int n_tiles = (2 * sm_count() + B - 1) / B;
    n_tiles = n_tiles < 1 ? 1 : n_tiles;
    if (n_tiles > (Ho + 31) / 32) n_tiles = (Ho + 31) / 32;
    g.rows = (Ho + n_tiles - 1) / n_tiles;
    g.n_tiles = (Ho + g.rows - 1) / g.rows;
    g.n_rg = kUpMaxThreads / n_cg;
    g.threads = (n_cg * g.n_rg + 31) & ~31;
    // coefficients + first taps | source rows | horizontal pass | row sums (MARG)
    g.smem = (size_t)g.rows * 36 + (((size_t)h * w + 15) & ~(size_t)15) + (((size_t)h * Wp + 15) & ~(size_t)15) +
             (size_t)g.rows * 4;
    g.ok = g.smem <= 200 * 1024;
    return g;
}

// Pillow's window of output coordinate xx (Resample.c precompute_coeffs, as build_table above): first tap, taps.
static void tap_window(int in_size, int out_size, int xx, int* first, int* count) {
    const double scale = (double)in_size / (double)out_size;
    const double fscale = scale < 1.0 ? 1.0 : scale;
    const double support = 3.0 * fscale;
    const double center = (xx + 0.5) * scale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    *first = xmin;
    *count = xmax - xmin;
}

// Launch geometry of the tensor-core up-scaling kernel: strips of 64 columns, one warp each, up to 8 per CTA; tiles
// of `rows` output rows (a multiple of 16) that tap at most 16 source rows; enough CTAs to fill the GPU a few times.
struct MmaGeometry { bool ok; int x_ctas, warps, rows, n_tiles; size_t smem; };
static MmaGeometry mma_geometry(int B, int h, int w, int Ho, int Wo, const uint8_t* dst, bool marg) {
    MmaGeometry g{};
    if (w > 1024 || B > 65535) return g;
    // the mask is stored in 16-byte groups; the marginals variant stores nothing and takes any width
    if (!marg && ((Wo & 15) != 0 || (reinterpret_cast<uintptr_t>(dst) & 15) != 0)) return g;
    const int strips = (Wo + kMmaStrip - 1) / kMmaStrip;
    g.x_ctas = (strips + kMmaMaxWarps - 1) / kMmaMaxWarps;
    g.warps = (strips + g.x_ctas - 1) / g.x_ctas;
    int want_tiles = (4 * sm_count() + B * g.x_ctas - 1) / (B * g.x_ctas);
    if (want_tiles < 1) want_tiles = 1;
    int rows = ((Ho + want_tiles - 1) / want_tiles + 15) & ~15;
    if (rows < 32) rows = 32;
    if (rows > 512) rows = 512;
    for (; rows >= 16; rows -= 16) {                     // the tallest tile whose rows tap <= 16 source rows
        bool fits = true;
        for (int y0 = 0; y0 < Ho && fits; y0 += rows) {
            const int y1 = (y0 + rows < Ho ? y0 + rows : Ho) - 1;
            int f0, c0, f1, c1;
            tap_window(h, Ho, y0, &f0, &c0);
            tap_window(h, Ho, y1, &f1, &c1);
            fits = f1 + c1 - f0 <= kMmaK;
        }
        if (fits) break;
    }
    if (rows < 16) return g;
    g.rows = rows;
    g.n_tiles = (Ho + rows - 1) / rows;
    if (g.n_tiles > 65535) return g;
    g.smem = (size_t)g.warps * kMmaStrip * kMmaK + (size_t)3 * rows * kMmaK + (size_t)rows * 4 + (((size_t)kMmaK * w + 15) & ~(size_t)15);
    g.ok = g.smem <= 160 * 1024;
    return g;
}
static bool lanczos_mma_enabled() {
    static const bool v = [] {
        const char* e = getenv("ATTWARP_LANCZOS_MMA");
        return e == nullptr || e[0] != '0';
    }();
    return v;
}

// Partial sums per image the fused kernel writes: column-sum chunks (0: this resize is not taken by the fused kernel)
// and row-sum partials (column tiles).  The tensor-core kernel when its geometry fits, else the register-window one.
int lanczos_marginals_chunks(int B, int h, int w, int H, int W, int* n_col_tiles) {
    *n_col_tiles = 1;
    if (H <= h || W <= w || h > 0xffff || w > 0xffff) return 0;
    if (lanczos_mma_enabled()) {
        const MmaGeometry mg = mma_geometry(B, h, w, H, W, nullptr, true);
        if (mg.ok) {
            *n_col_tiles = mg.x_ctas;
            return mg.n_tiles;
        }
    }
    // pure up-scaling: 3 * 2 + 1 = 7 taps per axis
    const UpGeometry g = up_geometry(B, h, w, H, W);
    return g.ok ? g.n_tiles * g.n_rg : 0;
}

// mask_u8 [B][h][w] (revise_mask's uint8 output) -> marginal partial sums of its LANCZOS resize to H x W, which is
// never written: colpart [B][chunks][W], rowpart [B][1][H].
int launch_lanczos_marginals(const uint8_t* src, int B, int h, int w, int H, int W, double* colpart, double* rowpart,
                             int* n_chunks, int* n_col_tiles, cudaStream_t st) {
    *n_col_tiles = 1;
    if (H > h && W > w && lanczos_mma_enabled()) {
        const MmaGeometry mg = mma_geometry(B, h, w, H, W, nullptr, true);
        CoeffTable tx, ty;
        if (mg.ok) {
            int rc = get_table(w, W, &tx);
            if (rc != ATTWARP_OK) return rc;
            rc = get_table(h, H, &ty);
            if (rc != ATTWARP_OK) return rc;
        }
        if (mg.ok && tx.ksize <= kUpTaps && ty.ksize <= kUpTaps) {
            if (mg.smem > 48 * 1024)
                AW_CUDA(cudaFuncSetAttribute(resize_lanczos_up_mma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mg.smem));
            const uint8_t* planes = nullptr;
            const int prc = get_planes(h, H, mg.rows, &planes);
            if (prc != ATTWARP_OK) return prc;
            resize_lanczos_up_mma_kernel<true><<<dim3(mg.x_ctas, mg.n_tiles, B), mg.warps * 32, mg.smem, st>>>(
                src, h, w, H, W, tx.bounds, tx.weights, tx.ksize, ty.bounds, planes, mg.rows, nullptr, colpart, rowpart);
            *n_chunks = mg.n_tiles;
            *n_col_tiles = mg.x_ctas;
            return check_launch("resize_lanczos_up_mma_kernel<marginals>");
        }
    }
    const UpGeometry ug = up_geometry(B, h, w, H, W);
    if (H <= h || W <= w || !ug.ok)
        return fail(ATTWARP_ERR_UNSUPPORTED, "lanczos_marginals: %dx%d -> %dx%d is not an up-scaling that fits shared memory", h, w, H, W);
    CoeffTable tx, ty;
    int rc = get_table(w, W, &tx);
    if (rc != ATTWARP_OK) return rc;
    rc = get_table(h, H, &ty);
    if (rc != ATTWARP_OK) return rc;
    if (tx.ksize > 7 || ty.ksize > 7) return fail(ATTWARP_ERR_UNSUPPORTED, "lanczos_marginals: too many taps");
    auto kern = resize_lanczos_up_kernel<7, true>;
    if (ug.smem > 48 * 1024)
        AW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ug.smem));
    kern<<<dim3(ug.n_tiles, B), ug.threads, ug.smem, st>>>(
        src, h, w, H, W, tx.bounds, tx.weights, tx.ksize, ty.bounds, ty.weights, ty.ksize, ug.rows, ug.n_rg, nullptr,
        colpart, rowpart);
    *n_chunks = ug.n_tiles * ug.n_rg;
    return check_launch("resize_lanczos_up_kernel<marginals>");
}

// The route launch_lanczos_marginals takes for B = 1, restated without the device: the tensor-core kernel when it is
// enabled and its geometry fits (an up-scaling has 7 taps per axis, within kUpTaps).
bool lanczos_ragged_geometry(int h, int w, int H, int W, int* rows, int* n_tiles, int* x_ctas, int* warps, size_t* smem) {
    if (H <= h || W <= w || h > 0xffff || w > 0xffff || !lanczos_mma_enabled()) return false;
    const MmaGeometry mg = mma_geometry(1, h, w, H, W, nullptr, true);
    if (!mg.ok || mg.x_ctas > 255) return false;
    *rows = mg.rows;
    *n_tiles = mg.n_tiles;
    *x_ctas = mg.x_ctas;
    *warps = mg.warps;
    *smem = mg.smem;
    return true;
}

int lanczos_ragged_tables(int h, int w, int H, int W, int rows, RaggedLanczos* l) {
    CoeffTable tx, ty;
    int rc = get_table(w, W, &tx);
    if (rc != ATTWARP_OK) return rc;
    rc = get_table(h, H, &ty);
    if (rc != ATTWARP_OK) return rc;
    if (tx.ksize > kUpTaps || ty.ksize > kUpTaps)
        return fail(ATTWARP_ERR_UNSUPPORTED, "lanczos_marginals: %dx%d -> %dx%d has more than %d taps", h, w, H, W, kUpTaps);
    l->bx = tx.bounds;
    l->kx = tx.weights;
    l->ksx = tx.ksize;
    l->by = ty.bounds;
    return get_planes(h, H, rows, &l->planes);
}

int launch_lanczos_marginals_ragged(const int2* dev_items, int64_t n_items, const RaggedAtt* dev_att,
                                    const RaggedLanczos* dev_lz, int w, size_t smem, double* partials, cudaStream_t st) {
    if (n_items <= 0 || n_items > 0x7fffffff)
        return fail(ATTWARP_ERR_UNSUPPORTED, "lanczos_marginals_ragged: %lld work items", (long long)n_items);
    if (smem > 48 * 1024)
        AW_CUDA(cudaFuncSetAttribute(resize_lanczos_up_mma_ragged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    resize_lanczos_up_mma_ragged_kernel<<<(unsigned)n_items, kMmaMaxWarps * 32, smem, st>>>(dev_items, dev_att, dev_lz, w,
                                                                                           partials);
    return check_launch("resize_lanczos_up_mma_ragged_kernel");
}

int launch_resize_lanczos_u8(const uint8_t* src, int B, int h, int w, int Ho, int Wo, uint8_t* dst, cudaStream_t st) {
    CoeffTable tx, ty;
    if (Wo != w) {
        const int rc = get_table(w, Wo, &tx);
        if (rc != ATTWARP_OK) return rc;
    }
    if (Ho != h) {
        const int rc = get_table(h, Ho, &ty);
        if (rc != ATTWARP_OK) return rc;
    }
    // pure up-scaling of both axes (7 taps), 16-byte aligned output rows: the vertical pass on the tensor cores
    if (Wo > w && Ho > h && tx.ksize <= kUpTaps && ty.ksize <= kUpTaps && lanczos_mma_enabled()) {
        const MmaGeometry mg = mma_geometry(B, h, w, Ho, Wo, dst, false);
        if (mg.ok) {
            if (mg.smem > 48 * 1024)
                AW_CUDA(cudaFuncSetAttribute(resize_lanczos_up_mma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mg.smem));
            const uint8_t* planes = nullptr;
            const int prc = get_planes(h, Ho, mg.rows, &planes);
            if (prc != ATTWARP_OK) return prc;
            resize_lanczos_up_mma_kernel<false><<<dim3(mg.x_ctas, mg.n_tiles, B), mg.warps * 32, mg.smem, st>>>(
                src, h, w, Ho, Wo, tx.bounds, tx.weights, tx.ksize, ty.bounds, planes, mg.rows, dst, nullptr, nullptr);
            return check_launch("resize_lanczos_up_mma_kernel");
        }
    }
    // up-scaling of both axes (7 taps each) the tensor-core kernel declined: the register-window kernel
    const UpGeometry ug = up_geometry(B, h, w, Ho, Wo);
    if (Wo != w && Ho != h && tx.ksize <= 7 && ty.ksize <= 7 && ug.ok) {
        auto kern = resize_lanczos_up_kernel<7, false>;
        if (ug.smem > 48 * 1024)
            AW_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ug.smem));
        kern<<<dim3(ug.n_tiles, B), ug.threads, ug.smem, st>>>(
            src, h, w, Ho, Wo, tx.bounds, tx.weights, tx.ksize, ty.bounds, ty.weights, ty.ksize, ug.rows, ug.n_rg, dst,
            nullptr, nullptr);
        return check_launch("resize_lanczos_up_kernel");
    }
    // shared memory: the source rows a tile taps (at most all of them) + their horizontal pass
    const size_t smem = (((size_t)h * w + 15) & ~(size_t)15) + (size_t)h * Wo;
    if (smem > 200 * 1024)
        return fail(ATTWARP_ERR_UNSUPPORTED, "resize_lanczos: %dx%d -> width %d does not fit shared memory", h, w, Wo);
    if (smem > 48 * 1024)
        AW_CUDA(cudaFuncSetAttribute(resize_lanczos_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    resize_lanczos_u8_kernel<<<dim3((Ho + kResizeRows - 1) / kResizeRows, B), kMaskThreads, smem, st>>>(
        src, h, w, Ho, Wo, tx.bounds, tx.weights, tx.ksize, ty.bounds, ty.weights, ty.ksize, dst);
    return check_launch("resize_lanczos_u8_kernel");
}

}  // namespace aw
