// overlay.cu -- the JET attention overlay save_warped_image writes (AGW/new_method.py, mirrored in
// attwarp_b200/new_method.py:save_warped_image) for a list of images of any sizes, in two launches.
//
// For a uint8 BGR (or grey, replicated) image and an attention map `a` of the image's size:
//   lo, hi = min(a), max(a)                    (NumPy: a NaN anywhere makes both NaN)
//   n      = (a - lo) / (hi - lo) if hi > lo + 1e-9 else 0
//   idx    = uint8(trunc(n * 255));  heat = JET[idx]
//   out    = saturate_u8(round_half_even(fmaf(heat, a32, base * b32)))   (cv2.addWeighted, gamma 0)
// in the precision NumPy 2 promotion gives each attention dtype: uint8 maps subtract in uint8 and divide, scale
// and compare in float64; float32 maps do everything in float32 (lo + 1e-9 included); float64 maps in float64.
// Every step is IEEE-exact, so the output is bit-identical to the host expression: the arithmetic uses explicit
// __f*_rn / __d*_rn intrinsics so that contraction cannot change it.
//
//   overlay_minmax_kernel<T>         one CTA per kMMChunk attention values of each image -> a (lo, hi) partial
//   overlay_minmax_tokens_kernel     token mode: one CTA per image, over the tokens the index upsampling reaches
//   overlay_blend_kernel<T, kVec>    one CTA per kBlendPix pixels of each image: the image's partials reduced,
//   overlay_blend_tokens_kernel<kVec>  normalise -> JET -> blend; kVec: 4 pixels per thread with 32-bit (image,
//                                    output, uint8 map) or 128-bit (float maps) accesses, when every base allows
//                                    them; otherwise one pixel per thread with byte accesses
#include <math.h>

#include <type_traits>
#include <vector>

#include "common.cuh"

namespace aw {

namespace {

constexpr int kMMThreads = 256;
constexpr int kMMChunk = 65536;                // attention values per min/max CTA (a multiple of 16)
constexpr int kBlendThreads = 256;
constexpr int kBlendPix = 4096;                // pixels per blend CTA: 4 rounds of 4 pixels per thread

// one image (device table; entry n is a sentinel carrying the totals in mm_begin / blk_begin)
struct OverlayImage {
    const uint8_t* src;                        // [H][W][C]
    const void* att;                           // [H][W] map, or the image's [gh][gw] float32 token map
    uint8_t* dst;                              // [H][W][3] BGR
    int32_t H, W, C;
    int32_t mm_begin;                          // first min/max partial of the image
    int32_t blk_begin;                         // first blend CTA of the image
    int32_t pad;
};
static_assert(sizeof(OverlayImage) == 48, "descriptor layout");

// cv2.applyColorMap(COLORMAP_JET) (OpenCV 4.13): entry i is B | G << 8 | R << 16
__device__ const uint32_t kJet[256] = {
    0x000080, 0x000084, 0x000088, 0x00008c, 0x000090, 0x000094, 0x000098, 0x00009c,
    0x0000a0, 0x0000a4, 0x0000a8, 0x0000ac, 0x0000b0, 0x0000b4, 0x0000b8, 0x0000bc,
    0x0000c0, 0x0000c4, 0x0000c8, 0x0000cc, 0x0000d0, 0x0000d4, 0x0000d8, 0x0000dc,
    0x0000e0, 0x0000e4, 0x0000e8, 0x0000ec, 0x0000f0, 0x0000f4, 0x0000f8, 0x0000fc,
    0x0000ff, 0x0004ff, 0x0008ff, 0x000cff, 0x0010ff, 0x0014ff, 0x0018ff, 0x001cff,
    0x0020ff, 0x0024ff, 0x0028ff, 0x002cff, 0x0030ff, 0x0034ff, 0x0038ff, 0x003cff,
    0x0040ff, 0x0044ff, 0x0048ff, 0x004cff, 0x0050ff, 0x0054ff, 0x0058ff, 0x005cff,
    0x0060ff, 0x0064ff, 0x0068ff, 0x006cff, 0x0070ff, 0x0074ff, 0x0078ff, 0x007cff,
    0x0080ff, 0x0084ff, 0x0088ff, 0x008cff, 0x0090ff, 0x0094ff, 0x0098ff, 0x009cff,
    0x00a0ff, 0x00a4ff, 0x00a8ff, 0x00acff, 0x00b0ff, 0x00b4ff, 0x00b8ff, 0x00bcff,
    0x00c0ff, 0x00c4ff, 0x00c8ff, 0x00ccff, 0x00d0ff, 0x00d4ff, 0x00d8ff, 0x00dcff,
    0x00e0ff, 0x00e4ff, 0x00e8ff, 0x00ecff, 0x00f0ff, 0x00f4ff, 0x00f8ff, 0x00fcff,
    0x02fffe, 0x06fffa, 0x0afff6, 0x0efff2, 0x12ffee, 0x16ffea, 0x1affe6, 0x1effe2,
    0x22ffde, 0x26ffda, 0x2affd6, 0x2effd2, 0x32ffce, 0x36ffca, 0x3affc6, 0x3effc2,
    0x42ffbe, 0x46ffba, 0x4affb6, 0x4effb2, 0x52ffae, 0x56ffaa, 0x5affa6, 0x5effa2,
    0x62ff9e, 0x66ff9a, 0x6aff96, 0x6eff92, 0x72ff8e, 0x76ff8a, 0x7aff86, 0x7eff82,
    0x82ff7e, 0x86ff7a, 0x8aff76, 0x8eff72, 0x92ff6e, 0x96ff6a, 0x9aff66, 0x9eff62,
    0xa2ff5e, 0xa6ff5a, 0xaaff56, 0xaeff52, 0xb2ff4e, 0xb6ff4a, 0xbaff46, 0xbeff42,
    0xc2ff3e, 0xc6ff3a, 0xcaff36, 0xceff32, 0xd2ff2e, 0xd6ff2a, 0xdaff26, 0xdeff22,
    0xe2ff1e, 0xe6ff1a, 0xeaff16, 0xeeff12, 0xf2ff0e, 0xf6ff0a, 0xfaff06, 0xfeff01,
    0xfffc00, 0xfff800, 0xfff400, 0xfff000, 0xffec00, 0xffe800, 0xffe400, 0xffe000,
    0xffdc00, 0xffd800, 0xffd400, 0xffd000, 0xffcc00, 0xffc800, 0xffc400, 0xffc000,
    0xffbc00, 0xffb800, 0xffb400, 0xffb000, 0xffac00, 0xffa800, 0xffa400, 0xffa000,
    0xff9c00, 0xff9800, 0xff9400, 0xff9000, 0xff8c00, 0xff8800, 0xff8400, 0xff8000,
    0xff7c00, 0xff7800, 0xff7400, 0xff7000, 0xff6c00, 0xff6800, 0xff6400, 0xff6000,
    0xff5c00, 0xff5800, 0xff5400, 0xff5000, 0xff4c00, 0xff4800, 0xff4400, 0xff4000,
    0xff3c00, 0xff3800, 0xff3400, 0xff3000, 0xff2c00, 0xff2800, 0xff2400, 0xff2000,
    0xff1c00, 0xff1800, 0xff1400, 0xff1000, 0xff0c00, 0xff0800, 0xff0400, 0xff0000,
    0xfc0000, 0xf80000, 0xf40000, 0xf00000, 0xec0000, 0xe80000, 0xe40000, 0xe00000,
    0xdc0000, 0xd80000, 0xd40000, 0xd00000, 0xcc0000, 0xc80000, 0xc40000, 0xc00000,
    0xbc0000, 0xb80000, 0xb40000, 0xb00000, 0xac0000, 0xa80000, 0xa40000, 0xa00000,
    0x9c0000, 0x980000, 0x940000, 0x900000, 0x8c0000, 0x880000, 0x840000, 0x800000
};

size_t table_bytes(int n) { return align_up(sizeof(OverlayImage) * (size_t)(n + 1), 256); }
int64_t pixels_of(const attwarp_overlay_image& im) { return (int64_t)im.H * im.W; }
int mm_ctas(const attwarp_overlay_image& im, int kind) {
    return kind == ATTWARP_OVERLAY_TOKENS ? 1 : (int)((pixels_of(im) + kMMChunk - 1) / kMMChunk);
}
int blend_ctas(const attwarp_overlay_image& im) { return (int)((pixels_of(im) + kBlendPix - 1) / kBlendPix); }

// NaN-propagating min / max (NumPy's np.min / np.max): once a NaN is in, it stays
template <typename T>
__device__ __forceinline__ T nan_min(T a, T b) { return (b < a || b != b) ? b : a; }
template <typename T>
__device__ __forceinline__ T nan_max(T a, T b) { return (b > a || b != b) ? b : a; }

// the image whose [begin, next begin) range holds `unit` (last entry with begin <= unit)
template <bool kMM>
__device__ __forceinline__ int find_image(const OverlayImage* imgs, int n, int unit) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((kMM ? imgs[mid].mm_begin : imgs[mid].blk_begin) <= unit) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// (lo, hi) of the block's threads -> part (thread 0 writes)
__device__ __forceinline__ void block_minmax_store(double lo, double hi, double2* part) {
    __shared__ double s_lo[kMMThreads / 32], s_hi[kMMThreads / 32];
    for (int o = 16; o > 0; o >>= 1) {
        lo = nan_min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = nan_max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_lo[warp] = lo; s_hi[warp] = hi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kMMThreads / 32; ++w) { lo = nan_min(lo, s_lo[w]); hi = nan_max(hi, s_hi[w]); }
        *part = make_double2(lo, hi);
    }
}

// ---- launch 1 -----------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kMMThreads) overlay_minmax_kernel(const OverlayImage* __restrict__ imgs, int n,
                                                                   double2* __restrict__ part) {
    const int unit = blockIdx.x;
    const OverlayImage im = imgs[find_image<true>(imgs, n, unit)];
    const int64_t N = (int64_t)im.H * im.W;
    const int64_t e0 = (int64_t)(unit - im.mm_begin) * kMMChunk;
    const int64_t e1 = min(N, e0 + (int64_t)kMMChunk);
    const T* a = static_cast<const T*>(im.att);
    using Acc = typename std::conditional<sizeof(T) == 1, int, T>::type;   // uint8: integer min / max
    Acc lo = sizeof(T) == 1 ? (Acc)255 : (Acc)INFINITY, hi = sizeof(T) == 1 ? (Acc)0 : (Acc)-INFINITY;
    int64_t e = e0 + threadIdx.x;
    if ((reinterpret_cast<uintptr_t>(a) & 15) == 0) {      // e0 is a multiple of 16: whole 16-byte vectors
        constexpr int V = 16 / sizeof(T);
        const int64_t nv = (e1 - e0) / V;
        const uint4* av = reinterpret_cast<const uint4*>(a + e0);
        for (int64_t k = threadIdx.x; k < nv; k += kMMThreads) {
            const uint4 u = __ldg(av + k);
            const T* v = reinterpret_cast<const T*>(&u);
#pragma unroll
            for (int j = 0; j < V; ++j) { lo = nan_min(lo, (Acc)v[j]); hi = nan_max(hi, (Acc)v[j]); }
        }
        e = e0 + nv * V + threadIdx.x;
    }
    for (; e < e1; e += kMMThreads) {
        const Acc v = (Acc)a[e];
        lo = nan_min(lo, v);
        hi = nan_max(hi, v);
    }
    block_minmax_store((double)lo, (double)hi, part + unit);
}

// token mode: row ty of the token map is reached iff some y in [0, H) has (y * gh) / H == ty: the least y with
// y * gh >= ty * H is below H and still maps to ty (likewise for columns)
__device__ __forceinline__ bool token_reached(uint32_t t, uint32_t g, uint32_t S) {
    const uint32_t y0 = (t * S + g - 1) / g;
    return y0 < S && y0 * g < (t + 1) * S;
}

__global__ void __launch_bounds__(kMMThreads) overlay_minmax_tokens_kernel(const OverlayImage* __restrict__ imgs,
                                                                          int gh, int gw, double2* __restrict__ part) {
    const OverlayImage im = imgs[blockIdx.x];
    const float* tok = static_cast<const float*>(im.att);
    double lo = INFINITY, hi = -INFINITY;
    for (int k = threadIdx.x; k < gh * gw; k += kMMThreads) {
        const int ty = k / gw, tx = k - ty * gw;
        if (token_reached(ty, gh, im.H) && token_reached(tx, gw, im.W)) {
            const double v = (double)tok[k];
            lo = nan_min(lo, v);
            hi = nan_max(hi, v);
        }
    }
    block_minmax_store(lo, hi, part + blockIdx.x);
}

// ---- launch 2 -----------------------------------------------------------------------------------------------------
// per-CTA state: the JET table, the image, its (lo, hi) and, for uint8 maps, the value -> heat index table
struct BlendShared {
    uint32_t jet[256];
    uint8_t lut[256];
    double lo, hi;
    int img;
};

__device__ __forceinline__ int trunc_index(float x) { return min(max(__float2int_rz(x), 0), 255); }
__device__ __forceinline__ int trunc_index(double x) { return min(max(__double2int_rz(x), 0), 255); }

// heat index of one attention value
template <typename T>
struct HeatIndex;

template <>
struct HeatIndex<uint8_t> {                    // uint8: a table over the 256 values, built once per CTA
    const uint8_t* lut;
    __device__ void init(BlendShared& s) {
        const uint8_t lo = (uint8_t)s.lo, hi = (uint8_t)s.hi;
        const int v = threadIdx.x;             // kBlendThreads == 256
        int idx = 0;
        // hi > lo + 1e-9 in float64; (a - lo) in uint8, the division and the scale in float64
        if (hi > __dadd_rn((double)lo, 1e-9) && v >= lo && v <= hi)
            idx = trunc_index(__dmul_rn(__ddiv_rn((double)(uint8_t)(v - lo), (double)(uint8_t)(hi - lo)), 255.0));
        s.lut[v] = (uint8_t)idx;
        lut = s.lut;
    }
    __device__ __forceinline__ int operator()(uint8_t v) const { return lut[v]; }
};

template <>
struct HeatIndex<float> {                      // float32 throughout; lo + 1e-9 rounds to float32 first
    float lo, range;
    bool zero;
    __device__ void init(const BlendShared& s) {
        lo = (float)s.lo;
        const float hi = (float)s.hi;
        zero = !(hi > __fadd_rn(lo, 1e-9f));
        range = __fsub_rn(hi, lo);
    }
    __device__ __forceinline__ int operator()(float v) const {
        return zero ? 0 : trunc_index(__fmul_rn(__fdiv_rn(__fsub_rn(v, lo), range), 255.0f));
    }
};

template <>
struct HeatIndex<double> {
    double lo, range;
    bool zero;
    __device__ void init(const BlendShared& s) {
        lo = s.lo;
        zero = !(s.hi > __dadd_rn(lo, 1e-9));
        range = __dsub_rn(s.hi, lo);
    }
    __device__ __forceinline__ int operator()(double v) const {
        return zero ? 0 : trunc_index(__dmul_rn(__ddiv_rn(__dsub_rn(v, lo), range), 255.0));
    }
};

// cv2.addWeighted(heat, alpha, base, 1 - alpha, 0) on one byte
__device__ __forceinline__ uint32_t blend_byte(uint32_t heat, uint32_t base, float a32, float b32) {
    const float v = __fmaf_rn((float)heat, a32, __fmul_rn((float)base, b32));
    return (uint32_t)min(max(__float2int_rn(v), 0), 255);
}

// the three output bytes (B | G << 8 | R << 16) of one pixel
__device__ __forceinline__ uint32_t blend_pixel(uint32_t heat, uint32_t b, uint32_t g, uint32_t r, float a32,
                                                float b32) {
    return blend_byte(heat & 255, b, a32, b32) | blend_byte((heat >> 8) & 255, g, a32, b32) << 8 |
           blend_byte(heat >> 16, r, a32, b32) << 16;
}

// CTA prologue: JET to shared memory, the image, its partials reduced (warp 0)
__device__ __forceinline__ void blend_prologue(const OverlayImage* imgs, int n, const double2* part, int img,
                                               BlendShared& s) {
    s.jet[threadIdx.x] = kJet[threadIdx.x];
    if (threadIdx.x < 32) {
        const int p0 = imgs[img].mm_begin, p1 = imgs[img + 1].mm_begin;
        double lo = INFINITY, hi = -INFINITY;
        for (int k = p0 + (int)threadIdx.x; k < p1; k += 32) {
            const double2 v = part[k];
            lo = nan_min(lo, v.x);
            hi = nan_max(hi, v.y);
        }
        for (int o = 16; o > 0; o >>= 1) {
            lo = nan_min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = nan_max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (threadIdx.x == 0) { s.lo = lo; s.hi = hi; }
    }
    __syncthreads();
}

// attention of pixel p: the map's own value, or the token its index upsampling picks
template <typename T, bool kTok>
struct AttSource {
    const T* a;
    uint32_t H, W, gh, gw;
    __device__ __forceinline__ T at(int64_t p) const {
        if constexpr (kTok) {
            const uint32_t y = (uint32_t)(p / W), x = (uint32_t)(p - (int64_t)y * W);
            return a[(y * gh / H) * gw + x * gw / W];
        } else {
            return a[p];
        }
    }
    // four consecutive pixels p..p+3 (p a multiple of 4; the map's base aligned for the vector path)
    __device__ __forceinline__ void at4(int64_t p, T (&v)[4]) const {
        if constexpr (kTok) {
            uint32_t y = (uint32_t)(p / W), x = (uint32_t)(p - (int64_t)y * W);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                v[j] = a[(y * gh / H) * gw + x * gw / W];
                if (++x == W) { x = 0; ++y; }
            }
        } else if constexpr (sizeof(T) == 1) {
            const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(a + p));
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = (T)(u >> (8 * j));
        } else if constexpr (sizeof(T) == 4) {
            const float4 f = __ldg(reinterpret_cast<const float4*>(a + p));
            v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
        } else {
            const double2 d0 = __ldg(reinterpret_cast<const double2*>(a + p));
            const double2 d1 = __ldg(reinterpret_cast<const double2*>(a + p) + 1);
            v[0] = d0.x; v[1] = d0.y; v[2] = d1.x; v[3] = d1.y;
        }
    }
};

template <typename T, bool kTok, bool kVec>
__device__ __forceinline__ void blend_body(const OverlayImage* __restrict__ imgs, int n,
                                           const double2* __restrict__ part, int gh, int gw, float a32, float b32) {
    __shared__ BlendShared s;
    if (threadIdx.x == 0) s.img = find_image<false>(imgs, n, blockIdx.x);
    __syncthreads();
    const int img = s.img;
    blend_prologue(imgs, n, part, img, s);
    const OverlayImage im = imgs[img];
    HeatIndex<T> hidx;
    hidx.init(s);
    if constexpr (sizeof(T) == 1 && !kTok) __syncthreads();     // the uint8 table is complete
    const AttSource<T, kTok> att{static_cast<const T*>(im.att), (uint32_t)im.H, (uint32_t)im.W, (uint32_t)gh,
                                 (uint32_t)gw};
    const int64_t N = (int64_t)im.H * im.W;
    const int64_t q0 = (int64_t)(blockIdx.x - im.blk_begin) * kBlendPix;
    const int64_t q1 = min(N, q0 + (int64_t)kBlendPix);
    const uint8_t* __restrict__ src = im.src;
    uint8_t* __restrict__ dst = im.dst;
    const bool grey = im.C == 1;

    auto one = [&](int64_t p) {                // one pixel, byte accesses
        uint32_t b, g, r;
        if (grey) {
            b = g = r = src[p];
        } else {
            b = src[3 * p]; g = src[3 * p + 1]; r = src[3 * p + 2];
        }
        const uint32_t o = blend_pixel(s.jet[hidx(att.at(p))], b, g, r, a32, b32);
        dst[3 * p] = (uint8_t)o;
        dst[3 * p + 1] = (uint8_t)(o >> 8);
        dst[3 * p + 2] = (uint8_t)(o >> 16);
    };

    if constexpr (kVec) {
        for (int64_t p = q0 + 4 * (int64_t)threadIdx.x; p < q1; p += 4 * kBlendThreads) {
            if (p + 4 > q1) {                  // the image's last pixels
                for (int64_t k = p; k < q1; ++k) one(k);
                continue;
            }
            T v[4];
            att.at4(p, v);
            uint32_t px[4];                    // B | G << 8 | R << 16
            if (grey) {
                const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(src + p));
#pragma unroll
                for (int j = 0; j < 4; ++j) px[j] = ((u >> (8 * j)) & 255) * 0x010101u;
            } else {
                const uint32_t* s32 = reinterpret_cast<const uint32_t*>(src + 3 * p);
                const uint32_t u0 = __ldg(s32), u1 = __ldg(s32 + 1), u2 = __ldg(s32 + 2);
                px[0] = u0 & 0xffffff;
                px[1] = (u0 >> 24) | (u1 & 0xffff) << 8;
                px[2] = (u1 >> 16) | (u2 & 0xff) << 16;
                px[3] = u2 >> 8;
            }
            uint32_t o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                o[j] = blend_pixel(s.jet[hidx(v[j])], px[j] & 255, (px[j] >> 8) & 255, px[j] >> 16, a32, b32);
            uint32_t* d32 = reinterpret_cast<uint32_t*>(dst + 3 * p);
            d32[0] = o[0] | o[1] << 24;
            d32[1] = o[1] >> 8 | o[2] << 16;
            d32[2] = o[2] >> 16 | o[3] << 8;
        }
    } else {
        for (int64_t p = q0 + threadIdx.x; p < q1; p += kBlendThreads) one(p);
    }
}

template <typename T, bool kVec>
__global__ void __launch_bounds__(kBlendThreads) overlay_blend_kernel(const OverlayImage* __restrict__ imgs, int n,
                                                                     const double2* __restrict__ part, float a32,
                                                                     float b32) {
    blend_body<T, false, kVec>(imgs, n, part, 0, 0, a32, b32);
}

template <bool kVec>
__global__ void __launch_bounds__(kBlendThreads) overlay_blend_tokens_kernel(const OverlayImage* __restrict__ imgs,
                                                                            int n, const double2* __restrict__ part,
                                                                            int gh, int gw, float a32, float b32) {
    blend_body<float, true, kVec>(imgs, n, part, gh, gw, a32, b32);
}

bool aligned(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

template <typename T>
int launch_map(const OverlayImage* d_table, int n, double2* d_part, int mm_total, int blk_total, bool vec, float a32,
               float b32, cudaStream_t st) {
    overlay_minmax_kernel<T><<<mm_total, kMMThreads, 0, st>>>(d_table, n, d_part);
    int rc = check_launch("overlay_minmax_kernel");
    if (rc != ATTWARP_OK) return rc;
    if (vec)
        overlay_blend_kernel<T, true><<<blk_total, kBlendThreads, 0, st>>>(d_table, n, d_part, a32, b32);
    else
        overlay_blend_kernel<T, false><<<blk_total, kBlendThreads, 0, st>>>(d_table, n, d_part, a32, b32);
    return check_launch("overlay_blend_kernel");
}

}  // namespace

size_t overlay_workspace_bytes_impl(const attwarp_overlay_image* images, int n, int att_kind) {
    size_t parts = 0;
    for (int i = 0; i < n; ++i) parts += (size_t)mm_ctas(images[i], att_kind);
    return table_bytes(n) + align_up(sizeof(double2) * parts, 256);
}

// arguments validated by the caller; ws of overlay_workspace_bytes_impl(images, n, att_kind) bytes
int launch_attention_overlay(const attwarp_overlay_image* images, int n, int att_dtype, int att_kind, int gh, int gw,
                             double alpha, void* ws, cudaStream_t st) {
    static thread_local std::vector<OverlayImage> host;
    host.assign((size_t)n + 1, OverlayImage{});
    int64_t mm = 0, blk = 0;
    // the 4-pixel path needs 4-byte aligned image and output bases and, for a map, 4 (uint8) or 16 (float) bytes
    bool vec = true;
    const uintptr_t att_align = att_dtype == ATTWARP_U8 ? 4 : 16;
    for (int i = 0; i < n; ++i) {
        const attwarp_overlay_image& in = images[i];
        OverlayImage& r = host[(size_t)i];
        r.src = static_cast<const uint8_t*>(in.src);
        r.att = in.att;
        r.dst = static_cast<uint8_t*>(in.dst);
        r.H = in.H;
        r.W = in.W;
        r.C = in.C;
        r.mm_begin = (int32_t)mm;
        r.blk_begin = (int32_t)blk;
        mm += mm_ctas(in, att_kind);
        blk += blend_ctas(in);
        vec = vec && aligned(in.src, 4) && aligned(in.dst, 4) &&
              (att_kind == ATTWARP_OVERLAY_TOKENS || aligned(in.att, att_align));
    }
    if (blk > INT32_MAX) return fail(ATTWARP_ERR_UNSUPPORTED, "attention_overlay: %lld CTAs in one call", (long long)blk);
    host[(size_t)n].mm_begin = (int32_t)mm;
    host[(size_t)n].blk_begin = (int32_t)blk;
    char* p = static_cast<char*>(ws);
    OverlayImage* d_table = reinterpret_cast<OverlayImage*>(p);
    double2* d_part = reinterpret_cast<double2*>(p + table_bytes(n));
    AW_CUDA(cudaMemcpyAsync(d_table, host.data(), sizeof(OverlayImage) * (size_t)(n + 1), cudaMemcpyHostToDevice, st));
    // addWeighted's weights: alpha and 1 - alpha (in double), each rounded to float32
    const float a32 = (float)alpha, b32 = (float)(1.0 - alpha);
    if (att_kind == ATTWARP_OVERLAY_TOKENS) {
        overlay_minmax_tokens_kernel<<<n, kMMThreads, 0, st>>>(d_table, gh, gw, d_part);
        int rc = check_launch("overlay_minmax_tokens_kernel");
        if (rc != ATTWARP_OK) return rc;
        if (vec)
            overlay_blend_tokens_kernel<true><<<(unsigned)blk, kBlendThreads, 0, st>>>(d_table, n, d_part, gh, gw, a32, b32);
        else
            overlay_blend_tokens_kernel<false><<<(unsigned)blk, kBlendThreads, 0, st>>>(d_table, n, d_part, gh, gw, a32, b32);
        return check_launch("overlay_blend_tokens_kernel");
    }
    switch (att_dtype) {
        case ATTWARP_U8: return launch_map<uint8_t>(d_table, n, d_part, (int)mm, (int)blk, vec, a32, b32, st);
        case ATTWARP_F32: return launch_map<float>(d_table, n, d_part, (int)mm, (int)blk, vec, a32, b32, st);
        case ATTWARP_F64: return launch_map<double>(d_table, n, d_part, (int)mm, (int)blk, vec, a32, b32, st);
        default: return fail(ATTWARP_ERR_INVALID_ARG, "attention_overlay: bad attention dtype %d", att_dtype);
    }
}

}  // namespace aw
