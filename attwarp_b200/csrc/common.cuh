// common.cuh -- error plumbing and block-level primitives shared by the kernels.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/attwarp.h"
#include "warp_math.h"

namespace aw {

// ---- error state (thread-local; surfaced through attwarp_last_error) -------------------------
void set_error(const char* fmt, ...);
int fail(int status, const char* fmt, ...);
int check_launch(const char* what);  // cudaGetLastError -> ATTWARP_ERR_CUDA

#define AW_REQUIRE(cond, ...)                                             \
    do {                                                                  \
        if (!(cond)) return ::aw::fail(ATTWARP_ERR_INVALID_ARG, __VA_ARGS__); \
    } while (0)

#define AW_CUDA(call)                                                                  \
    do {                                                                               \
        cudaError_t e__ = (call);                                                      \
        if (e__ != cudaSuccess)                                                        \
            return ::aw::fail(ATTWARP_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__)); \
    } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
int sm_count();
int sm_share();          // attwarp_set_sm_share: 1 = a launch may fill the SMs, 2 = half of each SM, ...

// ---- one image of a ragged batch (device table built by the launchers in remap_stream.cu / api.cu) ----
struct RaggedImage {
    const uint8_t* src;      // HWC uint8, dense
    uint8_t* dst;            // Ho x Wo x C, dense
    const float* map_x;      // Wo floats
    const float* map_y;      // Ho floats
    int H, W, Ho, Wo;
    // stage-5 plan (filled in by the stage-5 launcher): strips, row tiles, and the image's position in
    // the batch-wide cost axis that CTAs split evenly (a tile weighs tile_units units ~ its consumer warps)
    int strips_units;        // n_strips | tile_units << 16
    int strip_cols, n_rowtiles;
    int unit_begin;          // first cost unit of the image; its tiles are strip-major
};
static_assert(sizeof(RaggedImage) == 64, "descriptor layout");

// ---- the attention map of one image of a ragged batch (attwarp_warp_ragged_from_attention), kept beside its
// RaggedImage (same index) so that the stage-5 descriptor keeps its size.  Geometry: ragged_att_geometry.
struct RaggedAtt {
    const void* att;         // [H][W] map, dense rows, any base alignment (element-aligned for float maps)
    int64_t colpart;         // offset (in doubles) of the image's [n_chunks][W] column partials
    int64_t rowpart;         // offset of its [n_tiles][H] row partials
    int H, W;
    int chunk_rows, n_chunks;
    int tile_cols, n_tiles;
};
static_assert(sizeof(RaggedAtt) == 48, "descriptor layout");
// chunk / tile geometry of one map of a ragged batch: a function of (H, W) only
void ragged_att_geometry(int H, int W, int* chunk_rows, int* n_chunks, int* tile_cols, int* n_tiles);
// host_att[0..n): geometry and partial offsets filled in; uploads them with the work items to dev_att / dev_items,
// then launches the marginals kernel over all maps and the finish kernel that writes imgs[i].map_x / map_y
int launch_maps_from_attention_ragged(const RaggedAtt* host_att, int n, int att_dtype, const RaggedImage* dev_imgs,
                                      RaggedAtt* dev_att, int2* dev_items, int64_t n_items, double* partials,
                                      int max_h, int max_w, const attwarp_transform_params& tp, cudaStream_t st);
// the two launches of that call apart, for attwarp_warp_ragged_from_mask: the uint8 identity marginals over the items
// dev_items[0..n_items) (descriptors already on the device), and the finish over all n images
int launch_marginals_ragged_u8_identity(const int2* dev_items, int64_t n_items, const RaggedAtt* dev_att,
                                        double* partials, cudaStream_t st);
int launch_maps_from_partials_ragged(int n, const RaggedImage* dev_imgs, const RaggedAtt* dev_att, const double* partials,
                                     int max_h, int max_w, const attwarp_transform_params& tp, cudaStream_t st);

// ---- the LANCZOS coefficients of one mask of a ragged list (attwarp_warp_ragged_from_mask), beside its RaggedAtt
// (whose chunk_rows / n_chunks / tile_cols / n_tiles hold the fused kernel's rows per tile, row tiles, columns per CTA
// and column CTAs).  Device pointers into the coefficient tables mask.cu keeps per size.
struct RaggedLanczos {
    const int2* bx;          // horizontal pass: first tap per output column
    const int* kx;           //                  [W][ksx] 22-bit weights
    const int2* by;          // vertical pass: window per output row
    const uint8_t* planes;   //                [row tile][3][rows][16] coefficient byte planes
    int ksx, warps;          // taps per column; 64-column strips per CTA
};
static_assert(sizeof(RaggedLanczos) == 40, "descriptor layout");
// Geometry of the tensor-core marginals kernel for an h x w mask resized to H x W, as a call on that image alone takes
// it (false: that call would not run this kernel); pure host arithmetic
bool lanczos_ragged_geometry(int h, int w, int H, int W, int* rows, int* n_tiles, int* x_ctas, int* warps, size_t* smem);
// the coefficient tables of (h, w) -> (H, W) at `rows` rows per tile (built and uploaded once per size and device)
int lanczos_ragged_tables(int h, int w, int H, int W, int rows, RaggedLanczos* l);
// one launch over the items (image, row tile << 8 | column CTA); the descriptors are on the device
int launch_lanczos_marginals_ragged(const int2* dev_items, int64_t n_items, const RaggedAtt* dev_att,
                                    const RaggedLanczos* dev_lz, int w, size_t smem, double* partials, cudaStream_t st);

// ---- internal launchers (defined in the .cu files, used by the fused drivers in api.cu) -------
int launch_aggregate_partial(const void* attn, int dtype, int B, int L, int Hh, int T,
                             int64_t sb, int64_t sl, int64_t sh, const int32_t* tok_start,
                             float eps, float* partial, int nsplit, cudaStream_t st);
int aggregate_nsplit(int B, int L, int Hh);
int launch_aggregate_finalize(const float* partial, int B, int nsplit, int T, float scale,
                              float* out, int accumulate, float out_scale, cudaStream_t st);
int launch_maps_from_tokens(const float* tok, int nsplit, float scale, float* tok_out, int B,
                            int gh, int gw, int H, int W, int Wo, int Ho,
                            const attwarp_transform_params& tp, float* map_x, float* map_y,
                            int* fallback_flags, cudaStream_t st);
int launch_maps_from_attention(const void* att, int att_dtype, int B, int H, int W, int Wo,
                               int Ho, const attwarp_transform_params& tp, void* ws,
                               size_t ws_bytes, float* map_x, float* map_y, int* fallback_flags,
                               cudaStream_t st);
int launch_remap(const void* src, void* dst, int dtype, int layout, int B, int C, int H, int W,
                 int Ho, int Wo, const float* map_x, const float* map_y, cudaStream_t st);
int launch_pdf_to_cdf(const float* px, const float* py, int B, int Nx, int Ny, float alpha, const float* Mx,
                      const float* My, int W, int H, float* Fx, float* Fy, cudaStream_t st);
int launch_maps_from_cdf(const float* Fx, const float* Fy, int B, int H, int W, int Wo, int Ho, float* map_x,
                         float* map_y, cudaStream_t st);
// ragged batches: `imgs` is a device table of n entries (dims + map pointers are read per image)
int launch_maps_from_tokens_ragged(const float* tok, int n, int gh, int gw, const RaggedImage* imgs,
                                   int max_h, int max_w, const attwarp_transform_params& tp,
                                   int* fallback_flags, cudaStream_t st);
// stage 5 over a ragged batch, in two steps so that the maps kernel can run in between: `prepare` fills in the
// strip plan of host_table[0..n] (n + 1 entries) and uploads it to dev_table; `run` launches the kernel
int launch_remap_u8_stream_ragged_prepare(RaggedImage* host_table, int n, int C, RaggedImage* dev_table, cudaStream_t st);
int launch_remap_u8_stream_ragged_run(const RaggedImage* host_table, int n, int C, const RaggedImage* dev_table, cudaStream_t st);

int launch_safe_softmax_mix(const float* logits, int B, int N, float eps, float alpha, float* out, cudaStream_t st);
int launch_safe_softmax_mix_backward(const float* logits, const float* grad_out, int B, int N, float eps, float alpha,
                                     float* grad_logits, cudaStream_t st);
// fused image-resolution PDF-L1 loss (pdf_loss.cu); workspace: 2 B doubles + a zeroed 32-bit counter
int launch_pdf_l1_loss(const float* px, const float* py, const float* gx, const float* gy, int B, int Nx, int Ny, int Ngx,
                       int Ngy, const float* Mx, const float* My, const float* Mgx, const float* Mgy, int W, int H,
                       void* workspace, float* loss, cudaStream_t st);
int launch_pdf_l1_loss_backward(const float* px, const float* py, const float* gx, const float* gy, int B, int Nx, int Ny,
                                int Ngx, int Ngy, const float* Mx, const float* My, const float* Mgx, const float* Mgy,
                                int W, int H, const float* upstream, float* dpx, float* dpy, cudaStream_t st);
// the same for 3-channel images through remap_quad.cu (four adjacent pixels per thread)
bool remap_quad_enabled();
int launch_remap_u8_quad(const void* src, void* dst, int n_img, int H, int W, int Ho, int Wo, const float* map_x,
                         const float* map_y, cudaStream_t st);
// float32 images through remap_f32_stream.cu (ATTWARP_ERR_UNSUPPORTED: shape not taken, use the rows kernel)
bool remap_f32_stream_enabled();
int launch_remap_f32_stream(const float* src, float* dst, int n_planes, int E, int H, int W, int Ho, int Wo,
                            const float* map_x, const float* map_y, int map_div, cudaStream_t st);
// ragged: images grouped into width classes (one launch each); dev_main holds n + 1 entries in batch order,
// dev_sorted n + kRaggedClasses entries grouped by class
constexpr int kRaggedClasses = 28;     // 14 width classes x {rows 4-byte aligned, any alignment}
struct RaggedQuadPlan {
    int count[kRaggedClasses], offset[kRaggedClasses], total_units[kRaggedClasses], max_strip[kRaggedClasses],
        mode[kRaggedClasses];
};
int launch_remap_u8_quad_ragged_prepare(RaggedImage* host_table, int n, RaggedImage* dev_main, RaggedImage* dev_sorted,
                                        RaggedQuadPlan* plan, cudaStream_t st);
int ragged_quad_launches(const RaggedQuadPlan& plan);      // stage-5 launches the plan needs (one per non-empty class)
int launch_remap_u8_quad_ragged_run(const RaggedQuadPlan& plan, const RaggedImage* dev_sorted, cudaStream_t st);

#if defined(__CUDACC__)
// ---- warp / block reductions -----------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Block-wide sum, result broadcast to every thread.  `red` is >= 32 elements of shared memory.
// Deterministic: fixed shuffle tree per warp, then warp partials added in warp order.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();  // protect `red` from a previous use
    if (lane == 0) red[wid] = v;
    __syncthreads();
    T tot = (T)0;
    for (int i = 0; i < nw; ++i) tot += red[i];
    return tot;
}
template <typename T>
__device__ __forceinline__ T block_max(T v, T* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        T other = __shfl_xor_sync(0xffffffffu, v, o);
        v = other > v ? other : v;
    }
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    T m = red[0];
    for (int i = 1; i < nw; ++i) m = red[i] > m ? red[i] : m;
    return m;
}

// In-place inclusive scan of a[0..n) (shared memory, double) by the whole block.
// Each thread scans a contiguous chunk sequentially, chunk totals are scanned through `red`
// (>= blockDim.x doubles) by thread order, then offsets are added.  Deterministic.
__device__ __forceinline__ void block_inclusive_scan(double* a, int n, double* red) {
    const int nt = blockDim.x, t = threadIdx.x;
    const int per = (n + nt - 1) / nt;
    const int beg = min(t * per, n), end = min(beg + per, n);
    double run = 0.0;
    for (int i = beg; i < end; ++i) {
        run += a[i];
        a[i] = run;
    }
    __syncthreads();
    red[t] = run;
    __syncthreads();
    // exclusive prefix of chunk totals: warp 0 walks the (<= 1024) totals, 32 at a time
    if (t < 32) {
        double carry = 0.0;
        for (int base = 0; base < nt; base += 32) {
            const int i = base + t;
            double v = i < nt ? red[i] : 0.0;
            double inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                double up = __shfl_up_sync(0xffffffffu, inc, o);
                if (t >= o) inc += up;
            }
            if (i < nt) red[i] = carry + inc - v;  // exclusive
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
    }
    __syncthreads();
    const double off = red[t];
    if (off != 0.0)
        for (int i = beg; i < end; ++i) a[i] += off;
    __syncthreads();
}

// ---- thread groups: a contiguous run of warps of a CTA that synchronises on its own named barrier ----
// (lets the x axis and the y axis of one image be processed concurrently by the two halves of a CTA)
struct Group {
    int tid;  // thread index inside the group
    int nt;   // threads in the group (multiple of 32)
    int bar;  // hardware barrier id (1..15; 0 is __syncthreads)
    __device__ __forceinline__ void sync() const {
        asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(nt) : "memory");
    }
};

// Group-wide sum, result broadcast to every thread of the group.  `red` holds >= nt/32 elements and
// is private to the group.  Deterministic (shuffle tree per warp, warp partials added in warp order).
template <typename T>
__device__ __forceinline__ T group_sum(const Group& g, T v, T* red) {
    const int lane = g.tid & 31, wid = g.tid >> 5, nw = g.nt >> 5;
    v = warp_sum(v);
    g.sync();  // protect `red` from a previous use
    if (lane == 0) red[wid] = v;
    g.sync();
    T tot = (T)0;
    for (int i = 0; i < nw; ++i) tot += red[i];
    return tot;
}

// In-place inclusive scan of a[0..n) (shared memory, double) by one group.  Each thread scans a
// contiguous chunk, every warp shuffle-scans its 32 chunk totals, warp totals are added in warp
// order.  `red` holds >= nt/32 doubles.  Deterministic.
__device__ __forceinline__ void group_inclusive_scan(const Group& g, double* a, int n, double* red) {
    const int lane = g.tid & 31, wid = g.tid >> 5;
    const int per = (n + g.nt - 1) / g.nt;
    const int beg = min(g.tid * per, n), end = min(beg + per, n);
    double run = 0.0;
    for (int i = beg; i < end; ++i) {
        run += a[i];
        a[i] = run;
    }
    double inc = run;                                   // inclusive scan of the chunk totals in the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
    }
    g.sync();                                           // protect `red` from a previous use
    if (lane == 31) red[wid] = inc;
    g.sync();
    double off = inc - run;                             // chunks before mine in my warp
    for (int w = 0; w < wid; ++w) off += red[w];        // warps before mine, in order
    if (off != 0.0)
        for (int i = beg; i < end; ++i) a[i] += off;
    g.sync();
}

// ---- loads ------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_stream_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
template <typename T>
__device__ __forceinline__ double load_as_double(const T* p);
template <>
__device__ __forceinline__ double load_as_double<uint8_t>(const uint8_t* p) { return (double)__ldg(p); }
template <>
__device__ __forceinline__ double load_as_double<float>(const float* p) { return (double)__ldg(p); }
template <>
__device__ __forceinline__ double load_as_double<double>(const double* p) { return __ldg(p); }
#endif  // __CUDACC__

}  // namespace aw
