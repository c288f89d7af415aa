// api.cu -- the C ABI declared in include/attwarp.h: argument validation, error state, fused
// batch drivers and the host-buffer convenience entry point.  No kernels live here.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <vector>

#include "common.cuh"
#include "jpeg_decode.h"
#include "png_inflate.h"

namespace aw {

// declared in the other translation units
size_t maps_workspace_bytes_impl(int B, int H, int W);
int launch_gt_marginals(const float* A, int B, int H, int W, void* ws, size_t ws_bytes, float* px,
                        float* py, cudaStream_t st);
int launch_maps_from_cdf(const float* Fx, const float* Fy, int B, int H, int W, int Wo, int Ho,
                         float* map_x, float* map_y, cudaStream_t st);
int launch_safe_softmax(const float* logits, int B, int N, float eps, float* out, cudaStream_t st);
int launch_mix_with_uniform(const float* p, int B, int N, float alpha, float* out, cudaStream_t st);
int launch_cdf_from_density(const float* p, int B, int N, float* F, cudaStream_t st);
int launch_upsample_right_inverse(const float* y, const float* M, int B, int L_out, int L_in,
                                  float* x, cudaStream_t st);
int launch_mix_with_uniform_backward(const float* g, int B, int N, float alpha, float* gp, cudaStream_t st);
int launch_safe_softmax_backward(const float* logits, const float* grad_out, int B, int N, float eps,
                                 float* grad_logits, cudaStream_t st);
int launch_upsample_right_inverse_backward(const float* gx, const float* M, int B, int L_out, int L_in, float* gy,
                                           cudaStream_t st);
int launch_adaptive_avg_pool2d(const float* A, const uint8_t* sqrt_mask, int B, int H, int W, int gh, int gw,
                               float* out, cudaStream_t st);
int launch_revise_mask(const float* tok, int B, int gh, int gw, int ksize, float coe, float* revised,
                       uint8_t* mask_u8, cudaStream_t st);
int launch_resize_lanczos_u8(const uint8_t* src, int B, int h, int w, int Ho, int Wo, uint8_t* dst, cudaStream_t st);
size_t maps_from_mask_workspace_bytes_impl(int B, int h, int w, int H, int W);
int launch_maps_from_mask(const uint8_t* mask, int B, int h, int w, int H, int W, int Wo, int Ho,
                          const attwarp_transform_params& tp, void* ws, size_t ws_bytes, float* map_x, float* map_y,
                          cudaStream_t st);
int launch_strictly_increasing(const float* F, int B, int N, float eps, float* out, cudaStream_t st);
size_t png_max_bytes_impl(int H, int W, int C);
size_t png_workspace_bytes_impl(const attwarp_png_image* images, int n);
int launch_encode_png(const attwarp_png_image* images, int n, void* ws, uint8_t* out, int64_t* offsets,
                      cudaStream_t st);
size_t jpeg_workspace_bytes_impl(const jpeg::Header* headers, int n);
int launch_decode_jpeg(const attwarp_jpeg_image* images, const jpeg::Header* headers, int n, void* ws,
                       int32_t* status, cudaStream_t st);
size_t png_decode_workspace_bytes_impl(const png::Header* hs, int n);
int launch_decode_png(const attwarp_png_file* files, const png::Header* hs, int n, void* ws, int32_t* status,
                      cudaStream_t st);
int launch_interp_linear_rows(const float* F, int B, int N, int L, float* out, cudaStream_t st);
size_t overlay_workspace_bytes_impl(const attwarp_overlay_image* images, int n, int att_kind);
int launch_attention_overlay(const attwarp_overlay_image* images, int n, int att_dtype, int att_kind, int gh, int gw,
                             double alpha, void* ws, cudaStream_t st);

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int fail(int status, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return status;
}

int check_launch(const char* what) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ATTWARP_ERR_CUDA, "%s launch failed: %s", what, cudaGetErrorString(e));
    return ATTWARP_OK;
}

// How much of an SM one launch of the two streaming kernels (stage 1, stage 5) may fill: 1 = all of it (lowest
// latency for a single stream), 2 = half, so that kernels of two independent batches on different streams are
// co-resident on every SM (stage 1 is HBM-bound, stage 5 issue-bound: together they use both).
static std::atomic<int> g_sm_share{1};
int sm_share() { return g_sm_share.load(std::memory_order_relaxed); }

int sm_count() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached = n;
        cached_dev = dev;
    }
    return cached;
}

static int check_transform(const attwarp_transform_params* tp) {
    AW_REQUIRE(tp != nullptr, "transform params must not be NULL");
    AW_REQUIRE(tp->transform >= ATTWARP_T_IDENTITY && tp->transform <= ATTWARP_T_LOG,
               "unknown transform id %d", tp->transform);
    return ATTWARP_OK;
}

// The calls that upload descriptor tables from this thread's host buffers refuse a stream that is being captured into
// a CUDA graph: a captured copy node would read those buffers at replay time, after later calls have rewritten them.
static int refuse_graph_capture(cudaStream_t st, const char* what) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    AW_CUDA(cudaStreamIsCapturing(st, &cap));
    if (cap != cudaStreamCaptureStatusNone)
        return fail(ATTWARP_ERR_UNSUPPORTED, "%s: cannot be captured into a CUDA graph (host-side descriptor tables)", what);
    return ATTWARP_OK;
}

// ---- per-thread device scratch for the host-buffer entry point --------------------------------
struct HostArena {
    cudaStream_t stream = nullptr;
    void* dev = nullptr;
    size_t cap = 0;
    void* pin = nullptr;            // pinned staging for the caller's pageable buffers (see warp_image_host_impl)
    size_t pin_cap = 0;
    int device = -1;
    // Device memory and the stream belong to `device`: they are released when the calling thread moves to
    // another device and when the thread exits (errors ignored: at process exit the runtime may be gone).
    void release() {
        if (device >= 0 && (dev != nullptr || stream != nullptr)) {
            int cur = -1;
            const bool switched = cudaGetDevice(&cur) == cudaSuccess && cur != device &&
                                  cudaSetDevice(device) == cudaSuccess;
            if (stream != nullptr) { cudaStreamSynchronize(stream); cudaStreamDestroy(stream); }
            if (dev != nullptr) cudaFree(dev);
            if (pin != nullptr) cudaFreeHost(pin);
            if (switched) cudaSetDevice(cur);
            (void)cudaGetLastError();
        }
        stream = nullptr;
        dev = nullptr;
        cap = 0;
        pin = nullptr;
        pin_cap = 0;
        device = -1;
    }
    // Pinned staging of at least `bytes` (after ensure(): the stream exists); false when the host cannot pin that
    // much -- the caller then copies from / to the pageable buffers directly.
    bool ensure_pinned(size_t bytes) {
        if (bytes <= pin_cap) return true;
        if (stream != nullptr) cudaStreamSynchronize(stream);
        if (pin != nullptr) cudaFreeHost(pin);
        pin = nullptr;
        pin_cap = 0;
        const size_t want = align_up(bytes + bytes / 4, 1 << 20);
        if (cudaHostAlloc(&pin, want, cudaHostAllocDefault) != cudaSuccess) {
            (void)cudaGetLastError();
            pin = nullptr;
            return false;
        }
        pin_cap = want;
        return true;
    }
    ~HostArena() { release(); }
    int ensure(size_t bytes) {
        int cur = 0;
        AW_CUDA(cudaGetDevice(&cur));
        if (stream == nullptr || cur != device) {
            release();
            AW_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
            device = cur;
        }
        if (bytes > cap) {
            AW_CUDA(cudaStreamSynchronize(stream));
            if (dev != nullptr) AW_CUDA(cudaFree(dev));
            dev = nullptr;
            cap = 0;
            const size_t want = align_up(bytes + bytes / 4, 1 << 20);
            AW_CUDA(cudaMalloc(&dev, want));
            cap = want;
        }
        return ATTWARP_OK;
    }
    // error path of a host call: nothing of this call may still be pending when the next one reuses the arena
    int drain(int rc) {
        if (stream != nullptr) cudaStreamSynchronize(stream);
        return rc;
    }
};
static thread_local HostArena g_arena;

static size_t dtype_size(int dt) {
    switch (dt) {
        case ATTWARP_U8: return 1;
        case ATTWARP_F32: return 4;
        case ATTWARP_F64: return 8;
        case ATTWARP_BF16:
        case ATTWARP_F16: return 2;
        default: return 0;
    }
}

}  // namespace aw

using namespace aw;

extern "C" {

int attwarp_abi_version(void) { return ATTWARP_ABI_VERSION; }

const char* attwarp_last_error(void) { return g_err; }

int attwarp_set_sm_share(int share) {
    if (share < 1) share = 1;
    if (share > 4) share = 4;
    return g_sm_share.exchange(share, std::memory_order_relaxed);
}

int attwarp_device_info(int* sm, int* cc_major, int* cc_minor) {
    int dev = 0;
    AW_CUDA(cudaGetDevice(&dev));
    int n = 0, maj = 0, min = 0;
    AW_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    AW_CUDA(cudaDeviceGetAttribute(&maj, cudaDevAttrComputeCapabilityMajor, dev));
    AW_CUDA(cudaDeviceGetAttribute(&min, cudaDevAttrComputeCapabilityMinor, dev));
    if (sm) *sm = n;
    if (cc_major) *cc_major = maj;
    if (cc_minor) *cc_minor = min;
    return ATTWARP_OK;
}

// ---------------------------------------------------------------------------------------------
size_t attwarp_aggregate_workspace_bytes(int B, int L, int Hh, int T) {
    if (B <= 0 || L <= 0 || Hh <= 0 || T <= 0) return 0;
    return sizeof(float) * (size_t)B * aggregate_nsplit(B, L, Hh) * T;
}

int attwarp_aggregate_attention(const void* attn, int dtype, int B, int L, int Hh, int T,
                                int64_t stride_b, int64_t stride_l, int64_t stride_h,
                                const int32_t* tok_start, float eps, void* workspace,
                                size_t workspace_bytes, float* out, int accumulate,
                                float out_scale, void* stream) {
    AW_REQUIRE(attn && out, "aggregate: NULL pointer");
    AW_REQUIRE(B > 0 && L > 0 && Hh > 0 && T > 0, "aggregate: sizes must be positive (B=%d L=%d Hh=%d T=%d)", B, L, Hh, T);
    AW_REQUIRE(B <= 65535, "aggregate: B=%d exceeds 65535", B);
    if (workspace == nullptr || workspace_bytes < attwarp_aggregate_workspace_bytes(B, L, Hh, T))
        return fail(ATTWARP_ERR_WORKSPACE, "aggregate: workspace too small (%zu < %zu)", workspace_bytes,
                    attwarp_aggregate_workspace_bytes(B, L, Hh, T));
    const int nsplit = aggregate_nsplit(B, L, Hh);
    cudaStream_t st = as_stream(stream);
    int rc = launch_aggregate_partial(attn, dtype, B, L, Hh, T, stride_b, stride_l, stride_h, tok_start,
                                      eps, static_cast<float*>(workspace), nsplit, st);
    if (rc != ATTWARP_OK) return rc;
    return launch_aggregate_finalize(static_cast<const float*>(workspace), B, nsplit, T,
                                     1.0f / ((float)L * (float)Hh), out, accumulate, out_scale, st);
}

// ---------------------------------------------------------------------------------------------
size_t attwarp_maps_workspace_bytes(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    return maps_workspace_bytes_impl(B, H, W);
}

int attwarp_maps_from_attention(const void* att, int att_dtype, int B, int H, int W, int Wo, int Ho,
                                const attwarp_transform_params* tp, void* workspace,
                                size_t workspace_bytes, float* map_x, float* map_y, void* stream) {
    AW_REQUIRE(att && map_x && map_y, "maps_from_attention: NULL pointer");
    AW_REQUIRE(B > 0 && H > 0 && W > 0 && Wo > 0 && Ho > 0, "maps_from_attention: sizes must be positive");
    AW_REQUIRE(B <= 65535, "maps_from_attention: B=%d exceeds 65535", B);
    int rc = check_transform(tp);
    if (rc != ATTWARP_OK) return rc;
    return launch_maps_from_attention(att, att_dtype, B, H, W, Wo, Ho, *tp, workspace, workspace_bytes,
                                      map_x, map_y, nullptr, as_stream(stream));
}

size_t attwarp_maps_from_mask_workspace_bytes(int B, int h, int w, int H, int W) {
    if (B <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return 0;
    return maps_from_mask_workspace_bytes_impl(B, h, w, H, W);
}

int attwarp_maps_from_mask(const void* mask_u8, int B, int h, int w, int H, int W, int Wo, int Ho,
                           const attwarp_transform_params* tp, void* workspace, size_t workspace_bytes,
                           float* map_x, float* map_y, void* stream) {
    AW_REQUIRE(mask_u8 && map_x && map_y, "maps_from_mask: NULL pointer");
    AW_REQUIRE(B > 0 && h > 0 && w > 0 && H > 0 && W > 0 && Wo > 0 && Ho > 0, "maps_from_mask: sizes must be positive");
    AW_REQUIRE(B <= 65535, "maps_from_mask: B=%d exceeds 65535", B);
    int rc = check_transform(tp);
    if (rc != ATTWARP_OK) return rc;
    return launch_maps_from_mask(static_cast<const uint8_t*>(mask_u8), B, h, w, H, W, Wo, Ho, *tp, workspace,
                                 workspace_bytes, map_x, map_y, as_stream(stream));
}

int attwarp_maps_from_tokens(const float* tok, int B, int gh, int gw, int H, int W, int Wo, int Ho,
                             const attwarp_transform_params* tp, float* map_x, float* map_y,
                             void* stream) {
    AW_REQUIRE(tok && map_x && map_y, "maps_from_tokens: NULL pointer");
    AW_REQUIRE(B > 0 && gh > 0 && gw > 0 && H > 0 && W > 0 && Wo > 0 && Ho > 0, "maps_from_tokens: sizes must be positive");
    AW_REQUIRE(gh <= H && gw <= W, "maps_from_tokens: token grid %dx%d larger than the image %dx%d", gh, gw, H, W);
    int rc = check_transform(tp);
    if (rc != ATTWARP_OK) return rc;
    return launch_maps_from_tokens(tok, 1, 1.0f, nullptr, B, gh, gw, H, W, Wo, Ho, *tp, map_x, map_y,
                                   nullptr, as_stream(stream));
}

int attwarp_maps_from_cdf(const float* Fx, const float* Fy, int B, int H, int W, int Wo, int Ho,
                          float* map_x, float* map_y, void* stream) {
    AW_REQUIRE(Fx && Fy && map_x && map_y, "maps_from_cdf: NULL pointer");
    AW_REQUIRE(B > 0 && H > 0 && W > 0 && Wo > 0 && Ho > 0, "maps_from_cdf: sizes must be positive");
    AW_REQUIRE(B <= 65535, "maps_from_cdf: B=%d exceeds 65535", B);
    return launch_maps_from_cdf(Fx, Fy, B, H, W, Wo, Ho, map_x, map_y, as_stream(stream));
}

// ---------------------------------------------------------------------------------------------
int attwarp_remap_bilinear(const void* src, void* dst, int dtype, int layout, int B, int C, int H,
                           int W, int Ho, int Wo, const float* map_x, const float* map_y,
                           void* stream) {
    AW_REQUIRE(src && dst && map_x && map_y, "remap: NULL pointer");
    AW_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && Ho > 0 && Wo > 0, "remap: sizes must be positive");
    AW_REQUIRE(layout == ATTWARP_LAYOUT_HWC || layout == ATTWARP_LAYOUT_CHW, "remap: bad layout %d", layout);
    AW_REQUIRE(src != dst, "remap: in-place operation is not supported");
    return launch_remap(src, dst, dtype, layout, B, C, H, W, Ho, Wo, map_x, map_y, as_stream(stream));
}

// ---------------------------------------------------------------------------------------------
int attwarp_warp_from_attention_tokens(const void* attn, int attn_dtype, int B, int L, int Hh,
                                       int64_t stride_b, int64_t stride_l, int64_t stride_h,
                                       const int32_t* tok_start, int gh, int gw, const void* src,
                                       void* dst, int img_dtype, int layout, int C, int H, int W,
                                       int Ho, int Wo, const attwarp_transform_params* tp,
                                       void* workspace, size_t workspace_bytes, float* tok_out,
                                       float* map_x, float* map_y, void* const* stage_events,
                                       void* stream) {
    AW_REQUIRE(attn && src && dst && tok_out && map_x && map_y, "warp_from_attention_tokens: NULL pointer");
    AW_REQUIRE(B > 0 && L > 0 && Hh > 0 && gh > 0 && gw > 0 && C > 0 && H > 0 && W > 0 && Ho > 0 && Wo > 0,
               "warp_from_attention_tokens: sizes must be positive");
    AW_REQUIRE(B <= 65535, "warp_from_attention_tokens: B=%d exceeds 65535", B);
    AW_REQUIRE(gh <= H && gw <= W, "token grid %dx%d larger than the image %dx%d", gh, gw, H, W);
    int rc = check_transform(tp);
    if (rc != ATTWARP_OK) return rc;
    const int T = gh * gw;
    if (workspace == nullptr || workspace_bytes < attwarp_aggregate_workspace_bytes(B, L, Hh, T))
        return fail(ATTWARP_ERR_WORKSPACE, "warp_from_attention_tokens: workspace too small");
    cudaStream_t st = as_stream(stream);
    const int nsplit = aggregate_nsplit(B, L, Hh);
    float* partial = static_cast<float*>(workspace);
    auto mark = [&](int i) -> int {
        if (stage_events == nullptr) return ATTWARP_OK;
        AW_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(stage_events[i]), st));
        return ATTWARP_OK;
    };
    if ((rc = mark(0)) != ATTWARP_OK) return rc;
    rc = launch_aggregate_partial(attn, attn_dtype, B, L, Hh, T, stride_b, stride_l, stride_h, tok_start,
                                  1e-12f, partial, nsplit, st);
    if (rc != ATTWARP_OK) return rc;
    if ((rc = mark(1)) != ATTWARP_OK) return rc;
    // stage-1 finalize is fused into the maps kernel (it sums the split partials in order)
    rc = launch_maps_from_tokens(partial, nsplit, 1.0f / ((float)L * (float)Hh), tok_out, B, gh, gw, H, W,
                                 Wo, Ho, *tp, map_x, map_y, nullptr, st);
    if (rc != ATTWARP_OK) return rc;
    if ((rc = mark(2)) != ATTWARP_OK) return rc;
    rc = launch_remap(src, dst, img_dtype, layout, B, C, H, W, Ho, Wo, map_x, map_y, st);
    if (rc != ATTWARP_OK) return rc;
    return mark(3);
}

// ---------------------------------------------------------------------------------------------
int attwarp_warp_from_pdfs(const float* px, const float* py, int B, int Nx, int Ny, float alpha,
                           const float* Mx, const float* My, const void* src, void* dst, int dtype,
                           int layout, int C, int H, int W, int Ho, int Wo, float* Fx, float* Fy,
                           float* map_x, float* map_y, void* stream) {
    AW_REQUIRE(px && py && Mx && My && src && dst && Fx && Fy && map_x && map_y, "warp_from_pdfs: NULL pointer");
    AW_REQUIRE(B > 0 && Nx > 0 && Ny > 0 && C > 0 && H > 0 && W > 0 && Ho > 0 && Wo > 0,
               "warp_from_pdfs: sizes must be positive");
    AW_REQUIRE(B <= 65535, "warp_from_pdfs: B=%d exceeds 65535", B);
    AW_REQUIRE(layout == ATTWARP_LAYOUT_HWC || layout == ATTWARP_LAYOUT_CHW, "warp_from_pdfs: bad layout %d", layout);
    AW_REQUIRE(src != dst, "warp_from_pdfs: in-place operation is not supported");
    cudaStream_t st = as_stream(stream);
    int rc = launch_pdf_to_cdf(px, py, B, Nx, Ny, alpha, Mx, My, W, H, Fx, Fy, st);
    if (rc != ATTWARP_OK) return rc;
    rc = launch_maps_from_cdf(Fx, Fy, B, H, W, Wo, Ho, map_x, map_y, st);
    if (rc != ATTWARP_OK) return rc;
    return launch_remap(src, dst, dtype, layout, B, C, H, W, Ho, Wo, map_x, map_y, st);
}

}  // extern "C" (the ragged helpers below include templates, which cannot have C linkage)

// ---------------------------------------------------------------------------------------------
// Ragged batches.  Every call's workspace starts with the descriptor tables (n + 1 entries in list order, then
// n + kRaggedClasses entries grouped by width class for the stage-5 launches) and the map rows of every image.
static size_t ragged_table_bytes(int n) { return align_up(sizeof(RaggedImage) * (size_t)(2 * n + 1 + kRaggedClasses), 256); }

// bytes of that shared prefix, 0 when an image has invalid sizes
static size_t ragged_prefix_bytes(const attwarp_ragged_image* images, int n) {
    size_t floats = 0;
    for (int i = 0; i < n; ++i) {
        const attwarp_ragged_image& im = images[i];
        if (im.H <= 0 || im.W <= 0 || im.Ho <= 0 || im.Wo <= 0 || im.H >= 65536 || im.W >= 65536) return 0;
        floats += (size_t)im.Wo + (size_t)im.Ho;
    }
    return ragged_table_bytes(n) + align_up(floats * sizeof(float), 256);
}

// kernel launches of this thread's last ragged call (maps + one resample launch per class)
static thread_local int g_ragged_last_launches = 0;

// A ragged call's list: the host descriptor table (n + 1 entries, the last one for the stage-5 plan), the device table
// at the start of the workspace, and what the maps kernels need to know of the whole list.
struct RaggedList {
    RaggedImage* host = nullptr;
    RaggedImage* dev = nullptr;
    int max_h = 0, max_w = 0;
    bool degenerate = false;     // an image with a 1-pixel axis: the call goes image by image
};

// Checks every image and fills the host table in one pass.  Each image's map rows are taken from the workspace pool
// in list order (the attention and mask calls may point them at the caller's buffers afterwards; the pool keeps its
// layout either way).
static int ragged_list(const char* what, const attwarp_ragged_image* images, int n, void* workspace, RaggedList* l) {
    static thread_local std::vector<RaggedImage> host;
    host.assign((size_t)n + 1, RaggedImage{});
    l->host = host.data();
    l->dev = static_cast<RaggedImage*>(workspace);
    float* pool = reinterpret_cast<float*>(static_cast<char*>(workspace) + ragged_table_bytes(n));
    size_t off = 0;
    for (int i = 0; i < n; ++i) {
        const attwarp_ragged_image& im = images[i];
        AW_REQUIRE(im.src && im.dst && im.src != im.dst, "%s: image %d: bad pointers", what, i);
        AW_REQUIRE(im.H > 0 && im.W > 0 && im.Ho > 0 && im.Wo > 0, "%s: image %d: sizes must be positive", what, i);
        AW_REQUIRE(im.H < 65536 && im.W < 65536, "%s: image %d: H, W must be below 65536", what, i);
        RaggedImage& r = host[(size_t)i];
        r.src = static_cast<const uint8_t*>(im.src);
        r.dst = static_cast<uint8_t*>(im.dst);
        r.map_x = pool + off; off += (size_t)im.Wo;
        r.map_y = pool + off; off += (size_t)im.Ho;
        r.H = im.H; r.W = im.W; r.Ho = im.Ho; r.Wo = im.Wo;
        l->max_h = im.H > l->max_h ? im.H : l->max_h;
        l->max_w = im.W > l->max_w ? im.W : l->max_w;
        l->degenerate = l->degenerate || im.H < 2 || im.W < 2;
    }
    return ATTWARP_OK;
}

// A list with a 1-pixel axis goes image by image through the uniform entry points (the streaming kernel needs two
// source rows and columns); such lists are not a throughput case.  maps(i, r) writes image i's maps.
template <class Maps>
static int ragged_per_image(const RaggedList& l, int n, int C, cudaStream_t st, int launches, Maps&& maps) {
    for (int i = 0; i < n; ++i) {
        const RaggedImage& r = l.host[i];
        int rc = maps(i, r);
        if (rc != ATTWARP_OK) return rc;
        rc = launch_remap(r.src, r.dst, ATTWARP_U8, ATTWARP_LAYOUT_HWC, 1, C, r.H, r.W, r.Ho, r.Wo, r.map_x, r.map_y, st);
        if (rc != ATTWARP_OK) return rc;
    }
    g_ragged_last_launches = launches;
    return ATTWARP_OK;
}

// The strip plan of stage 5 is part of the table both the maps and the resample kernels read: plan + upload, then
// maps() enqueues the `maps_launches` maps launches, then the resample.
template <class Maps>
static int ragged_stage5(const RaggedList& l, int n, int C, cudaStream_t st, int maps_launches, Maps&& maps) {
    const bool quad = C == 3 && remap_quad_enabled();
    RaggedQuadPlan plan;
    RaggedImage* dev_sorted = l.dev + (n + 1);
    int rc = quad ? launch_remap_u8_quad_ragged_prepare(l.host, n, l.dev, dev_sorted, &plan, st)
                  : launch_remap_u8_stream_ragged_prepare(l.host, n, C, l.dev, st);
    if (rc != ATTWARP_OK) return rc;
    if ((rc = maps()) != ATTWARP_OK) return rc;
    g_ragged_last_launches = maps_launches + (quad ? ragged_quad_launches(plan) : 1);
    return quad ? launch_remap_u8_quad_ragged_run(plan, dev_sorted, st)
                : launch_remap_u8_stream_ragged_run(l.host, n, C, l.dev, st);
}

extern "C" {

size_t attwarp_ragged_workspace_bytes(const attwarp_ragged_image* images, int n) {
    if (images == nullptr || n <= 0) return 0;
    return ragged_prefix_bytes(images, n);
}

int attwarp_warp_ragged_from_tokens(const float* tok, int n, int gh, int gw,
                                    const attwarp_ragged_image* images, int C,
                                    const attwarp_transform_params* tp, void* workspace,
                                    size_t workspace_bytes, void* stream) {
    AW_REQUIRE(tok && images && workspace, "warp_ragged: NULL pointer");
    AW_REQUIRE(n > 0 && gh > 0 && gw > 0, "warp_ragged: sizes must be positive");
    AW_REQUIRE(C == 1 || C == 3 || C == 4, "warp_ragged: C must be 1, 3 or 4 (got %d)", C);
    int rc = check_transform(tp);
    if (rc != ATTWARP_OK) return rc;
    RaggedList l;
    if ((rc = ragged_list("warp_ragged", images, n, workspace, &l)) != ATTWARP_OK) return rc;
    const size_t need = ragged_prefix_bytes(images, n);
    if (workspace_bytes < need)
        return fail(ATTWARP_ERR_WORKSPACE, "warp_ragged: workspace too small (%zu < %zu)", workspace_bytes, need);
    cudaStream_t st = as_stream(stream);
    if ((rc = refuse_graph_capture(st, "warp_ragged")) != ATTWARP_OK) return rc;
    if (l.degenerate)          // maps + resample per image
        return ragged_per_image(l, n, C, st, 2 * n, [&](int i, const RaggedImage& r) {
            return launch_maps_from_tokens(tok + (size_t)i * gh * gw, 1, 1.0f, nullptr, 1, gh, gw, r.H, r.W, r.Wo, r.Ho,
                                           *tp, const_cast<float*>(r.map_x), const_cast<float*>(r.map_y), nullptr, st);
        });
    return ragged_stage5(l, n, C, st, 1, [&] {
        return launch_maps_from_tokens_ragged(tok, n, gh, gw, l.dev, l.max_h, l.max_w, *tp, nullptr, st);
    });
}

int attwarp_ragged_last_launches(void) { return g_ragged_last_launches; }

// ---------------------------------------------------------------------------------------------
// Ragged batch warped by per-image maps.  Workspace: the shared prefix, then the maps' descriptors (RaggedAtt) followed
// by the work items, then the partials: every image's at its own offset (ragged geometry), or one image's of the
// uniform geometry when the call goes image by image.
struct RaggedAttLayout {
    int64_t items = 0;
    size_t att = 0, item_at = 0, partials = 0, part_bytes = 0, total = 0;     // byte offsets and sizes
};
static bool ragged_att_layout(const attwarp_ragged_image* images, int n, RaggedAttLayout* w) {
    const size_t prefix = ragged_prefix_bytes(images, n);
    if (prefix == 0) return false;
    size_t part_doubles = 0, uniform_bytes = 0;
    for (int i = 0; i < n; ++i) {
        const attwarp_ragged_image& im = images[i];
        int rows, nrc, tc, nct;
        ragged_att_geometry(im.H, im.W, &rows, &nrc, &tc, &nct);
        part_doubles += (size_t)nrc * im.W + (size_t)nct * im.H;
        w->items += (int64_t)nrc * nct;
        const size_t u = maps_workspace_bytes_impl(1, im.H, im.W);
        uniform_bytes = u > uniform_bytes ? u : uniform_bytes;
    }
    const size_t desc = align_up(sizeof(RaggedAtt) * (size_t)n, 16), part = part_doubles * sizeof(double);
    w->att = prefix;
    w->item_at = prefix + desc;
    w->partials = prefix + align_up(desc + sizeof(int2) * (size_t)w->items, 256);
    w->part_bytes = part > uniform_bytes ? part : uniform_bytes;
    w->total = w->partials + w->part_bytes;
    return true;
}

size_t attwarp_ragged_attention_workspace_bytes(const attwarp_ragged_image* images, int n) {
    RaggedAttLayout w;
    if (images == nullptr || n <= 0 || !ragged_att_layout(images, n, &w)) return 0;
    return w.total;
}

int attwarp_warp_ragged_from_attention(const attwarp_ragged_image* images, const attwarp_ragged_attention* att,
                                       int n, int att_dtype, int C, const attwarp_transform_params* tp,
                                       void* workspace, size_t workspace_bytes, void* stream) {
    const char* const what = "warp_ragged_from_attention";
    AW_REQUIRE(images && att && workspace, "%s: NULL pointer", what);
    AW_REQUIRE(n > 0, "%s: n must be positive (got %d)", what, n);
    AW_REQUIRE(C == 1 || C == 3 || C == 4, "%s: C must be 1, 3 or 4 (got %d)", what, C);
    AW_REQUIRE(att_dtype == ATTWARP_U8 || att_dtype == ATTWARP_F32 || att_dtype == ATTWARP_F64,
               "%s: attention dtype must be U8, F32 or F64 (got %d)", what, att_dtype);
    int rc = check_transform(tp);
    if (rc != ATTWARP_OK) return rc;
    RaggedList l;
    if ((rc = ragged_list(what, images, n, workspace, &l)) != ATTWARP_OK) return rc;
    const size_t es = dtype_size(att_dtype);
    static thread_local std::vector<RaggedAtt> host_att;
    host_att.assign((size_t)n, RaggedAtt{});
    int64_t part_off = 0;
    for (int i = 0; i < n; ++i) {
        AW_REQUIRE(att[i].att != nullptr, "%s: image %d: NULL attention map", what, i);
        AW_REQUIRE((reinterpret_cast<uintptr_t>(att[i].att) & (es - 1)) == 0,
                   "%s: image %d: attention map not aligned to its %zu-byte elements", what, i, es);
        RaggedImage& r = l.host[i];
        if (att[i].map_x != nullptr) r.map_x = att[i].map_x;
        if (att[i].map_y != nullptr) r.map_y = att[i].map_y;
        RaggedAtt& a = host_att[(size_t)i];
        a.att = att[i].att;
        a.H = r.H; a.W = r.W;
        ragged_att_geometry(r.H, r.W, &a.chunk_rows, &a.n_chunks, &a.tile_cols, &a.n_tiles);
        a.colpart = part_off; part_off += (int64_t)a.n_chunks * r.W;
        a.rowpart = part_off; part_off += (int64_t)a.n_tiles * r.H;
    }
    RaggedAttLayout w;
    ragged_att_layout(images, n, &w);
    if (workspace_bytes < w.total)
        return fail(ATTWARP_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", what, workspace_bytes, w.total);
    cudaStream_t st = as_stream(stream);
    if ((rc = refuse_graph_capture(st, what)) != ATTWARP_OK) return rc;
    char* ws = static_cast<char*>(workspace);
    double* partials = reinterpret_cast<double*>(ws + w.partials);
    if (l.degenerate)          // marginals + finish + resample per image
        return ragged_per_image(l, n, C, st, 3 * n, [&](int i, const RaggedImage& r) {
            return launch_maps_from_attention(att[i].att, att_dtype, 1, r.H, r.W, r.Wo, r.Ho, *tp, partials,
                                              w.part_bytes, const_cast<float*>(r.map_x), const_cast<float*>(r.map_y),
                                              nullptr, st);
        });
    return ragged_stage5(l, n, C, st, 2, [&] {
        return launch_maps_from_attention_ragged(host_att.data(), n, att_dtype, l.dev,
                                                 reinterpret_cast<RaggedAtt*>(ws + w.att),
                                                 reinterpret_cast<int2*>(ws + w.item_at), w.items, partials, l.max_h,
                                                 l.max_w, *tp, st);
    });
}

// ---------------------------------------------------------------------------------------------
// Ragged batch warped by each image's LANCZOS-resized mask.  Workspace: the shared prefix, then RaggedAtt [n],
// RaggedLanczos [n] and the work items (fused kernel's, then the uint8 marginals'), then the image-size masks of the
// images the fused kernel does not take, then the partials (every image's at its own offset, or one image's of the
// uniform entry points when the call goes image by image).
struct RaggedMaskLayout {
    int64_t fused_items = 0, att_items = 0;
    size_t smem = 0;                                       // the fused kernel's shared memory
    size_t tables = 0, lz = 0, item_at = 0, table_bytes = 0;   // the uploaded tables; lz, item_at: offsets into them
    size_t masks = 0, partials = 0, part_bytes = 0, total = 0;
};
static bool ragged_mask_layout(const attwarp_ragged_image* images, int n, int gh, int gw, RaggedMaskLayout* w) {
    const size_t prefix = ragged_prefix_bytes(images, n);
    if (prefix == 0) return false;
    size_t part_doubles = 0, mask_bytes = 0, uniform_bytes = 0;
    for (int i = 0; i < n; ++i) {
        const attwarp_ragged_image& im = images[i];
        int rows, nt, nx, warps;
        size_t smem, part;
        if (lanczos_ragged_geometry(gh, gw, im.H, im.W, &rows, &nt, &nx, &warps, &smem)) {
            part = (size_t)nt * im.W + (size_t)nx * im.H;
            w->fused_items += (int64_t)nt * nx;
            w->smem = smem > w->smem ? smem : w->smem;
        } else {
            int nrc, tc, nct;
            ragged_att_geometry(im.H, im.W, &rows, &nrc, &tc, &nct);
            part = (size_t)nrc * im.W + (size_t)nct * im.H;
            w->att_items += (int64_t)nrc * nct;
            mask_bytes += align_up((size_t)im.H * im.W, 16);
            const size_t u = maps_workspace_bytes_impl(1, im.H, im.W);
            uniform_bytes = u > uniform_bytes ? u : uniform_bytes;
        }
        part_doubles += part;
        uniform_bytes = part * sizeof(double) > uniform_bytes ? part * sizeof(double) : uniform_bytes;
    }
    w->tables = prefix;
    w->lz = align_up(sizeof(RaggedAtt) * (size_t)n, 16);
    w->item_at = w->lz + sizeof(RaggedLanczos) * (size_t)n;
    w->table_bytes = w->item_at + sizeof(int2) * (size_t)(w->fused_items + w->att_items);
    w->masks = w->tables + align_up(w->table_bytes, 256);
    w->partials = w->masks + align_up(mask_bytes, 256);
    const size_t part = part_doubles * sizeof(double);
    w->part_bytes = part > uniform_bytes ? part : uniform_bytes;
    w->total = w->partials + w->part_bytes;
    return true;
}

size_t attwarp_ragged_mask_workspace_bytes(const attwarp_ragged_image* images, int n, int gh, int gw) {
    RaggedMaskLayout w;
    if (images == nullptr || n <= 0 || gh <= 0 || gw <= 0 || !ragged_mask_layout(images, n, gh, gw, &w)) return 0;
    return w.total;
}

int attwarp_warp_ragged_from_mask(const attwarp_ragged_image* images, const void* mask_u8, int n, int gh, int gw, int C,
                                  const attwarp_transform_params* tp, void* workspace, size_t workspace_bytes,
                                  float* map_x_opt, float* map_y_opt, void* stream) {
    const char* const what = "warp_ragged_from_mask";
    AW_REQUIRE(images && mask_u8 && workspace, "%s: NULL pointer", what);
    AW_REQUIRE(n > 0 && gh > 0 && gw > 0, "%s: n, gh, gw must be positive (got %d, %d, %d)", what, n, gh, gw);
    AW_REQUIRE(C == 1 || C == 3 || C == 4, "%s: C must be 1, 3 or 4 (got %d)", what, C);
    int rc = check_transform(tp);
    if (rc != ATTWARP_OK) return rc;
    if (tp->transform != ATTWARP_T_IDENTITY)
        return fail(ATTWARP_ERR_UNSUPPORTED, "%s: identity transform only (got %d; resize the masks and "
                    "use warp_ragged_from_attention)", what, tp->transform);
    RaggedList l;
    if ((rc = ragged_list(what, images, n, workspace, &l)) != ATTWARP_OK) return rc;
    RaggedMaskLayout w;
    ragged_mask_layout(images, n, gh, gw, &w);
    if (workspace_bytes < w.total)
        return fail(ATTWARP_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", what, workspace_bytes, w.total);
    cudaStream_t st = as_stream(stream);
    if ((rc = refuse_graph_capture(st, what)) != ATTWARP_OK) return rc;
    char* ws = static_cast<char*>(workspace);
    uint8_t* masks = reinterpret_cast<uint8_t*>(ws + w.masks);
    double* partials = reinterpret_cast<double*>(ws + w.partials);

    static thread_local std::vector<char> host_tables;
    host_tables.assign(w.table_bytes, 0);
    RaggedAtt* host_att = reinterpret_cast<RaggedAtt*>(host_tables.data());
    RaggedLanczos* host_lz = reinterpret_cast<RaggedLanczos*>(host_tables.data() + w.lz);
    int2* fused_items = reinterpret_cast<int2*>(host_tables.data() + w.item_at);
    int2* att_items = fused_items + w.fused_items;
    int launches = 0;
    size_t mask_off = 0, mx_off = 0, my_off = 0;
    int64_t part_off = 0, nf = 0, na = 0;
    const uint8_t* mask = static_cast<const uint8_t*>(mask_u8);
    for (int i = 0; i < n; ++i) {
        RaggedImage& r = l.host[i];
        if (map_x_opt != nullptr) r.map_x = map_x_opt + mx_off;
        if (map_y_opt != nullptr) r.map_y = map_y_opt + my_off;
        mx_off += (size_t)r.Wo;
        my_off += (size_t)r.Ho;
        RaggedAtt& a = host_att[i];
        a.H = r.H; a.W = r.W;
        int rows, nt, nx, warps;
        size_t smem;
        if (lanczos_ragged_geometry(gh, gw, r.H, r.W, &rows, &nt, &nx, &warps, &smem)) {
            // the fused kernel: row tiles as chunks, column CTAs as tiles of the finish kernel's partial layout
            a.att = mask + (size_t)i * gh * gw;
            a.chunk_rows = rows; a.n_chunks = nt;
            a.tile_cols = warps * 64; a.n_tiles = nx;
            rc = lanczos_ragged_tables(gh, gw, r.H, r.W, rows, &host_lz[i]);
            if (rc != ATTWARP_OK) return rc;
            host_lz[i].warps = warps;
            for (int t = 0; t < nt; ++t)
                for (int x = 0; x < nx; ++x) fused_items[nf++] = make_int2(i, t << 8 | x);
        } else {
            // resized to image size first, then summed by the ragged uint8 marginals kernel
            a.att = masks + mask_off;
            mask_off += align_up((size_t)r.H * r.W, 16);
            ragged_att_geometry(r.H, r.W, &a.chunk_rows, &a.n_chunks, &a.tile_cols, &a.n_tiles);
            for (int c = 0; c < a.n_chunks; ++c)
                for (int t = 0; t < a.n_tiles; ++t) att_items[na++] = make_int2(i, c << 8 | t);
            rc = launch_resize_lanczos_u8(mask + (size_t)i * gh * gw, 1, gh, gw, r.H, r.W,
                                          static_cast<uint8_t*>(const_cast<void*>(a.att)), st);
            if (rc != ATTWARP_OK) return rc;
            ++launches;
        }
        a.colpart = part_off; part_off += (int64_t)a.n_chunks * r.W;
        a.rowpart = part_off; part_off += (int64_t)a.n_tiles * r.H;
    }
    if (l.degenerate)          // resizes + marginals, finish and resample per image
        return ragged_per_image(l, n, C, st, launches + 3 * n, [&](int i, const RaggedImage& r) {
            float* mx = const_cast<float*>(r.map_x);
            float* my = const_cast<float*>(r.map_y);
            if (host_lz[i].planes != nullptr)           // taken by the fused kernel
                return launch_maps_from_mask(mask + (size_t)i * gh * gw, 1, gh, gw, r.H, r.W, r.Wo, r.Ho, *tp, partials,
                                             w.part_bytes, mx, my, st);
            return launch_maps_from_attention(host_att[i].att, ATTWARP_U8, 1, r.H, r.W, r.Wo, r.Ho, *tp, partials,
                                              w.part_bytes, mx, my, nullptr, st);
        });
    char* dev_tables = ws + w.tables;
    const RaggedAtt* dev_att = reinterpret_cast<const RaggedAtt*>(dev_tables);
    const int2* dev_items = reinterpret_cast<const int2*>(dev_tables + w.item_at);
    const int maps_launches = launches + (w.fused_items > 0) + (w.att_items > 0) + 1;
    return ragged_stage5(l, n, C, st, maps_launches, [&]() -> int {
        AW_CUDA(cudaMemcpyAsync(dev_tables, host_tables.data(), host_tables.size(), cudaMemcpyHostToDevice, st));
        if (w.fused_items > 0) {
            rc = launch_lanczos_marginals_ragged(dev_items, w.fused_items, dev_att,
                                                 reinterpret_cast<const RaggedLanczos*>(dev_tables + w.lz), gw, w.smem,
                                                 partials, st);
            if (rc != ATTWARP_OK) return rc;
        }
        if (w.att_items > 0) {
            rc = launch_marginals_ragged_u8_identity(dev_items + w.fused_items, w.att_items, dev_att, partials, st);
            if (rc != ATTWARP_OK) return rc;
        }
        return launch_maps_from_partials_ragged(n, l.dev, dev_att, partials, l.max_h, l.max_w, *tp, st);
    });
}

// ---------------------------------------------------------------------------------------------
static bool png_shape_ok(int H, int W, int C) {
    return H > 0 && W > 0 && (C == 1 || C == 3 || C == 4) && (int64_t)W * C < ((int64_t)1 << 30);
}

size_t attwarp_png_max_bytes(int H, int W, int C) { return png_shape_ok(H, W, C) ? png_max_bytes_impl(H, W, C) : 0; }

size_t attwarp_png_workspace_bytes(const attwarp_png_image* images, int n) {
    if (images == nullptr || n <= 0) return 0;
    for (int i = 0; i < n; ++i)
        if (!png_shape_ok(images[i].H, images[i].W, images[i].C)) return 0;
    return png_workspace_bytes_impl(images, n);
}

int attwarp_encode_png(const attwarp_png_image* images, int n, void* workspace, size_t workspace_bytes, void* out,
                       size_t out_capacity, int64_t* offsets, void* stream) {
    AW_REQUIRE(images && out && offsets, "encode_png: NULL pointer");
    AW_REQUIRE(n > 0, "encode_png: n must be positive (got %d)", n);
    size_t need_out = 0;
    for (int i = 0; i < n; ++i) {
        const attwarp_png_image& im = images[i];
        AW_REQUIRE(im.src, "encode_png: image %d: NULL pointer", i);
        AW_REQUIRE(im.C == 1 || im.C == 3 || im.C == 4, "encode_png: image %d: C must be 1, 3 or 4 (got %d)", i, im.C);
        AW_REQUIRE(png_shape_ok(im.H, im.W, im.C), "encode_png: image %d: sizes must be positive and W*C below 2^30", i);
        need_out += png_max_bytes_impl(im.H, im.W, im.C);
    }
    AW_REQUIRE(out_capacity >= need_out, "encode_png: output buffer too small (%zu < %zu)", out_capacity, need_out);
    const size_t need = png_workspace_bytes_impl(images, n);
    if (workspace == nullptr || workspace_bytes < need)
        return fail(ATTWARP_ERR_WORKSPACE, "encode_png: workspace too small (%zu < %zu)", workspace_bytes, need);
    cudaStream_t st = as_stream(stream);
    const int rc = refuse_graph_capture(st, "encode_png");
    if (rc != ATTWARP_OK) return rc;
    return launch_encode_png(images, n, workspace, static_cast<uint8_t*>(out), offsets, st);
}

// ---------------------------------------------------------------------------------------------
int attwarp_jpeg_probe(const void* bytes, size_t nbytes, attwarp_jpeg_info* info) {
    AW_REQUIRE(bytes && info, "jpeg_probe: NULL pointer");
    aw::jpeg::Header h;
    aw::jpeg::parse_header(static_cast<const uint8_t*>(bytes), nbytes, &h);
    info->H = h.H;
    info->W = h.W;
    info->components = h.ncomp;
    info->support = h.support;
    return ATTWARP_OK;
}

// the headers of `images`, parsed into a per-thread vector; ATTWARP_OK when every image is device-decodable
static int jpeg_headers(const attwarp_jpeg_image* images, int n, std::vector<aw::jpeg::Header>& hs) {
    hs.resize((size_t)n);
    for (int i = 0; i < n; ++i) {
        const attwarp_jpeg_image& im = images[i];
        AW_REQUIRE(im.host && im.dev && im.dst, "decode_jpeg: image %d: NULL pointer", i);
        const int s = aw::jpeg::parse_header(static_cast<const uint8_t*>(im.host), im.nbytes, &hs[(size_t)i]);
        if (s != aw::jpeg::kOk)
            return fail(ATTWARP_ERR_UNSUPPORTED, "decode_jpeg: image %d is not device-decodable (support code %d)", i, s);
        AW_REQUIRE(im.H == hs[(size_t)i].H && im.W == hs[(size_t)i].W,
                   "decode_jpeg: image %d: dst is %d x %d, the file is %d x %d", i, im.H, im.W, hs[(size_t)i].H,
                   hs[(size_t)i].W);
    }
    return ATTWARP_OK;
}

size_t attwarp_jpeg_workspace_bytes(const attwarp_jpeg_image* images, int n) {
    if (images == nullptr || n <= 0) return 0;
    static thread_local std::vector<aw::jpeg::Header> hs;
    if (jpeg_headers(images, n, hs) != ATTWARP_OK) return 0;
    return jpeg_workspace_bytes_impl(hs.data(), n);
}

int attwarp_decode_jpeg(const attwarp_jpeg_image* images, int n, void* workspace, size_t workspace_bytes,
                        int32_t* status_out, void* stream) {
    AW_REQUIRE(images && status_out, "decode_jpeg: NULL pointer");
    AW_REQUIRE(n > 0, "decode_jpeg: n must be positive (got %d)", n);
    static thread_local std::vector<aw::jpeg::Header> hs;
    int rc = jpeg_headers(images, n, hs);
    if (rc != ATTWARP_OK) return rc;
    const size_t need = jpeg_workspace_bytes_impl(hs.data(), n);
    if (workspace == nullptr || workspace_bytes < need)
        return fail(ATTWARP_ERR_WORKSPACE, "decode_jpeg: workspace too small (%zu < %zu)", workspace_bytes, need);
    cudaStream_t st = as_stream(stream);
    if ((rc = refuse_graph_capture(st, "decode_jpeg")) != ATTWARP_OK) return rc;
    return launch_decode_jpeg(images, hs.data(), n, workspace, status_out, st);
}

// ---------------------------------------------------------------------------------------------
int attwarp_png_probe(const void* bytes, size_t nbytes, attwarp_png_info* info) {
    AW_REQUIRE(bytes && info, "png_probe: NULL pointer");
    aw::png::Header h;
    aw::png::parse_png(static_cast<const uint8_t*>(bytes), nbytes, &h, [](uint32_t, uint32_t) {});
    info->H = h.H;
    info->W = h.W;
    info->colour_type = h.colour;
    info->bit_depth = h.depth;
    info->support = h.support;
    return ATTWARP_OK;
}

// the headers of `files`, parsed into a per-thread vector; ATTWARP_OK when every file is device-decodable
static int png_headers(const attwarp_png_file* files, int n, std::vector<aw::png::Header>& hs) {
    hs.resize((size_t)n);
    for (int i = 0; i < n; ++i) {
        const attwarp_png_file& f = files[i];
        AW_REQUIRE(f.host && f.dev && f.dst, "decode_png: file %d: NULL pointer", i);
        aw::png::Header& h = hs[(size_t)i];
        const int s = aw::png::parse_png(static_cast<const uint8_t*>(f.host), f.nbytes, &h, [](uint32_t, uint32_t) {});
        if (s != aw::png::kPngOk)
            return fail(ATTWARP_ERR_UNSUPPORTED, "decode_png: file %d is not device-decodable (support code %d)", i, s);
        AW_REQUIRE(f.H == h.H && f.W == h.W, "decode_png: file %d: dst is %d x %d, the file is %d x %d", i, f.H, f.W,
                   h.H, h.W);
    }
    return ATTWARP_OK;
}

size_t attwarp_png_decode_workspace_bytes(const attwarp_png_file* files, int n) {
    if (files == nullptr || n <= 0) return 0;
    static thread_local std::vector<aw::png::Header> hs;
    if (png_headers(files, n, hs) != ATTWARP_OK) return 0;
    return png_decode_workspace_bytes_impl(hs.data(), n);
}

int attwarp_decode_png(const attwarp_png_file* files, int n, void* workspace, size_t workspace_bytes,
                       int32_t* status_out, void* stream) {
    AW_REQUIRE(files && status_out, "decode_png: NULL pointer");
    AW_REQUIRE(n > 0, "decode_png: n must be positive (got %d)", n);
    static thread_local std::vector<aw::png::Header> hs;
    int rc = png_headers(files, n, hs);
    if (rc != ATTWARP_OK) return rc;
    const size_t need = png_decode_workspace_bytes_impl(hs.data(), n);
    if (workspace == nullptr || workspace_bytes < need)
        return fail(ATTWARP_ERR_WORKSPACE, "decode_png: workspace too small (%zu < %zu)", workspace_bytes, need);
    cudaStream_t st = as_stream(stream);
    if ((rc = refuse_graph_capture(st, "decode_png")) != ATTWARP_OK) return rc;
    return launch_decode_png(files, hs.data(), n, workspace, status_out, st);
}

// ---------------------------------------------------------------------------------------------
static bool overlay_shape_ok(const attwarp_overlay_image& im) {
    return im.H > 0 && im.W > 0 && im.H <= 65535 && im.W <= 65535 && (im.C == 1 || im.C == 3);
}

size_t attwarp_overlay_workspace_bytes(const attwarp_overlay_image* images, int n, int att_kind) {
    if (images == nullptr || n <= 0 || (att_kind != ATTWARP_OVERLAY_MAP && att_kind != ATTWARP_OVERLAY_TOKENS))
        return 0;
    for (int i = 0; i < n; ++i)
        if (!overlay_shape_ok(images[i])) return 0;
    return overlay_workspace_bytes_impl(images, n, att_kind);
}

int attwarp_attention_overlay(const attwarp_overlay_image* images, int n, int att_dtype, int att_kind, int gh, int gw,
                              double alpha, void* workspace, size_t workspace_bytes, void* stream) {
    AW_REQUIRE(images, "attention_overlay: NULL pointer");
    AW_REQUIRE(n > 0, "attention_overlay: n must be positive (got %d)", n);
    AW_REQUIRE(att_kind == ATTWARP_OVERLAY_MAP || att_kind == ATTWARP_OVERLAY_TOKENS,
               "attention_overlay: bad attention kind %d", att_kind);
    if (att_kind == ATTWARP_OVERLAY_MAP)
        AW_REQUIRE(att_dtype == ATTWARP_U8 || att_dtype == ATTWARP_F32 || att_dtype == ATTWARP_F64,
                   "attention_overlay: attention dtype must be U8, F32 or F64 (got %d)", att_dtype);
    else
        AW_REQUIRE(att_dtype == ATTWARP_F32, "attention_overlay: token maps must be F32 (got dtype %d)", att_dtype);
    AW_REQUIRE(att_kind == ATTWARP_OVERLAY_MAP || (gh > 0 && gw > 0 && gh <= 65535 && gw <= 65535),
               "attention_overlay: token grid %d x %d outside [1, 65535]", gh, gw);
    AW_REQUIRE(isfinite(alpha), "attention_overlay: alpha must be finite");
    for (int i = 0; i < n; ++i) {
        const attwarp_overlay_image& im = images[i];
        AW_REQUIRE(im.src && im.att && im.dst, "attention_overlay: image %d: NULL pointer", i);
        AW_REQUIRE(im.src != im.dst, "attention_overlay: image %d: dst must not be src", i);
        AW_REQUIRE(im.C == 1 || im.C == 3, "attention_overlay: image %d: C must be 1 or 3 (got %d)", i, im.C);
        AW_REQUIRE(overlay_shape_ok(im), "attention_overlay: image %d: H, W must lie in [1, 65535] (got %d x %d)", i,
                   im.H, im.W);
    }
    const size_t need = overlay_workspace_bytes_impl(images, n, att_kind);
    if (workspace == nullptr || workspace_bytes < need)
        return fail(ATTWARP_ERR_WORKSPACE, "attention_overlay: workspace too small (%zu < %zu)", workspace_bytes, need);
    cudaStream_t st = as_stream(stream);
    const int rc = refuse_graph_capture(st, "attention_overlay");
    if (rc != ATTWARP_OK) return rc;
    return launch_attention_overlay(images, n, att_dtype, att_kind, gh, gw, alpha, workspace, st);
}

static int warp_image_host_impl(const void* image_host, int img_dtype, int C, int H, int W,
                                const void* att_host, int att_dtype, int Wo, int Ho,
                                const attwarp_transform_params* tp, void* out_host, int* used_fallback);

int attwarp_warp_image_host(const void* image_host, int img_dtype, int C, int H, int W,
                            const void* att_host, int att_dtype, int Wo, int Ho,
                            const attwarp_transform_params* tp, void* out_host, int* used_fallback) {
    const int rc = warp_image_host_impl(image_host, img_dtype, C, H, W, att_host, att_dtype, Wo, Ho, tp, out_host,
                                        used_fallback);
    // an early return leaves transfers or kernels of this call pending on the arena stream: drain them before
    // the next call reuses the arena (and before the caller frees its host buffers)
    return rc == ATTWARP_OK ? rc : g_arena.drain(rc);
}

static int warp_image_host_impl(const void* image_host, int img_dtype, int C, int H, int W,
                                const void* att_host, int att_dtype, int Wo, int Ho,
                                const attwarp_transform_params* tp, void* out_host, int* used_fallback) {
    AW_REQUIRE(image_host && att_host && out_host, "warp_image_host: NULL pointer");
    AW_REQUIRE(C > 0 && H > 0 && W > 0 && Wo > 0 && Ho > 0, "warp_image_host: sizes must be positive");
    AW_REQUIRE(img_dtype == ATTWARP_U8 || img_dtype == ATTWARP_F32, "warp_image_host: image dtype must be u8/f32");
    AW_REQUIRE(att_dtype == ATTWARP_U8 || att_dtype == ATTWARP_F32 || att_dtype == ATTWARP_F64,
               "warp_image_host: attention dtype must be u8/f32/f64");
    int rc = check_transform(tp);
    if (rc != ATTWARP_OK) return rc;
    const size_t es = dtype_size(img_dtype);
    const size_t img_b = align_up((size_t)H * W * C * es, 256);
    const size_t out_b = align_up((size_t)Ho * Wo * C * es, 256);
    const size_t att_b = align_up((size_t)H * W * dtype_size(att_dtype), 256);
    const size_t ws_b = align_up(maps_workspace_bytes_impl(1, H, W), 256);
    const size_t mx_b = align_up(sizeof(float) * Wo, 256), my_b = align_up(sizeof(float) * Ho, 256);
    rc = g_arena.ensure(img_b + out_b + att_b + ws_b + mx_b + my_b + 256);
    if (rc != ATTWARP_OK) return rc;
    char* p = static_cast<char*>(g_arena.dev);
    void* d_img = p; p += img_b;
    void* d_out = p; p += out_b;
    void* d_att = p; p += att_b;
    void* d_ws = p; p += ws_b;
    float* d_mx = reinterpret_cast<float*>(p); p += mx_b;
    float* d_my = reinterpret_cast<float*>(p); p += my_b;
    int* d_flag = reinterpret_cast<int*>(p);
    cudaStream_t st = g_arena.stream;
    const size_t n_att = (size_t)H * W * dtype_size(att_dtype), n_img = (size_t)H * W * C * es;
    const size_t n_out = (size_t)Ho * Wo * C * es;
    // The caller's buffers are pageable: the copies are most of the call (100 of 112 us at 336^2; the kernels take
    // 14 us).  Measured per direction (profiles/r08i_pinned_modes.txt): receiving the output in pinned memory of this
    // thread's arena and copying it to the caller with memcpy saves 9-14 us per call (112.8 -> 98.6 us at 336^2,
    // 141 -> 132 us for a 500^2 output); staging the INPUTS the same way gains nothing (the driver's pageable
    // host-to-device path already returns as soon as it has taken its copy), so they are passed as they are.
    // ATTWARP_HOST_PINNED: 0 off, 1 both directions, 2 inputs only, 3 output only (default).
    static const int pinned_mode = [] {
        const char* e = getenv("ATTWARP_HOST_PINNED");
        return e == nullptr ? 3 : atoi(e);
    }();
    const bool use_pinned = pinned_mode != 0, pin_in = pinned_mode != 3, pin_out = pinned_mode != 2;
    if (use_pinned && att_b + img_b + out_b + 256 <= ((size_t)1 << 30) && g_arena.ensure_pinned(att_b + img_b + out_b + 256)) {
        char* q = static_cast<char*>(g_arena.pin);
        void* p_att = q; q += att_b;
        void* p_img = q; q += img_b;
        void* p_out = q; q += out_b;
        int* p_flag = reinterpret_cast<int*>(q);
        if (pin_in) memcpy(p_att, att_host, n_att);
        AW_CUDA(cudaMemcpyAsync(d_att, pin_in ? p_att : att_host, n_att, cudaMemcpyHostToDevice, st));
        rc = launch_maps_from_attention(d_att, att_dtype, 1, H, W, Wo, Ho, *tp, d_ws, ws_b, d_mx, d_my, d_flag, st);
        if (rc != ATTWARP_OK) return rc;
        if (pin_in) memcpy(p_img, image_host, n_img);   // while the map is on its way and the maps kernels run
        AW_CUDA(cudaMemcpyAsync(d_img, pin_in ? p_img : image_host, n_img, cudaMemcpyHostToDevice, st));
        rc = launch_remap(d_img, d_out, img_dtype, ATTWARP_LAYOUT_HWC, 1, C, H, W, Ho, Wo, d_mx, d_my, st);
        if (rc != ATTWARP_OK) return rc;
        AW_CUDA(cudaMemcpyAsync(pin_out ? p_out : out_host, d_out, n_out, cudaMemcpyDeviceToHost, st));
        AW_CUDA(cudaMemcpyAsync(p_flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        AW_CUDA(cudaStreamSynchronize(st));
        if (pin_out) memcpy(out_host, p_out, n_out);
        if (used_fallback) *used_fallback = *p_flag;
        return ATTWARP_OK;
    }
    AW_CUDA(cudaMemcpyAsync(d_att, att_host, n_att, cudaMemcpyHostToDevice, st));
    AW_CUDA(cudaMemcpyAsync(d_img, image_host, n_img, cudaMemcpyHostToDevice, st));
    rc = launch_maps_from_attention(d_att, att_dtype, 1, H, W, Wo, Ho, *tp, d_ws, ws_b, d_mx, d_my, d_flag, st);
    if (rc != ATTWARP_OK) return rc;
    rc = launch_remap(d_img, d_out, img_dtype, ATTWARP_LAYOUT_HWC, 1, C, H, W, Ho, Wo, d_mx, d_my, st);
    if (rc != ATTWARP_OK) return rc;
    AW_CUDA(cudaMemcpyAsync(out_host, d_out, n_out, cudaMemcpyDeviceToHost, st));
    int flag = 0;
    AW_CUDA(cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    AW_CUDA(cudaStreamSynchronize(st));
    if (used_fallback) *used_fallback = flag;
    return ATTWARP_OK;
}

// ---------------------------------------------------------------------------------------------
int attwarp_safe_softmax(const float* logits, int B, int N, float eps, float* out, void* stream) {
    AW_REQUIRE(logits && out, "safe_softmax: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0, "safe_softmax: sizes must be positive");
    return launch_safe_softmax(logits, B, N, eps, out, as_stream(stream));
}

int attwarp_safe_softmax_mix(const float* logits, int B, int N, float eps, float alpha, float* out, void* stream) {
    AW_REQUIRE(logits && out, "safe_softmax_mix: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0, "safe_softmax_mix: sizes must be positive");
    return launch_safe_softmax_mix(logits, B, N, eps, alpha, out, as_stream(stream));
}

int attwarp_safe_softmax_mix_backward(const float* logits, const float* grad_out, int B, int N, float eps, float alpha,
                                      float* grad_logits, void* stream) {
    AW_REQUIRE(logits && grad_out && grad_logits, "safe_softmax_mix_backward: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0, "safe_softmax_mix_backward: sizes must be positive");
    return launch_safe_softmax_mix_backward(logits, grad_out, B, N, eps, alpha, grad_logits, as_stream(stream));
}

int attwarp_mix_with_uniform(const float* p, int B, int N, float alpha, float* out, void* stream) {
    AW_REQUIRE(p && out, "mix_with_uniform: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0, "mix_with_uniform: sizes must be positive");
    return launch_mix_with_uniform(p, B, N, alpha, out, as_stream(stream));
}

// ---------------------------------------------------------------------------------------------
int attwarp_revise_mask(const float* tok, int B, int gh, int gw, int kernel_size, float enhance_coe,
                        float* revised, void* mask_u8, void* stream) {
    AW_REQUIRE(tok && (revised || mask_u8), "revise_mask: NULL pointer");
    AW_REQUIRE(B > 0 && gh > 0 && gw > 0 && gh * gw > 1, "revise_mask: sizes must be positive (and more than one token)");
    AW_REQUIRE(kernel_size > 0 && (kernel_size & 1), "revise_mask: kernel_size must be odd (got %d)", kernel_size);
    return launch_revise_mask(tok, B, gh, gw, kernel_size, enhance_coe, revised, static_cast<uint8_t*>(mask_u8),
                              as_stream(stream));
}

int attwarp_resize_lanczos_u8(const void* src, int B, int h, int w, int Ho, int Wo, void* dst, void* stream) {
    AW_REQUIRE(src && dst && src != dst, "resize_lanczos_u8: bad pointers");
    AW_REQUIRE(B > 0 && h > 0 && w > 0 && Ho > 0 && Wo > 0, "resize_lanczos_u8: sizes must be positive");
    AW_REQUIRE(B <= 65535, "resize_lanczos_u8: B=%d exceeds 65535", B);
    return launch_resize_lanczos_u8(static_cast<const uint8_t*>(src), B, h, w, Ho, Wo, static_cast<uint8_t*>(dst),
                                    as_stream(stream));
}

int attwarp_make_strictly_increasing(const float* F, int B, int N, float eps, float* out, void* stream) {
    AW_REQUIRE(F && out, "make_strictly_increasing: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0, "make_strictly_increasing: sizes must be positive");
    return launch_strictly_increasing(F, B, N, eps, out, as_stream(stream));
}

int attwarp_interp_linear_rows(const float* F, int B, int N, int L, float* out, void* stream) {
    AW_REQUIRE(F && out, "interp_linear_rows: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0 && L > 0, "interp_linear_rows: sizes must be positive");
    AW_REQUIRE(B <= 65535, "interp_linear_rows: B=%d exceeds 65535", B);
    return launch_interp_linear_rows(F, B, N, L, out, as_stream(stream));
}

int attwarp_cdf_from_density(const float* p, int B, int N, float* F, void* stream) {
    AW_REQUIRE(p && F, "cdf_from_density: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0, "cdf_from_density: sizes must be positive");
    return launch_cdf_from_density(p, B, N, F, as_stream(stream));
}

int attwarp_gt_marginals(const float* A, int B, int H, int W, void* workspace, size_t workspace_bytes,
                         float* px, float* py, void* stream) {
    AW_REQUIRE(A && px && py, "gt_marginals: NULL pointer");
    AW_REQUIRE(B > 0 && H > 0 && W > 0, "gt_marginals: sizes must be positive");
    AW_REQUIRE(B <= 65535, "gt_marginals: B=%d exceeds 65535", B);
    return launch_gt_marginals(A, B, H, W, workspace, workspace_bytes, px, py, as_stream(stream));
}

int attwarp_upsample_right_inverse(const float* y, const float* M, int B, int L_out, int L_in, float* x,
                                   void* stream) {
    AW_REQUIRE(y && M && x, "upsample_right_inverse: NULL pointer");
    AW_REQUIRE(B > 0 && L_out > 0 && L_in > 0, "upsample_right_inverse: sizes must be positive");
    AW_REQUIRE(B <= 65535 && L_out <= 4096, "upsample_right_inverse: B<=65535 and L_out<=4096 required");
    return launch_upsample_right_inverse(y, M, B, L_out, L_in, x, as_stream(stream));
}

int attwarp_safe_softmax_backward(const float* logits, const float* grad_out, int B, int N, float eps,
                                  float* grad_logits, void* stream) {
    AW_REQUIRE(logits && grad_out && grad_logits, "safe_softmax_backward: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0, "safe_softmax_backward: sizes must be positive");
    return launch_safe_softmax_backward(logits, grad_out, B, N, eps, grad_logits, as_stream(stream));
}

int attwarp_mix_with_uniform_backward(const float* grad_out, int B, int N, float alpha, float* grad_p, void* stream) {
    AW_REQUIRE(grad_out && grad_p, "mix_with_uniform_backward: NULL pointer");
    AW_REQUIRE(B > 0 && N > 0, "mix_with_uniform_backward: sizes must be positive");
    return launch_mix_with_uniform_backward(grad_out, B, N, alpha, grad_p, as_stream(stream));
}

int attwarp_upsample_right_inverse_backward(const float* grad_x, const float* M, int B, int L_out, int L_in,
                                            float* grad_y, void* stream) {
    AW_REQUIRE(grad_x && M && grad_y, "upsample_right_inverse_backward: NULL pointer");
    AW_REQUIRE(B > 0 && L_out > 0 && L_in > 0, "upsample_right_inverse_backward: sizes must be positive");
    return launch_upsample_right_inverse_backward(grad_x, M, B, L_out, L_in, grad_y, as_stream(stream));
}

int attwarp_adaptive_avg_pool2d(const float* A, int B, int H, int W, int gh, int gw, float* out,
                                void* stream) {
    AW_REQUIRE(A && out, "adaptive_avg_pool2d: NULL pointer");
    AW_REQUIRE(B > 0 && H > 0 && W > 0 && gh > 0 && gw > 0, "adaptive_avg_pool2d: sizes must be positive");
    AW_REQUIRE(B <= 65535, "adaptive_avg_pool2d: B=%d exceeds 65535", B);
    return launch_adaptive_avg_pool2d(A, nullptr, B, H, W, gh, gw, out, as_stream(stream));
}

int attwarp_pool_attention(const float* A, const unsigned char* sqrt_mask, int B, int H, int W, int gh, int gw,
                           float* out, void* stream) {
    AW_REQUIRE(A && sqrt_mask && out, "pool_attention: NULL pointer");
    AW_REQUIRE(B > 0 && H > 0 && W > 0 && gh > 0 && gw > 0, "pool_attention: sizes must be positive");
    AW_REQUIRE(B <= 65535, "pool_attention: B=%d exceeds 65535", B);
    return launch_adaptive_avg_pool2d(A, sqrt_mask, B, H, W, gh, gw, out, as_stream(stream));
}

// ---------------------------------------------------------------------------------------------
size_t attwarp_pdf_l1_loss_workspace_bytes(int B) { return B > 0 ? sizeof(double) * 2 * (size_t)B + 16 : 0; }

static int check_pdf_loss_args(const float* px, const float* py, const float* gx, const float* gy, int B, int Nx, int Ny,
                               int Ngx, int Ngy, const float* Mx, const float* My, const float* Mgx, const float* Mgy,
                               int W, int H) {
    AW_REQUIRE(px && py && gx && gy && Mx && My && Mgx && Mgy, "pdf_l1_loss: NULL pointer");
    AW_REQUIRE(B > 0 && Nx > 0 && Ny > 0 && Ngx > 0 && Ngy > 0 && W > 0 && H > 0, "pdf_l1_loss: sizes must be positive");
    AW_REQUIRE(B <= 65535, "pdf_l1_loss: B=%d exceeds 65535", B);
    return ATTWARP_OK;
}

int attwarp_pdf_l1_loss(const float* px, const float* py, const float* gx, const float* gy, int B, int Nx, int Ny,
                        int Ngx, int Ngy, const float* Mx, const float* My, const float* Mgx, const float* Mgy, int W,
                        int H, void* workspace, size_t workspace_bytes, float* loss, void* stream) {
    int rc = check_pdf_loss_args(px, py, gx, gy, B, Nx, Ny, Ngx, Ngy, Mx, My, Mgx, Mgy, W, H);
    if (rc != ATTWARP_OK) return rc;
    AW_REQUIRE(loss, "pdf_l1_loss: NULL pointer");
    if (workspace == nullptr || workspace_bytes < attwarp_pdf_l1_loss_workspace_bytes(B))
        return fail(ATTWARP_ERR_WORKSPACE, "pdf_l1_loss: workspace too small");
    return launch_pdf_l1_loss(px, py, gx, gy, B, Nx, Ny, Ngx, Ngy, Mx, My, Mgx, Mgy, W, H, workspace, loss,
                              as_stream(stream));
}

int attwarp_pdf_l1_loss_backward(const float* px, const float* py, const float* gx, const float* gy, int B, int Nx,
                                 int Ny, int Ngx, int Ngy, const float* Mx, const float* My, const float* Mgx,
                                 const float* Mgy, int W, int H, const float* upstream, float* grad_px, float* grad_py,
                                 void* stream) {
    int rc = check_pdf_loss_args(px, py, gx, gy, B, Nx, Ny, Ngx, Ngy, Mx, My, Mgx, Mgy, W, H);
    if (rc != ATTWARP_OK) return rc;
    AW_REQUIRE(upstream && grad_px && grad_py, "pdf_l1_loss_backward: NULL pointer");
    return launch_pdf_l1_loss_backward(px, py, gx, gy, B, Nx, Ny, Ngx, Ngy, Mx, My, Mgx, Mgy, W, H, upstream, grad_px,
                                       grad_py, as_stream(stream));
}

}  // extern "C"
