/*
 * attwarp.h -- C ABI of libattwarp_sm100.so: the B200 (sm_100a) implementation of AttWarp's
 * attention-guided warp hot path.
 *
 * The reference (dwipddalal/AttWarp) has no FFI/plugin layer: its boundary is a set of Python
 * functions that run NumPy/OpenCV/PyTorch on the host.  Each entry point below names the
 * reference function (file:line under the reference root) whose arithmetic it replaces.
 * `AGW/`  = "Attention Guided Warping/",  `mnfd/` = "model/marginalnet_full_dataset/".
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is
 *     enqueued on it and nothing synchronises, except the `*_host` convenience entry points
 *     which block until their result is in the caller's host buffer;
 *   - return value: ATTWARP_OK (0) or a negative attwarp_status; attwarp_last_error() returns a
 *     thread-local human-readable message for the last failure on the calling thread;
 *   - no global mutable state (the reference's module-global transform selection,
 *     AGW/new_method.py:191,378-403, travels in attwarp_transform_params instead);
 *   - inputs are never written; outputs and workspaces are caller-allocated.
 */
#ifndef ATTWARP_H_
#define ATTWARP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ATTWARP_ABI_VERSION 1

typedef enum attwarp_status {
    ATTWARP_OK = 0,
    ATTWARP_ERR_INVALID_ARG = -1,  /* NULL pointer, non-positive size, bad enum            */
    ATTWARP_ERR_UNSUPPORTED = -2,  /* valid request outside the implemented envelope        */
    ATTWARP_ERR_CUDA = -3,         /* CUDA runtime / launch failure (message has the cause) */
    ATTWARP_ERR_WORKSPACE = -4     /* workspace pointer NULL or too small                   */
} attwarp_status;

typedef enum attwarp_dtype {
    ATTWARP_U8 = 0,
    ATTWARP_F32 = 1,
    ATTWARP_F64 = 2,
    ATTWARP_BF16 = 3,
    ATTWARP_F16 = 4
} attwarp_dtype;

/* AGW/new_method.py:133-188 (transform registry) */
typedef enum attwarp_transform {
    ATTWARP_T_IDENTITY = 0,
    ATTWARP_T_SQUARE = 1,
    ATTWARP_T_SQRT = 2,
    ATTWARP_T_EXP = 3, /* exp(exp_scale*x)/exp_divisor */
    ATTWARP_T_LOG = 4  /* log(x + 1e-5)                */
} attwarp_transform;

/* Replaces the module globals ATTENTION_TRANSFORM, EXP_SCALE, EXP_DIVISOR,
 * APPLY_INVERSE_TO_MARGINALS (AGW/new_method.py:159-191) set by set_transform_function
 * (AGW/new_method.py:378-403).  BASE_ATTENTION and EPSILON are fixed at 1e-9 (:194-195). */
typedef struct attwarp_transform_params {
    int32_t transform;     /* attwarp_transform */
    int32_t apply_inverse; /* 0/1 */
    double exp_scale;
    double exp_divisor;
} attwarp_transform_params;

typedef enum attwarp_layout {
    ATTWARP_LAYOUT_HWC = 0, /* [B][H][W][C]  (cv2 / NumPy images, AGW/new_method.py:198)       */
    ATTWARP_LAYOUT_CHW = 1  /* [B][C][H][W]  (torch images, mnfd/checkpoint_utils.py:133-147)   */
} attwarp_layout;

/* ------------------------------------------------------------------------------------------ */
int attwarp_abi_version(void);
const char* attwarp_last_error(void);
/* Number of SMs of the current device and whether it is compute capability 10.x. */
int attwarp_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* How much of each SM one launch of the two streaming kernels (stage 1 aggregation, stage 5 resample) may occupy.
 * 1 (default): the whole SM -- the lowest latency for one batch at a time.  2: half, so that the kernels of two
 * independent batches enqueued on different streams are co-resident on every SM (stage 1 is HBM-bound and leaves
 * issue slots idle, stage 5 the opposite): +9 % images/s at BASELINE configs[1] over four streams, at the price of a
 * slower single batch.  Process-wide, read at every launch; returns the previous value.  (No reference counterpart:
 * the reference warps one image at a time on the host.) */
int attwarp_set_sm_share(int share);

/* ------------------------------------------------------------------------------------------
 * Stage 1 -- attention aggregation.
 * Replaces MaskHookLogger._process_attention + finalize
 *   (AGW/attention_extraction/llava.py:94-116, 124-132) and
 *   BatchMaskHookLogger._process_attention + finalize_batch (llava.py:385-396, 401-411):
 *
 *   out[b,t] = 1/(L*Hh) * sum_l sum_h  a[b,l,h,t] / (sum_t' a[b,l,h,t'] + eps)
 *   with a[b,l,h,t] = attn[b*stride_b + l*stride_l + h*stride_h + tok_start[b] + t]
 *
 * The reference appends one head-mean per hooked forward call ("step") and averages the list;
 * `L` plays the role of that step list (SURVEY.md "fact 3").  The live hook layout
 * [B,Hh,q,kv] is addressed with L=1, stride_h = q*kv and the base pointer advanced to the last
 * query row.  Input is upcast to fp32; accumulation is fp32 in a fixed (deterministic) order.
 *
 * attn      : dtype BF16 / F16 / F32, T contiguous elements per (b,l,h) row
 * tok_start : int32[B] per-sample offset into the row (NULL = 0), llava.py:99-105, 389-391
 * workspace : attwarp_aggregate_workspace_bytes(B,L,Hh,T) bytes of device scratch
 * out       : float32 [B,T]
 * accumulate/out_scale: out = (accumulate ? out : 0) + out_scale * mean  (running step mean
 *             for a live hook; use accumulate=0, out_scale=1 for a one-shot reduction)
 */
size_t attwarp_aggregate_workspace_bytes(int B, int L, int Hh, int T);
int attwarp_aggregate_attention(const void* attn, int dtype, int B, int L, int Hh, int T,
                                int64_t stride_b, int64_t stride_l, int64_t stride_h,
                                const int32_t* tok_start, float eps, void* workspace,
                                size_t workspace_bytes, float* out, int accumulate,
                                float out_scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stages 2b-4, NumPy path -- attention map -> separable inverse-CDF warp maps.
 * Replaces warp_image_by_attention up to the np.interp calls (AGW/new_method.py:207-261):
 * clamp>=0, transform, +1e-9, axis sums, optional inverse on the marginals, near-zero fallback,
 * cumsum/total, forward knots (last forced to the output size), np.interp inversion, float32
 * cast.  All of it in float64 like the reference.
 *
 * att        : [B][H][W] dense, dtype U8 / F32 / F64
 * map_x/map_y: float32 [B][Wo] / [B][Ho]  -- the rows/cols of the reference's meshgrid
 *              (AGW/new_method.py:263-265); the 2-D grid is never materialised
 * workspace  : attwarp_maps_workspace_bytes(B,H,W) bytes
 */
size_t attwarp_maps_workspace_bytes(int B, int H, int W);
int attwarp_maps_from_attention(const void* att, int att_dtype, int B, int H, int W, int Wo,
                                int Ho, const attwarp_transform_params* tp, void* workspace,
                                size_t workspace_bytes, float* map_x, float* map_y,
                                void* stream);

/* Same arithmetic when the full-resolution map is an index-upsampled token grid
 * att[y][x] = tok[(y*gh)/H][(x*gw)/W]  (configs[1]/[2] of BASELINE.json: 24x24 LLaVA grid to
 * 336x336, 48x48 to 1344x1344).  The full-resolution map is never materialised.
 * tok: float32 [B][gh][gw];  no workspace. */
int attwarp_maps_from_tokens(const float* tok, int B, int gh, int gw, int H, int W, int Wo,
                             int Ho, const attwarp_transform_params* tp, float* map_x,
                             float* map_y, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage 4, torch path -- CDFs -> warp maps.
 * Replaces the per-sample loop body of warp_from_cdf_torch (mnfd/checkpoint_utils.py:157-189):
 * knots [0,F]*out_size in float64, last forced to out_size, the tie-break branch (:181-184,
 * float32 increments), np.interp, float32 cast.
 * Fx: float32 [B][W], Fy: float32 [B][H] -> map_x float32 [B][Wo], map_y float32 [B][Ho]. */
int attwarp_maps_from_cdf(const float* Fx, const float* Fy, int B, int H, int W, int Wo, int Ho,
                          float* map_x, float* map_y, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage 5 -- bilinear resample through separable maps, bit-compatible with
 * cv2.remap(img, meshgrid(map_x,map_y), INTER_LINEAR, BORDER_REPLICATE) as called at
 * AGW/new_method.py:268-271 and mnfd/checkpoint_utils.py:195-198: coordinates quantised to 1/32
 * px by round-half-even, replicate border, uint8 through 15-bit fixed-point weights, float32
 * through float32 weights without FMA contraction.
 * src: [B] images HxW, C channels, dtype U8 / F32, layout HWC or CHW, dense.
 * dst: [B] images HoxWo, same dtype/layout.  map_x: [B][Wo], map_y: [B][Ho]. */
int attwarp_remap_bilinear(const void* src, void* dst, int dtype, int layout, int B, int C,
                           int H, int W, int Ho, int Wo, const float* map_x, const float* map_y,
                           void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused batch drivers (one host call per batch; kernels back to back on `stream`).
 *
 * attwarp_warp_from_attention_tokens: stages 1-5 for a uniform batch (BASELINE configs[1]):
 *   attention [B,L,Hh,*] -> token map [B,gh*gw] -> maps -> warped uint8/float32 images.
 * tok_out / map_x / map_y are outputs the caller may inspect (required, not optional).
 * workspace: attwarp_aggregate_workspace_bytes(B,L,Hh,gh*gw).
 * stage_events: NULL, or 4 cudaEvent_t handles recorded on `stream` before stage 1, after
 *   stage 1, after stages 2-4 and after stage 5 (per-kernel timing for the roofline report). */
int attwarp_warp_from_attention_tokens(const void* attn, int attn_dtype, int B, int L, int Hh,
                                       int64_t stride_b, int64_t stride_l, int64_t stride_h,
                                       const int32_t* tok_start, int gh, int gw,
                                       const void* src, void* dst, int img_dtype, int layout,
                                       int C, int H, int W, int Ho, int Wo,
                                       const attwarp_transform_params* tp, void* workspace,
                                       size_t workspace_bytes, float* tok_out, float* map_x,
                                       float* map_y, void* const* stage_events, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Mask post-processing of the driver flow (AGW/attention_extraction/llava.py:207-256, called at
 * AGW/main.py:361 and AGW/main_batched.py:268), SURVEY section 8(f) N2.
 *
 * attwarp_revise_mask: tok [B][gh*gw] float32 -> revise_mask (min-max, z-score x enhance_coe, sigmoid,
 *   clamp, kernel_size x kernel_size box filter with replicate padding; llava.py:207-238) as float32
 *   `revised` [B][gh*gw] (nullable) and, like ToPILImage, as uint8 `mask_u8` [B][gh*gw] (nullable).
 * attwarp_resize_lanczos_u8: src [B][h][w] uint8 -> dst [B][Ho][Wo], bit-identical to
 *   PIL.Image.resize((Wo, Ho), LANCZOS) on mode-'L' images (llava.py:195-196, 253).
 * The mask at image size is what the drivers hand to save_warped_image as att_map; feed it to
 * attwarp_maps_from_attention (ATTWARP_U8).
 */
int attwarp_revise_mask(const float* tok, int B, int gh, int gw, int kernel_size, float enhance_coe,
                        float* revised, void* mask_u8, void* stream);
int attwarp_resize_lanczos_u8(const void* src, int B, int h, int w, int Ho, int Wo, void* dst, void* stream);

/* attwarp_maps_from_mask: the two steps above fused with stage 2b for the flow that only warps (the mask itself
 * is not kept): mask_u8 [B][h][w] (attwarp_revise_mask's uint8 output) -> separable maps of the image whose
 * attention is that mask resized to H x W with LANCZOS -- llava.py:253 followed by new_method.py:207-261 -- with
 * the H x W mask never written to memory (its marginal sums are taken where it is computed; exact integers).
 * Identity transform and up-scaling (H > h, W > w) only: ATTWARP_ERR_UNSUPPORTED otherwise (resize, then
 * attwarp_maps_from_attention).  Workspace: attwarp_maps_from_mask_workspace_bytes (0 = shape not supported).
 */
size_t attwarp_maps_from_mask_workspace_bytes(int B, int h, int w, int H, int W);
int attwarp_maps_from_mask(const void* mask_u8, int B, int h, int w, int H, int W, int Wo, int Ho,
                           const attwarp_transform_params* tp, void* workspace, size_t workspace_bytes,
                           float* map_x, float* map_y, void* stream);

/* ---------------------------------------------------------------------------------------------
 * attwarp_warp_from_pdfs: predicted marginal PDFs -> warped images in three launches (BASELINE
 * configs[4]).  Replaces the chain of model/marginalnet_full_dataset/trainer.py:212-218, 285-289:
 *   mix_with_uniform(p, alpha) -> upsample_pdf_right_inverse(p, L).clamp_min(0) -> cdf_from_density
 *   -> warp_from_cdf_torch(img, Fx, Fy, out_size)
 * px [B][Nx], py [B][Ny] : float32 PDFs over the token grid (MarginalNet outputs, model.py:93-95)
 * Mx [W][Nx], My [H][Ny] : right-inverse matrices as for attwarp_upsample_right_inverse
 * src/dst                : images as for attwarp_remap_bilinear (dtype u8/f32, layout HWC/CHW)
 * Fx [B][W], Fy [B][H], map_x [B][Wo], map_y [B][Ho] : device scratch owned by the caller; on return
 *                          (in stream order) they hold the CDFs and the separable maps
 */
int attwarp_warp_from_pdfs(const float* px, const float* py, int B, int Nx, int Ny, float alpha,
                           const float* Mx, const float* My, const void* src, void* dst, int dtype,
                           int layout, int C, int H, int W, int Ho, int Wo, float* Fx, float* Fy,
                           float* map_x, float* map_y, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Ragged batches (BASELINE configs[3]: mixed resolutions): n independent images of different
 * shapes in ONE launch per stage.  Replaces the per-image loop of the reference drivers
 * (AGW/main.py:395-533 and AGW/main_batched.py:243-287 call save_warped_image ->
 * warp_image_by_attention once per image).
 *
 * images    : HOST array of n descriptors; src/dst are DEVICE pointers to dense HWC uint8 images
 *             ([H][W][C] -> [Ho][Wo][C]) that must stay valid until the stream has run the call
 * tok       : device [n][gh*gw] float32 token maps (stage-1 output), index-upsampled to each
 *             image's H x W exactly like attwarp_maps_from_tokens
 * workspace : attwarp_ragged_workspace_bytes(images, n) bytes of device scratch (descriptor table
 *             + the per-image map rows)
 * The call uploads its descriptor tables from host memory and fans the stage-5 launches out over internal streams;
 * it returns ATTWARP_ERR_UNSUPPORTED on a stream that is being captured into a CUDA graph.
 */
typedef struct attwarp_ragged_image {
    const void* src;
    void* dst;
    int32_t H, W, Ho, Wo;
} attwarp_ragged_image;

size_t attwarp_ragged_workspace_bytes(const attwarp_ragged_image* images, int n);
int attwarp_warp_ragged_from_tokens(const float* tok, int n, int gh, int gw,
                                    const attwarp_ragged_image* images, int C,
                                    const attwarp_transform_params* tp, void* workspace,
                                    size_t workspace_bytes, void* stream);

/* Ragged batch warped by each image's OWN attention map (warp_image_by_attention(image, att_map, w, h) per image,
 * AGW/new_method.py:198-283, for a mixed-size list): stages 2b-5 with one marginals launch for all maps, one
 * finish launch, and the stage-5 launches of attwarp_warp_ragged_from_tokens.
 *
 * images    : as for attwarp_warp_ragged_from_tokens
 * att       : HOST array of n entries:
 *               att    device [H][W] map of att_dtype (the image's own size), dense rows, any byte alignment
 *                      (float32 / float64 maps: aligned to their element size)
 *               map_x  device [Wo] floats or NULL: receives the image's map_x (else it stays in the workspace)
 *               map_y  device [Ho] floats or NULL
 * att_dtype : ATTWARP_U8, ATTWARP_F32 or ATTWARP_F64, one for all maps
 * tp        : NumPy semantics (clamp at 0, transform, + 1e-9, float64 sums), as attwarp_maps_from_attention
 * workspace : attwarp_ragged_attention_workspace_bytes(images, n) bytes of device scratch (0: invalid sizes)
 * An image's maps depend on its own map only (its chunk / tile geometry follows from its H x W), so they are
 * bit-identical to those of a call on that image alone.  Images with H or W below 2 make the call go image by
 * image through the uniform entry points.  Host-side descriptor tables: ATTWARP_ERR_UNSUPPORTED under CUDA-graph
 * capture; ATTWARP_ERR_UNSUPPORTED when the largest H + W do not fit the shared-memory knots. */
typedef struct attwarp_ragged_attention {
    const void* att;
    float* map_x;
    float* map_y;
} attwarp_ragged_attention;

size_t attwarp_ragged_attention_workspace_bytes(const attwarp_ragged_image* images, int n);
int attwarp_warp_ragged_from_attention(const attwarp_ragged_image* images, const attwarp_ragged_attention* att,
                                       int n, int att_dtype, int C, const attwarp_transform_params* tp,
                                       void* workspace, size_t workspace_bytes, void* stream);

/* Ragged batch warped by the drivers' own attention, built from token maps: per image blend_mask's uint8 mask
 * (revise_mask, then Pillow's LANCZOS resize to the image's own size; llava.py:240-256) followed by
 * save_warped_image(..., "identity") (new_method.py:207-283), for a mixed-size list -- attwarp_maps_from_mask for
 * every image, with one launch per stage for the whole list and no image-size mask written for the images the fused
 * kernel takes.
 *
 * images    : as for attwarp_warp_ragged_from_tokens
 * mask_u8   : device [n][gh][gw] uint8, attwarp_revise_mask's uint8 output for the n token maps
 * tp        : identity transform only (apply_inverse 0 or 1); ATTWARP_ERR_UNSUPPORTED otherwise
 * workspace : attwarp_ragged_mask_workspace_bytes(images, n, gh, gw) bytes of device scratch (0: invalid sizes)
 * map_x_opt : NULL, or device floats [sum of Wo]: receives the images' map_x rows back to back, in list order
 * map_y_opt : NULL, or device floats [sum of Ho]: the same for map_y
 * An image whose resize attwarp_maps_from_mask takes on the tensor cores (an up-scaling of both axes that fits its
 * tiles) keeps the tiles, coefficients and partial sums of a call on that image alone, so its maps are bit-identical
 * to attwarp_maps_from_mask on that image; the others (down-scaling, image smaller than the token grid, ...) are
 * resized with attwarp_resize_lanczos_u8 into the workspace and summed with the marginals kernel of
 * attwarp_warp_ragged_from_attention.  Then one finish launch for all images and the stage-5 launches of
 * attwarp_warp_ragged_from_tokens.  Images with H or W below 2 make the call go image by image.  The coefficient
 * tables are built on the host and uploaded once per size and device, like attwarp_maps_from_mask's.  Host-side
 * descriptor tables: ATTWARP_ERR_UNSUPPORTED under CUDA-graph capture. */
size_t attwarp_ragged_mask_workspace_bytes(const attwarp_ragged_image* images, int n, int gh, int gw);
int attwarp_warp_ragged_from_mask(const attwarp_ragged_image* images, const void* mask_u8, int n, int gh, int gw, int C,
                                  const attwarp_transform_params* tp, void* workspace, size_t workspace_bytes,
                                  float* map_x_opt, float* map_y_opt, void* stream);

/* Kernel launches the calling thread's last attwarp_warp_ragged_from_tokens / attwarp_warp_ragged_from_attention /
 * attwarp_warp_ragged_from_mask call enqueued: the maps launches (tokens: one; attention: marginals + finish; mask:
 * one resize per image the fused kernel does not take, the fused marginals, the uint8 marginals when some image
 * needs them, finish) + one stage-5 launch per non-empty class (images are grouped by the consumer warps their
 * strips need and by whether their destination rows are 4-byte aligned).  For accounting (bench.py's
 * gpu_launches). */
int attwarp_ragged_last_launches(void);

/* attwarp_warp_image_host: the whole of warp_image_by_attention (AGW/new_method.py:198-283) for
 * ONE image with HOST buffers, as the NumPy signature implies: H2D, stages 2b-5 on the device,
 * D2H, blocking.  image_host: uint8/float32 [H][W][C]; att_host: U8/F32/F64 [H][W];
 * out_host: [Ho][Wo][C].  Uses an internal per-thread device scratch arena that grows on demand.
 * used_fallback (nullable) receives 1 when the near-zero branch (:231-239) fired. */
int attwarp_warp_image_host(const void* image_host, int img_dtype, int C, int H, int W,
                            const void* att_host, int att_dtype, int Wo, int Ho,
                            const attwarp_transform_params* tp, void* out_host,
                            int* used_fallback);

/* ---------------------------------------------------------------------------------------------
 * PNG encode of n uint8 images of any shapes in two launches (the warped images' way to disk;
 * the reference writes each with cv2.imwrite, AGW/new_method.py:491).
 *
 * images : HOST array of n descriptors; src is a DEVICE pointer to a dense [H][W][C] uint8 image,
 *          C = 1 (stored as grey), 3 (BGR, stored as RGB) or 4 (BGRA, stored as RGBA), as
 *          cv2.imwrite stores them.  src must stay valid until the stream has run the call.
 * Each file: signature, IHDR (bit depth 8, no interlace), IDAT chunks whose payloads are one zlib
 * stream (78 01, deflate, Adler-32), IEND.  Every row has the Sub filter; the stream is coded in
 * independent segments of 32 KiB (distance-1 matches under a dynamic Huffman code, or stored).
 * A file's bytes depend only on its image's pixels.  The bytes differ from cv2's encoder; the
 * decoded pixels are the same.
 * attwarp_png_max_bytes       : the largest file an H x W x C image can give (host arithmetic)
 * attwarp_png_workspace_bytes : device scratch one call over `images` needs
 * out      : device buffer of out_capacity >= sum over images of attwarp_png_max_bytes bytes;
 *            receives the files back to back
 * offsets  : device int64 [n + 1]: file i is out[offsets[i] .. offsets[i + 1])
 * The call uploads its descriptor table from host memory: ATTWARP_ERR_UNSUPPORTED on a stream
 * that is being captured into a CUDA graph.
 */
typedef struct attwarp_png_image {
    const void* src;
    int32_t H, W, C;
} attwarp_png_image;

size_t attwarp_png_max_bytes(int H, int W, int C);
size_t attwarp_png_workspace_bytes(const attwarp_png_image* images_host, int n);
int attwarp_encode_png(const attwarp_png_image* images_host, int n, void* workspace, size_t workspace_bytes,
                       void* out, size_t out_capacity, int64_t* offsets, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Attention overlay of n uint8 images of any sizes in two launches: the JET heat map blended
 * onto the image, the file save_warped_image writes as masked_overlay_save_path
 * (AGW/new_method.py, attwarp_b200/new_method.py:save_warped_image).  Bit-identical to that host
 * expression for a map `a` of the image's size:
 *   lo, hi = min(a), max(a)  (a NaN anywhere: both NaN)
 *   n = (a - lo) / (hi - lo) if hi > lo + 1e-9 else 0, in NumPy 2's precision for the dtype:
 *       uint8: a - lo in uint8, the rest in float64; float32: all float32; float64: all float64
 *   out = cv2.addWeighted(JET[uint8(n * 255)], alpha, base, 1 - alpha, 0)
 *
 * images   : HOST array of n descriptors; DEVICE pointers src (dense [H][W][C] uint8, C = 3 BGR
 *            or C = 1 grey, replicated to BGR), att and dst (dense [H][W][3] uint8 BGR, not src);
 *            any byte alignment.  1 <= H, W <= 65535.  They must stay valid until the stream has
 *            run the call.
 * att_kind : ATTWARP_OVERLAY_MAP    att is the image's own [H][W] map of att_dtype U8, F32 or F64
 *                                   (gh, gw ignored)
 *            ATTWARP_OVERLAY_TOKENS att is the image's [gh][gw] F32 token map, read at
 *                                   ((y * gh) / H, (x * gw) / W) (the index upsampling of
 *                                   attwarp_maps_from_tokens); lo and hi are taken over the tokens
 *                                   that rule reaches.  1 <= gh, gw <= 65535.
 * alpha    : finite; the weights are float(alpha) and float(1 - alpha), as cv2.addWeighted takes them
 * workspace: attwarp_overlay_workspace_bytes(images, n, att_kind) bytes of device scratch
 * The call uploads its descriptor table from host memory: ATTWARP_ERR_UNSUPPORTED on a stream
 * that is being captured into a CUDA graph.
 */
typedef enum attwarp_overlay_kind {
    ATTWARP_OVERLAY_MAP = 0,
    ATTWARP_OVERLAY_TOKENS = 1
} attwarp_overlay_kind;

typedef struct attwarp_overlay_image {
    const void* src;
    const void* att;
    void* dst;
    int32_t H, W, C;
} attwarp_overlay_image;

size_t attwarp_overlay_workspace_bytes(const attwarp_overlay_image* images_host, int n, int att_kind);
int attwarp_attention_overlay(const attwarp_overlay_image* images_host, int n, int att_dtype, int att_kind, int gh,
                              int gw, double alpha, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stages 2-3, torch path (all float32 [B][N] row-major unless noted).
 */
/* safe_softmax, dim=1 (mnfd/model.py:8-14). */
int attwarp_safe_softmax(const float* logits, int B, int N, float eps, float* out, void* stream);
/* safe_softmax (mnfd/model.py:8-14) followed by mix_with_uniform (model.py:98-101) in ONE launch -- what
 * MarginalNet.forward + trainer.py:212-214 compute back to back; alpha <= 0 is plain safe_softmax.  Bit-identical to
 * the two stand-alone entry points run in turn.  backward: grad_out [B][N] -> grad_logits [B][N]. */
int attwarp_safe_softmax_mix(const float* logits, int B, int N, float eps, float alpha, float* out, void* stream);
int attwarp_safe_softmax_mix_backward(const float* logits, const float* grad_out, int B, int N, float eps, float alpha,
                                      float* grad_logits, void* stream);
/* mix_with_uniform (mnfd/model.py:98-101): alpha<=0 copies. */
int attwarp_mix_with_uniform(const float* p, int B, int N, float alpha, float* out,
                             void* stream);
/* cdf_from_density (mnfd/checkpoint_utils.py:30-41). */
int attwarp_cdf_from_density(const float* p, int B, int N, float* F, void* stream);
/* _make_strictly_increasing (mnfd/checkpoint_utils.py:17-28): F [B][N] -> out [B][N]; and the row-wise
 * F.interpolate(mode='linear', align_corners=True) of resample_cdf (:53-62), F [B][N] -> out [B][L].
 * resample_cdf(F, L) = strictly_increasing(interp(strictly_increasing(F), L)). */
int attwarp_make_strictly_increasing(const float* F, int B, int N, float eps, float* out, void* stream);
int attwarp_interp_linear_rows(const float* F, int B, int N, int L, float* out, void* stream);
/* gt_marginals (mnfd/checkpoint_utils.py:43-51): A float32 [B][H][W] (the singleton channel is
 * dropped) -> px [B][W], py [B][H].  workspace: attwarp_maps_workspace_bytes(B,H,W). */
int attwarp_gt_marginals(const float* A, int B, int H, int W, void* workspace,
                         size_t workspace_bytes, float* px, float* py, void* stream);
/* upsample_pdf_right_inverse (mnfd/checkpoint_utils.py:64-131) as x = y * M^T with the
 * precomputed M = A^T (A A^T + eps I)^-1, float32 [L_in][L_out] row-major (depends only on
 * (L_in, L_out, eps); the host mirror builds and caches it).  y [B][L_out] -> x [B][L_in]. */
int attwarp_upsample_right_inverse(const float* y, const float* M, int B, int L_out, int L_in,
                                   float* x, void* stream);
/* Backward passes of the three helpers the reference trains through (mnfd/trainer.py:209-250: MarginalNet ->
 * safe_softmax (model.py:93-94) -> mix_with_uniform (:213-214) -> upsample_pdf_right_inverse (:217-218) -> loss);
 * what torch.autograd computes for the reference's own expressions.
 *   safe_softmax_backward            : logits, grad_out [B][N] -> grad_logits [B][N]
 *   mix_with_uniform_backward        : grad_out [B][N] -> grad_p = (1 - alpha) grad_out (alpha <= 0 copies)
 *   upsample_right_inverse_backward  : grad_x [B][L_in], M [L_in][L_out] -> grad_y = grad_x M  [B][L_out] */
int attwarp_safe_softmax_backward(const float* logits, const float* grad_out, int B, int N, float eps,
                                  float* grad_logits, void* stream);
int attwarp_mix_with_uniform_backward(const float* grad_out, int B, int N, float alpha, float* grad_p,
                                      void* stream);
int attwarp_upsample_right_inverse_backward(const float* grad_x, const float* M, int B, int L_out, int L_in,
                                            float* grad_y, void* stream);
/* The image-resolution PDF-L1 loss MarginalNet is trained with, forward and backward in one launch each
 * (mnfd/trainer.py:217-250):
 *     p_img = upsample_pdf_right_inverse(p_s, L).clamp_min(0);  p_img /= p_img.sum(1).clamp_min(1e-6)
 *     g_img = upsample_pdf_right_inverse(g,   L).clamp_min(0);  g_img /= g_img.sum(1).clamp_min(1e-6)
 *     loss  = F.l1_loss(px_img, gx_img) + F.l1_loss(py_img, gy_img)
 * px [B][Nx], py [B][Ny]: predicted PDFs (after mix_with_uniform); gx [B][Ngx], gy [B][Ngy]: gt_marginals of the
 * pooled attention; Mx [W][Nx], My [H][Ny], Mgx [W][Ngx], Mgy [H][Ngy]: right-inverse matrices.  The [B][L] rows
 * never reach global memory.  workspace: attwarp_pdf_l1_loss_workspace_bytes(B) bytes, ZEROED once by the caller
 * (the kernel leaves it ready for the next launch); loss: one float.
 * backward: upstream = d(objective)/d(loss), one float ON THE DEVICE; grad_px [B][Nx], grad_py [B][Ny] (the ground
 * truth carries no gradient). */
size_t attwarp_pdf_l1_loss_workspace_bytes(int B);
int attwarp_pdf_l1_loss(const float* px, const float* py, const float* gx, const float* gy, int B, int Nx, int Ny,
                        int Ngx, int Ngy, const float* Mx, const float* My, const float* Mgx, const float* Mgy, int W,
                        int H, void* workspace, size_t workspace_bytes, float* loss, void* stream);
int attwarp_pdf_l1_loss_backward(const float* px, const float* py, const float* gx, const float* gy, int B, int Nx,
                                 int Ny, int Ngx, int Ngy, const float* Mx, const float* My, const float* Mgx,
                                 const float* Mgy, int W, int H, const float* upstream, float* grad_px, float* grad_py,
                                 void* stream);
/* F.adaptive_avg_pool2d(A, (gh,gw)) (mnfd/trainer.py:197): A [B][H][W] -> out [B][gh][gw]. */
int attwarp_adaptive_avg_pool2d(const float* A, int B, int H, int W, int gh, int gw, float* out,
                                void* stream);
/* The trainer's prologue in one pass (mnfd/trainer.py:186-197): A.clamp_min(0), float32 sqrt for the samples
 * whose sqrt_mask byte is non-zero (device array [B]; "sqrt" vs "iden"/"none" transform of the sample), then
 * adaptive_avg_pool2d to (gh, gw).  The transformed full-resolution map is never written. */
int attwarp_pool_attention(const float* A, const unsigned char* sqrt_mask, int B, int H, int W, int gh, int gw,
                           float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ATTWARP_H_ */
