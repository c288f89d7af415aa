// png.cu -- PNG encode of a batch of uint8 images of mixed shapes in two launches.
//
// The file of one image is the signature, IHDR, one IDAT chunk holding the zlib header (78 01), one IDAT chunk per
// segment, one IDAT chunk holding the Adler-32, IEND.  The zlib stream is the image's filtered scanlines (filter
// byte 1 = Sub, then p[i] - p[i-C] in file channel order: RGB(A) for BGR(A) input, as cv2.imwrite stores it) cut
// into segments of at most kSegBytes.  Each segment is one deflate block on its own -- greedy distance-1 matches
// (run-length coding, what zlib's Z_RLE strategy emits) under a dynamic Huffman code fitted to the segment, or a
// stored block when that is not smaller -- ended by a sync flush (an empty stored block) so that it is byte
// aligned; the image's last segment carries BFINAL instead.  The bytes of a file depend only on its pixels.
//
//   png_segment_kernel   one CTA per segment of every image: filter, tokenise, Huffman code, pack, Adler-32 of the
//                        raw segment, CRC-32 of its IDAT chunk -> a worst-case-sized slot of the workspace
//   png_assemble_kernel  one CTA per image: file offset (sum of the sizes of the files before it), chunk headers,
//                        CRCs and the combined Adler-32, segment bytes copied to the contiguous output
#include <vector>

#include "common.cuh"
#include "png_deflate.h"

namespace aw {

namespace {

constexpr int kSegBytes = 32768;               // raw bytes per segment (a stored block holds up to 65535)
constexpr int kSlotBytes = kSegBytes + 16;     // a segment's worst case (stored: 5 + kSegBytes), 16-byte multiple
constexpr int kSegThreads = 256;
constexpr int kAsmThreads = 256;
constexpr int kFileOverhead = 8 + 25 + 14 + 16 + 12;   // signature, IHDR, zlib header chunk, Adler chunk, IEND
constexpr int kChunkOverhead = 12;             // length, type, CRC
constexpr uint32_t kAdlerMod = 65521;

// one image of the batch (device table; entry n is a sentinel whose seg_begin is the total segment count)
struct PngImage {
    const uint8_t* src;
    int64_t stream_bytes;                      // H * (1 + W * C): filtered scanlines
    int32_t H, W, C, seg_begin;
};
static_assert(sizeof(PngImage) == 32, "descriptor layout");

struct PngSegment {
    uint32_t bytes;                            // deflate bytes in the slot
    uint32_t crc;                              // CRC-32 of "IDAT" + those bytes
    uint32_t adler_a, adler_b;                 // sum b_k and sum (len - k) b_k of the raw segment, mod 65521
    uint32_t len;                              // raw bytes
    uint32_t pad[3];
};

size_t seg_count(int64_t stream_bytes) { return (size_t)((stream_bytes + kSegBytes - 1) / kSegBytes); }
int64_t stream_bytes_of(int H, int W, int C) { return (int64_t)H * (1 + (int64_t)W * C); }

size_t table_bytes(int n) { return align_up(sizeof(PngImage) * (size_t)(n + 1), 256); }
size_t results_bytes(size_t segs) { return align_up(sizeof(PngSegment) * segs, 256); }

__device__ __forceinline__ void store_be32(uint8_t* p, uint32_t v) {
    p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}

// ---- block scans over one value per thread (deterministic) -------------------------------------------------------
// max over the threads before this one (-1 if none)
__device__ int block_prev_max(int v, int* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc = max(inc, up);
    }
    int ex = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) ex = -1;
    if (lane == 31) red[wid] = inc;
    __syncthreads();
    for (int w = 0; w < wid; ++w) ex = max(ex, red[w]);
    __syncthreads();
    return ex;
}
// min over the threads after this one (`none` if none)
__device__ int block_next_min(int v, int none, int* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int dn = __shfl_down_sync(0xffffffffu, inc, o);
        if (lane + o < 32) inc = min(inc, dn);
    }
    int ex = __shfl_down_sync(0xffffffffu, inc, 1);
    if (lane == 31) ex = none;
    if (lane == 0) red[wid] = inc;
    __syncthreads();
    for (int w = wid + 1; w < nw; ++w) ex = min(ex, red[w]);
    __syncthreads();
    return ex;
}
// exclusive prefix sum; *total receives the block's sum
template <typename T>
__device__ T block_prev_sum(T v, T* red, T* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
    }
    if (lane == 31) red[wid] = inc;
    __syncthreads();
    T ex = inc - v, tot = 0;
    for (int w = 0; w < nw; ++w) {
        if (w < wid) ex += red[w];
        tot += red[w];
    }
    __syncthreads();
    *total = tot;
    return ex;
}

// ---- kernel 1: one CTA per segment -------------------------------------------------------------------------------
__global__ void __launch_bounds__(kSegThreads, 3)
png_segment_kernel(const PngImage* __restrict__ imgs, int n, PngSegment* __restrict__ res, uint8_t* __restrict__ slots) {
    extern __shared__ uint4 png_smem[];
    uint8_t* in = reinterpret_cast<uint8_t*>(png_smem);                       // the filtered segment
    uint32_t* obuf = reinterpret_cast<uint32_t*>(in + kSegBytes);             // the deflate bytes, as words
    uint8_t* obytes = reinterpret_cast<uint8_t*>(obuf);
    __shared__ uint32_t hist[png::kLitLenSymbols], work[png::kLitLenSymbols], crc_tab[256];
    __shared__ uint16_t sorted[png::kLitLenSymbols], codes[png::kLitLenSymbols];
    __shared__ uint8_t lens[png::kLitLenSymbols];
    __shared__ int ired[32];
    __shared__ unsigned long long lred[32];
    __shared__ uint32_t crc_op[6], wcrc[32];
    __shared__ int s_m, s_hdr_bits;

    const int tid = threadIdx.x, nt = blockDim.x;
    const int seg = blockIdx.x;
    int lo = 0, hi = n - 1;                    // the image: last entry with seg_begin <= seg
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (imgs[mid].seg_begin <= seg) lo = mid; else hi = mid - 1;
    }
    const PngImage im = imgs[lo];
    const int64_t q0 = (int64_t)(seg - im.seg_begin) * kSegBytes;
    const int len = (int)min((int64_t)kSegBytes, im.stream_bytes - q0);
    const bool last = q0 + len == im.stream_bytes;
    const int C = im.C, rowb = 1 + im.W * C;

    // load + Sub filter, zero the output words, CRC table
    for (int i = tid; i < png::kLitLenSymbols; i += nt) hist[i] = 0;
    if (tid == 0) s_m = 0;
    for (int i = tid; i < kSlotBytes / 4; i += nt) obuf[i] = 0;
    if (tid < 256) {
        uint32_t c = (uint32_t)tid;
        for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ png::kCrcPoly : c >> 1;
        crc_tab[tid] = c;
    }
    {
        const int64_t r0 = q0 / rowb;
        const int c0 = (int)(q0 - r0 * rowb);
        for (int i = tid; i < len; i += nt) {
            const int cc = c0 + i, dr = cc / rowb, c = cc - dr * rowb;
            uint8_t v = 1;
            if (c != 0) {
                const int x = c - 1, px = x / C, ch = x - px * C;
                const int mch = (C >= 3 && ch < 3) ? 2 - ch : ch;          // file order RGB(A) <- BGR(A)
                const uint8_t* p = im.src + ((r0 + dr) * im.W + px) * (int64_t)C + mch;
                v = (uint8_t)(__ldg(p) - (px > 0 ? __ldg(p - C) : 0));
            }
            in[i] = v;
        }
    }
    __syncthreads();

    // this thread's chunk: Adler-32 sums and the run breaks at its ends
    const int per = (len + nt - 1) / nt;
    const int a = min(tid * per, len), b = min(a + per, len);
    uint32_t sa = 0;
    unsigned long long sb = 0;
    int first_brk = len, last_brk = -1;
    for (int i = a; i < b; ++i) {
        const uint32_t v = in[i];
        sa += v;
        sb += (unsigned long long)(len - i) * v;
        if (i == 0 || in[i] != in[i - 1]) {
            first_brk = min(first_brk, i);
            last_brk = i;
        }
    }
    const int prev_brk = block_prev_max(last_brk, ired);
    const int next_brk = block_next_min(first_brk, len, ired);
    unsigned long long tot;
    block_prev_sum<unsigned long long>(sa, lred, &tot);
    const uint32_t adler_a = (uint32_t)(tot % kAdlerMod);
    block_prev_sum<unsigned long long>(sb, lred, &tot);
    const uint32_t adler_b = (uint32_t)(tot % kAdlerMod);

    // literal/length histogram
    png::rle_tokens(in, len, a, b, prev_brk, next_brk, [&](int lit, int mlen) {
        int sym = lit, extra, nextra;
        if (lit < 0) png::length_symbol(mlen, sym, extra, nextra);
        atomicAdd(&hist[sym], 1u);
    });
    __syncthreads();
    if (tid == 0) hist[256] = 1;
    __syncthreads();
    // symbols in ascending (count, symbol) order, ranked in parallel
    {
        int used = 0;                          // symbols this thread ranked (at most two)
        for (int s = tid; s < png::kLitLenSymbols; s += nt) {
            const uint32_t f = hist[s];
            if (f == 0) continue;
            ++used;
            int rank = 0;
            for (int t = 0; t < png::kLitLenSymbols; ++t) {
                const uint32_t g = hist[t];
                rank += g != 0 && (g < f || (g == f && t < s));
            }
            sorted[rank] = (uint16_t)s;
        }
        if (used) atomicAdd(&s_m, used);
    }
    __syncthreads();
    if (tid == 0) {
        const int m = s_m;
        png::huff_lengths_sorted(hist, sorted, m, png::kLitLenSymbols, png::kMaxBits, lens, work);
        png::huff_codes(lens, png::kLitLenSymbols, codes);
        const uint8_t d_lens[2] = {1, 1};    // distance 1 only: code 0 (a second code keeps the code complete)
        png::BitWriter bw{obytes, 0, 0, 0};
        png::write_dynamic_header(bw, last ? 1 : 0, lens, d_lens, 2);
        bw.flush_partial();
        s_hdr_bits = bw.bits();
    }
    __syncthreads();

    // bit offsets of this thread's tokens
    auto token_code = [&](int lit, int mlen, uint32_t& v, int& nb) {
        if (lit >= 0) {
            v = codes[lit];
            nb = lens[lit];
        } else {
            int sym, extra, nextra;
            png::length_symbol(mlen, sym, extra, nextra);
            v = codes[sym] | ((uint32_t)extra << lens[sym]);
            nb = lens[sym] + nextra + 1;       // + distance code 0, one 0 bit
        }
    };
    int my_bits = 0;
    png::rle_tokens(in, len, a, b, prev_brk, next_brk, [&](int lit, int mlen) {
        uint32_t v;
        int nb;
        token_code(lit, mlen, v, nb);
        my_bits += nb;
    });
    int token_bits;
    const int my_off = block_prev_sum<int>(my_bits, ired, &token_bits);
    const int hdr_bits = s_hdr_bits;
    const int bits = hdr_bits + token_bits + lens[256];
    const int comp_bytes = last ? (bits + 7) / 8 : (bits + 3 + 7) / 8 + 4;
    const bool stored = comp_bytes >= 5 + len;
    int nbytes;
    if (!stored) {
        int pos = hdr_bits + my_off;
        png::rle_tokens(in, len, a, b, prev_brk, next_brk, [&](int lit, int mlen) {
            uint32_t v;
            int nb;
            token_code(lit, mlen, v, nb);
            const int w = pos >> 5, sh = pos & 31;
            atomicOr(&obuf[w], v << sh);
            if (sh + nb > 32) atomicOr(&obuf[w + 1], v >> (32 - sh));
            pos += nb;
        });
        if (tid == 0) {
            const int pos_eob = hdr_bits + token_bits, w = pos_eob >> 5, sh = pos_eob & 31;
            atomicOr(&obuf[w], (uint32_t)codes[256] << sh);
            if (sh + lens[256] > 32) atomicOr(&obuf[w + 1], (uint32_t)codes[256] >> (32 - sh));
        }
        __syncthreads();
        if (!last && tid == 0) {               // sync flush: empty stored block 000, pad, 00 00 FF FF
            const int p = (bits + 3 + 7) / 8;
            obytes[p + 2] = 0xFF;
            obytes[p + 3] = 0xFF;
        }
        nbytes = comp_bytes;
    } else {
        for (int i = tid; i < len; i += nt) obytes[5 + i] = in[i];
        if (tid == 0) {
            obytes[0] = last ? 1 : 0;          // BFINAL, BTYPE = 00
            obytes[1] = (uint8_t)len;
            obytes[2] = (uint8_t)(len >> 8);
            obytes[3] = (uint8_t)~len;
            obytes[4] = (uint8_t)(~len >> 8);
        }
        nbytes = 5 + len;
    }
    __syncthreads();

    // CRC-32 of "IDAT" + the bytes: equal chunks per thread, the short one first, combined as a tree
    const int N = 4 + nbytes, L = (N + nt - 1) / nt;
    if (tid < 6) crc_op[tid] = png::crc_shift_operator((uint64_t)L << tid);
    {
        const int end = N - (nt - 1 - tid) * L, beg = max(end - L, 0);
        uint32_t crc = 0xFFFFFFFFu;
        for (int j = beg; j < end; ++j) {
            const uint8_t byte = j < 4 ? (uint8_t)("IDAT"[j]) : obytes[j - 4];
            crc = crc_tab[(crc ^ byte) & 0xFF] ^ (crc >> 8);
        }
        crc = ~crc;                            // 0 for an empty chunk
        __syncthreads();
        const int lane = tid & 31;
#pragma unroll
        for (int s = 0; s < 5; ++s) {          // a right half of 2^s full chunks, or an empty left half
            const uint32_t other = __shfl_down_sync(0xffffffffu, crc, 1 << s);
            if ((lane & ((2 << s) - 1)) == 0) crc = png::crc_combine(crc, other, crc_op[s]);
        }
        if (lane == 0) wcrc[tid >> 5] = crc;
    }
    // copy out
    {
        const uint4* s4 = reinterpret_cast<const uint4*>(obuf);
        uint4* d4 = reinterpret_cast<uint4*>(slots + (size_t)seg * kSlotBytes);
        for (int i = tid; i < (nbytes + 15) / 16; i += nt) d4[i] = s4[i];
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t crc = wcrc[0];
        for (int w = 1; w < nt / 32; ++w) crc = png::crc_combine(crc, wcrc[w], crc_op[5]);
        PngSegment r;
        r.bytes = (uint32_t)nbytes;
        r.crc = crc;
        r.adler_a = adler_a;
        r.adler_b = adler_b;
        r.len = (uint32_t)len;
        r.pad[0] = r.pad[1] = r.pad[2] = 0;
        res[seg] = r;
    }
}

// ---- kernel 2: one CTA per image ---------------------------------------------------------------------------------
__device__ uint32_t small_crc(const uint8_t* p, int n) { return ~png::crc_update_bitwise(0xFFFFFFFFu, p, n); }

__global__ void __launch_bounds__(kAsmThreads)
png_assemble_kernel(const PngImage* __restrict__ imgs, int n, const PngSegment* __restrict__ res,
                    const uint8_t* __restrict__ slots, uint8_t* __restrict__ out, int64_t* __restrict__ offsets) {
    __shared__ unsigned long long lred[32];
    __shared__ int64_t s_off[kAsmThreads];
    __shared__ uint32_t s_adler_a, s_adler_b;
    const int tid = threadIdx.x, nt = blockDim.x, img = blockIdx.x;
    const PngImage im = imgs[img];
    const int sb = im.seg_begin, se = imgs[img + 1].seg_begin;
    // file offset: the files of the images before this one
    unsigned long long before = 0, mine = 0;
    for (int s = tid; s < se; s += nt) {
        const unsigned long long v = kChunkOverhead + res[s].bytes;
        if (s < sb) before += v; else mine += v;
    }
    unsigned long long tot;
    block_prev_sum<unsigned long long>(before, lred, &tot);
    const int64_t off = (int64_t)tot + (int64_t)kFileOverhead * img;
    block_prev_sum<unsigned long long>(mine, lred, &tot);
    const int64_t size = (int64_t)tot + kFileOverhead;
    uint8_t* f = out + off;
    if (tid == 0) {
        const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1A, '\n'};
        for (int k = 0; k < 8; ++k) f[k] = sig[k];
        uint8_t ihdr[17] = {'I', 'H', 'D', 'R'};
        store_be32(ihdr + 4, (uint32_t)im.W);
        store_be32(ihdr + 8, (uint32_t)im.H);
        ihdr[12] = 8;                                               // bit depth
        ihdr[13] = im.C == 1 ? 0 : (im.C == 3 ? 2 : 6);             // grey, RGB, RGBA
        ihdr[14] = ihdr[15] = ihdr[16] = 0;                         // deflate, adaptive filters, no interlace
        store_be32(f + 8, 13);
        for (int k = 0; k < 17; ++k) f[12 + k] = ihdr[k];
        store_be32(f + 29, small_crc(ihdr, 17));
        const uint8_t zh[6] = {'I', 'D', 'A', 'T', 0x78, 0x01};
        store_be32(f + 33, 2);
        for (int k = 0; k < 6; ++k) f[37 + k] = zh[k];
        store_be32(f + 43, small_crc(zh, 6));
        s_adler_a = 1;
        s_adler_b = 0;
    }
    // segment chunks, kAsmThreads segments at a time
    int64_t pos = off + 47;
    for (int base = sb; base < se; base += nt) {
        const int s = base + tid;
        const unsigned long long v = s < se ? kChunkOverhead + res[s].bytes : 0;
        const unsigned long long rel = block_prev_sum<unsigned long long>(v, lred, &tot);
        s_off[tid] = pos + (int64_t)rel;
        __syncthreads();
        if (tid == 0) {                                             // Adler-32 of the stream so far
            uint32_t aa = s_adler_a, bb = s_adler_b;
            for (int k = base; k < min(base + nt, se); ++k) {
                const PngSegment& r = res[k];
                bb = (uint32_t)(((uint64_t)bb + (uint64_t)aa * r.len + r.adler_b) % kAdlerMod);
                aa = (aa + r.adler_a) % kAdlerMod;
            }
            s_adler_a = aa;
            s_adler_b = bb;
        }
        for (int k = base; k < min(base + nt, se); ++k) {
            const PngSegment r = res[k];
            uint8_t* c = out + s_off[k - base];
            const uint8_t* src = slots + (size_t)k * kSlotBytes;
            if (tid == 0) {
                store_be32(c, r.bytes);
                c[4] = 'I'; c[5] = 'D'; c[6] = 'A'; c[7] = 'T';
                store_be32(c + 8 + r.bytes, r.crc);
            }
            for (uint32_t i = tid; i < r.bytes; i += nt) c[8 + i] = src[i];
        }
        pos += (int64_t)tot;
        __syncthreads();
    }
    if (tid == 0) {
        uint8_t* t = out + pos;
        uint8_t ad[8] = {'I', 'D', 'A', 'T'};
        store_be32(ad + 4, (s_adler_b << 16) | s_adler_a);
        store_be32(t, 4);
        for (int k = 0; k < 8; ++k) t[4 + k] = ad[k];
        store_be32(t + 12, small_crc(ad, 8));
        const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
        for (int k = 0; k < 12; ++k) t[16 + k] = iend[k];
        offsets[img] = off;
        if (img == n - 1) offsets[n] = off + size;
    }
}

}  // namespace

size_t png_max_bytes_impl(int H, int W, int C) {
    const int64_t S = stream_bytes_of(H, W, C);
    return (size_t)S + (size_t)(kChunkOverhead + 5) * seg_count(S) + kFileOverhead;
}

size_t png_workspace_bytes_impl(const attwarp_png_image* images, int n) {
    size_t segs = 0;
    for (int i = 0; i < n; ++i) segs += seg_count(stream_bytes_of(images[i].H, images[i].W, images[i].C));
    return table_bytes(n) + results_bytes(segs) + segs * kSlotBytes;
}

// images: validated by the caller; ws of png_workspace_bytes_impl(images, n) bytes
int launch_encode_png(const attwarp_png_image* images, int n, void* ws, uint8_t* out, int64_t* offsets,
                      cudaStream_t st) {
    static thread_local std::vector<PngImage> host;
    host.assign((size_t)n + 1, PngImage{});
    int64_t segs = 0;
    for (int i = 0; i < n; ++i) {
        PngImage& r = host[(size_t)i];
        r.src = static_cast<const uint8_t*>(images[i].src);
        r.H = images[i].H;
        r.W = images[i].W;
        r.C = images[i].C;
        r.stream_bytes = stream_bytes_of(r.H, r.W, r.C);
        r.seg_begin = (int32_t)segs;
        segs += (int64_t)seg_count(r.stream_bytes);
    }
    if (segs > INT32_MAX) return fail(ATTWARP_ERR_UNSUPPORTED, "encode_png: %lld segments in one call", (long long)segs);
    host[(size_t)n].seg_begin = (int32_t)segs;
    char* p = static_cast<char*>(ws);
    PngImage* d_table = reinterpret_cast<PngImage*>(p);
    PngSegment* d_res = reinterpret_cast<PngSegment*>(p + table_bytes(n));
    uint8_t* d_slots = reinterpret_cast<uint8_t*>(p + table_bytes(n) + results_bytes((size_t)segs));
    AW_CUDA(cudaMemcpyAsync(d_table, host.data(), sizeof(PngImage) * (size_t)(n + 1), cudaMemcpyHostToDevice, st));
    const size_t smem = kSegBytes + kSlotBytes;
    static thread_local int smem_set_dev = -1;
    int dev = 0;
    AW_CUDA(cudaGetDevice(&dev));
    if (smem_set_dev != dev) {
        AW_CUDA(cudaFuncSetAttribute(png_segment_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set_dev = dev;
    }
    png_segment_kernel<<<(unsigned)segs, kSegThreads, smem, st>>>(d_table, n, d_res, d_slots);
    int rc = check_launch("png_segment_kernel");
    if (rc != ATTWARP_OK) return rc;
    png_assemble_kernel<<<n, kAsmThreads, 0, st>>>(d_table, n, d_res, d_slots, out, offsets);
    return check_launch("png_assemble_kernel");
}

}  // namespace aw
