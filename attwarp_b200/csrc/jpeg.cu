// jpeg.cu -- baseline JPEG decode of a list of files of mixed sizes and samplings in seven launches, bit-identical to
// libjpeg-turbo as Pillow runs it (jpeg_decode.h).  Only the compressed bytes are on the device; each image is
// written to its caller's dense [H][W][3] BGR buffer.
//
//   jpeg_destuff_kernel  one CTA per file: Huffman decode tables; the scan de-stuffed (FF 00 -> FF, fill bytes and
//                        RSTn dropped) with block-wide prefix sums; RSTn numbering checked; the restart intervals
//                        cut into windows of kWinBits bits (every interval starts a window)
//   jpeg_sync_kernel     one thread per window, kChunk windows per CTA: self-synchronising decode (Weissenberger &
//                        Schmidt, ICPP 2018).  A window's entry state is the exit state of the window before it; a
//                        window that starts an interval knows its entry, the others start from a guess (window
//                        start, block 0, coefficient 0).  The CTA re-decodes the windows whose entry changed until
//                        no entry changes.  Run twice: the second pass starts each CTA's first window from the
//                        first pass's exit of the CTA before it (right unless that CTA never synchronised) and
//                        re-decodes only the windows before the trajectories meet.  The state is (bit position, block of the MCU, coefficient index):
//                        two decodes at the same bit position with a different block or coefficient index read the
//                        next bits differently, so a match on the position alone is not synchronisation.
//   jpeg_chain_kernel    one thread per file: the first window of each CTA takes the true exit of the window before
//                        it; windows are re-decoded until the new exit equals the one stored, after which the CTA's
//                        fixed point holds from the true entry
//   jpeg_scan_kernel     one CTA per file: prefix sums of the blocks and of the per-component DC differences each
//                        window starts, restarted at every interval; an interval with too few blocks fails
//   jpeg_blocks_kernel   one thread per window: decodes the blocks that start in it (DC value = prefix + the
//                        differences so far), dequantisation + ISLOW IDCT, 8 x 8 samples to the component plane
//   jpeg_color_kernel    one CTA per strip of kStripRows output rows: up-sampling + YCbCr -> BGR to the caller's buffer
#include <vector>

#include "common.cuh"
#include "jpeg_decode.h"

namespace aw {

namespace {

using namespace jpeg;

constexpr int kWinBits = 512;
constexpr int kChunk = 128;                      // windows per CTA of the sync and blocks kernels
constexpr int kDestuffThreads = 512;
constexpr int kDestuffPer = 16;                  // bytes per thread and tile
constexpr int kScanThreads = 256;
constexpr int kStripRows = 4;
constexpr int kColorThreads = 256;
constexpr uint64_t kErrCoef = kErrState - 1;     // an index past 63 (a distinct terminal state)

struct Win {
    uint64_t entry, exit;
    int32_t nblk, dc[kMaxComps];                 // blocks whose DC symbol lies in the window, their DC differences
    int32_t cum_blk, cum_dc[kMaxComps];          // inclusive prefix over the file's windows
};
static_assert(sizeof(Win) == 48, "window record layout");

struct JpegImage {
    Header h;
    const uint8_t* src;
    uint8_t* dst;
    uint8_t* scan;                               // de-stuffed entropy-coded data
    uint32_t* istart;                            // [n_intervals + 1] byte offsets of the intervals in `scan`
    int32_t* wbegin;                             // [n_intervals + 1] first window of each interval; [n] = windows
    Win* win;
    HuffDerived* tabs;                           // DC of component c at c, AC at kMaxComps + c
    uint8_t* plane[kMaxComps];
    int32_t chunk_begin, strip_begin;            // first CTA of the sync / blocks and of the colour kernels
};

__device__ __forceinline__ bool is_err(uint64_t s) { return s >= kErrCoef; }

__device__ uint64_t dstep(const ScanTables& t, const uint8_t* d, uint32_t end_byte, uint64_t s, bool* is_dc,
                          int* value, int* zz) {
    const uint64_t n = step(t, d, end_byte, s, is_dc, value, zz);
    if (n == kErrState && state_k(s) != 0) {
        // an AC symbol: tell a bad code from an index past 63
        const uint32_t v = peek32(d, state_pos(s), end_byte);
        int sym;
        if (huff_decode(t.ac[state_blk(s)], v, &sym) != 0) return kErrCoef;
    }
    return n;
}

__device__ void scan_tables(const JpegImage& J, ScanTables* t) {
    t->bpm = J.h.bpm;
    for (int b = 0; b < J.h.bpm; ++b) {
        t->dc[b] = J.tabs + J.h.blk_comp[b];
        t->ac[b] = J.tabs + kMaxComps + J.h.blk_comp[b];
    }
}

// interval of window w (last interval whose first window is <= w) and the window's bit range
struct WinGeom {
    int iv;
    uint32_t s, e, end_byte;
    bool first;
};
__device__ WinGeom win_geom(const JpegImage& J, int w) {
    int lo = 0, hi = J.h.n_intervals - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (J.wbegin[mid] <= w) lo = mid; else hi = mid - 1;
    }
    WinGeom g;
    g.iv = lo;
    const int j = w - J.wbegin[lo];
    g.end_byte = J.istart[lo + 1];
    g.s = J.istart[lo] * 8u + (uint32_t)j * kWinBits;
    g.e = min(g.s + (uint32_t)kWinBits, g.end_byte * 8u);
    g.first = j == 0;
    return g;
}

// Decode from `entry` until the first symbol boundary at or past bit e.  After an invalid code or an index past 63
// the decode goes on from (next bit, block 0, coefficient 0): a guessed entry that meets one keeps a trajectory that
// can still synchronise (an error state never would, and every window after it would wait for the true chain).  The
// exit stays a function of the entry alone; on the true trajectory the blocks kernel meets the same error and
// reports it.
__device__ uint64_t run_window(const JpegImage& J, const ScanTables& t, const WinGeom& g, uint64_t entry,
                               int32_t* nblk, int32_t* dc) {
    uint64_t s = entry;
    *nblk = 0;
    for (int c = 0; c < kMaxComps; ++c) dc[c] = 0;
    while (state_pos(s) < g.e) {
        const int comp = J.h.blk_comp[state_blk(s)];
        bool is_dc;
        int v, zz;
        const uint64_t nx = step(t, J.scan, g.end_byte, s, &is_dc, &v, &zz);
        if (nx == kErrState) {
            s = pack_state(state_pos(s) + 1, 0, 0);
            continue;
        }
        s = nx;
        if (is_dc) {
            ++*nblk;
            dc[comp] += v;
        }
    }
    return s;
}

__device__ int find_image(const JpegImage* imgs, int n, int cta, bool strips) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((strips ? imgs[mid].strip_begin : imgs[mid].chunk_begin) <= cta) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// exclusive block-wide prefix sum; *total receives the sum (blockDim.x a multiple of 32)
__device__ int block_excl_sum(int v, int* red, int* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
    }
    if (lane == 31) red[wid] = inc;
    __syncthreads();
    int ex = inc - v, tot = 0;
    for (int w = 0; w < nw; ++w) {
        if (w < wid) ex += red[w];
        tot += red[w];
    }
    __syncthreads();
    *total = tot;
    return ex;
}

// ---- kernel 1: one CTA per file ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(kDestuffThreads)
jpeg_destuff_kernel(const JpegImage* __restrict__ imgs, int32_t* __restrict__ status) {
    __shared__ int red[32];
    __shared__ int s_status;
    const JpegImage& J = imgs[blockIdx.x];
    const int tid = threadIdx.x;
    if (tid == 0) s_status = kStOk;
    if (tid < 2 * J.h.ncomp) {
        const int slot = tid < J.h.ncomp ? tid : kMaxComps + tid - J.h.ncomp;
        build_derived(J.h.hbits[slot], J.h.hval[slot], slot < kMaxComps, J.tabs + slot);
    }
    const uint8_t* raw = J.src + J.h.scan_off;
    const uint32_t len = J.h.scan_len;
    const int nint = J.h.n_intervals;
    uint32_t out_base = 0;
    int rst_base = 0;
    for (uint32_t base = 0; base < len; base += kDestuffThreads * kDestuffPer) {
        const uint32_t i0 = base + (uint32_t)tid * kDestuffPer, i1 = min(i0 + kDestuffPer, len);
        int keep = 0, rst = 0;
        for (uint32_t i = i0; i < i1; ++i) {
            const int b = raw[i], prev = i > 0 ? raw[i - 1] : 0, next = i + 1 < len ? raw[i + 1] : 0xFF;
            if (b == 0xFF) keep += next == 0x00;
            else if (prev == 0xFF) rst += b >= 0xD0 && b <= 0xD7;
            else ++keep;
        }
        int tk, tr;
        uint32_t o = out_base + (uint32_t)block_excl_sum(keep, red, &tk);
        int r = rst_base + block_excl_sum(rst, red, &tr);
        for (uint32_t i = i0; i < i1; ++i) {
            const int b = raw[i], prev = i > 0 ? raw[i - 1] : 0, next = i + 1 < len ? raw[i + 1] : 0xFF;
            if (b == 0xFF) {
                if (next == 0x00) J.scan[o++] = 0xFF;
            } else if (prev == 0xFF) {
                if (b >= 0xD0 && b <= 0xD7) {
                    if (r + 1 >= nint || (b - 0xD0) != (r & 7)) atomicMax(&s_status, kStRestart);
                    else J.istart[r + 1] = o;
                    ++r;
                } else if (b != 0x00) {
                    atomicMax(&s_status, kStMarker);
                }
            } else {
                J.scan[o++] = (uint8_t)b;
            }
        }
        out_base += (uint32_t)tk;
        rst_base += tr;
    }
    if (tid == 0) {
        if (rst_base != nint - 1) atomicMax(&s_status, kStRestart);
        J.istart[0] = 0;
        J.istart[nint] = out_base;
    }
    __syncthreads();
    if (s_status == kStOk) {
        int wbase = 0;
        for (int i0 = 0; i0 < nint; i0 += kDestuffThreads) {
            const int i = i0 + tid;
            int cnt = 0;
            if (i < nint) {
                const uint32_t bits = (J.istart[i + 1] - J.istart[i]) * 8u;
                cnt = max(1, (int)((bits + kWinBits - 1) / kWinBits));
            }
            int tot;
            const int ex = block_excl_sum(cnt, red, &tot);
            if (i < nint) J.wbegin[i] = wbase + ex;
            wbase += tot;
        }
        if (tid == 0) J.wbegin[nint] = wbase;
    }
    if (tid == 0) status[blockIdx.x] = s_status;
}

// ---- kernel 2: one thread per window ----------------------------------------------------------------------------
// second: false -- every window that does not start an interval starts from the guess (window start, block 0,
// coefficient 0); the CTA's last exit goes to chunk_exit.  true -- the CTA's first window starts from the first
// pass's last exit of the CTA before it, the others from their first-pass fixed point, so that only the windows
// before the two trajectories meet are decoded again.
__global__ void __launch_bounds__(kChunk)
jpeg_sync_kernel(const JpegImage* __restrict__ imgs, int n, const int32_t* __restrict__ status,
                 uint64_t* __restrict__ chunk_exit, bool second) {
    __shared__ uint64_t sx[kChunk];
    __shared__ int changed;
    const int img = find_image(imgs, n, blockIdx.x, false);
    const JpegImage& J = imgs[img];
    if (status[img] != kStOk) return;
    const int nwin = J.wbegin[J.h.n_intervals];
    const int c0 = (blockIdx.x - J.chunk_begin) * kChunk;
    if (c0 >= nwin) return;
    const int t = threadIdx.x, w = c0 + t;
    const bool active = w < nwin;
    ScanTables tb;
    scan_tables(J, &tb);
    WinGeom g{};
    if (active) g = win_geom(J, w);
    const bool fixed = !active || g.first || t == 0;
    uint64_t entry = active ? pack_state(g.s, 0, 0) : 0, exit = 0;
    int32_t nblk = 0, dc[kMaxComps] = {0, 0, 0};
    bool dirty = active;
    if (second && active) {
        const Win& r = J.win[w];
        entry = r.entry;
        exit = r.exit;
        nblk = r.nblk;
        for (int c = 0; c < kMaxComps; ++c) dc[c] = r.dc[c];
        dirty = false;
        if (t == 0 && !g.first) {
            entry = chunk_exit[blockIdx.x - 1];
            dirty = entry != r.entry;
        }
    }
    for (;;) {
        if (dirty) exit = run_window(J, tb, g, entry, &nblk, dc);
        dirty = false;
        if (t == 0) changed = 0;
        sx[t] = exit;
        __syncthreads();
        if (!fixed && sx[t - 1] != entry) {
            entry = sx[t - 1];
            dirty = true;
            changed = 1;
        }
        __syncthreads();
        const int again = changed;
        __syncthreads();
        if (!again) break;
    }
    if (active) {
        Win& r = J.win[w];
        r.entry = entry;
        r.exit = exit;
        r.nblk = nblk;
        for (int c = 0; c < kMaxComps; ++c) r.dc[c] = dc[c];
        if (!second && (t == kChunk - 1 || w == nwin - 1)) chunk_exit[blockIdx.x] = exit;
    }
}

// ---- kernel 3: one thread per file (after the second sync pass, usually one comparison per CTA) -----------------
__global__ void jpeg_chain_kernel(const JpegImage* __restrict__ imgs, int n, const int32_t* __restrict__ status) {
    const int img = blockIdx.x * blockDim.x + threadIdx.x;
    if (img >= n || status[img] != kStOk) return;
    const JpegImage& J = imgs[img];
    const int nwin = J.wbegin[J.h.n_intervals];
    ScanTables tb;
    scan_tables(J, &tb);
    int w = kChunk;
    while (w < nwin) {
        WinGeom g = win_geom(J, w);
        uint64_t ent = J.win[w - 1].exit;
        while (!g.first && ent != J.win[w].entry) {
            Win& r = J.win[w];
            int32_t nblk, dc[kMaxComps];
            r.entry = ent;
            ent = r.exit = run_window(J, tb, g, ent, &nblk, dc);
            r.nblk = nblk;
            for (int c = 0; c < kMaxComps; ++c) r.dc[c] = dc[c];
            if (++w >= nwin) break;
            g = win_geom(J, w);
        }
        w = (w / kChunk + 1) * kChunk;
    }
}

// ---- kernel 4: one CTA per file ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(kScanThreads)
jpeg_scan_kernel(const JpegImage* __restrict__ imgs, int32_t* __restrict__ status) {
    __shared__ int red[32];
    const JpegImage& J = imgs[blockIdx.x];
    if (status[blockIdx.x] != kStOk) return;
    const int tid = threadIdx.x;
    const int nwin = J.wbegin[J.h.n_intervals];
    int base[1 + kMaxComps] = {0, 0, 0, 0};
    for (int w0 = 0; w0 < nwin; w0 += kScanThreads) {
        const int w = w0 + tid;
        int v[1 + kMaxComps] = {0, 0, 0, 0};
        if (w < nwin) {
            v[0] = J.win[w].nblk;
            for (int c = 0; c < kMaxComps; ++c) v[1 + c] = J.win[w].dc[c];
        }
        for (int k = 0; k < 1 + kMaxComps; ++k) {
            int tot;
            const int ex = block_excl_sum(v[k], red, &tot);
            // DC sums wrap like the int accumulation they stand for; only differences of them are used
            const int inc = (int)((uint32_t)base[k] + (uint32_t)ex + (uint32_t)v[k]);
            if (w < nwin) {
                if (k == 0) J.win[w].cum_blk = inc; else J.win[w].cum_dc[k - 1] = inc;
            }
            base[k] = (int)((uint32_t)base[k] + (uint32_t)tot);
        }
    }
    __syncthreads();
    for (int i = tid; i < J.h.n_intervals; i += kScanThreads) {
        const int a = J.wbegin[i], b = J.wbegin[i + 1];
        const int before = a > 0 ? J.win[a - 1].cum_blk : 0;
        const int64_t have = (int64_t)J.win[b - 1].cum_blk - before;
        if (have < interval_mcus(J.h, i) * J.h.bpm) atomicMax(&status[blockIdx.x], kStShortData);
    }
}

// ---- kernel 5: one thread per window ----------------------------------------------------------------------------
__global__ void __launch_bounds__(kChunk)
jpeg_blocks_kernel(const JpegImage* __restrict__ imgs, int n, int32_t* __restrict__ status) {
    const int img = find_image(imgs, n, blockIdx.x, false);
    const JpegImage& J = imgs[img];
    if (status[img] >= kStRestart) return;       // no windows; an interval short of blocks may still hide a bad code
    const int nwin = J.wbegin[J.h.n_intervals];
    const int w = (blockIdx.x - J.chunk_begin) * kChunk + threadIdx.x;
    if (w >= nwin) return;
    ScanTables tb;
    scan_tables(J, &tb);
    const WinGeom g = win_geom(J, w);
    const Win& r = J.win[w];
    uint64_t s = r.entry;
    const int a = J.wbegin[g.iv];
    int64_t q = (int64_t)r.cum_blk - r.nblk - (a > 0 ? J.win[a - 1].cum_blk : 0);
    int pred[kMaxComps];
    for (int c = 0; c < kMaxComps; ++c)
        pred[c] = (int)((uint32_t)r.cum_dc[c] - (uint32_t)r.dc[c] - (a > 0 ? (uint32_t)J.win[a - 1].cum_dc[c] : 0u));
    const int64_t expected = interval_mcus(J.h, g.iv) * J.h.bpm;
    bool is_dc;
    int v, zz;
    while (!is_err(s) && state_k(s) != 0) s = dstep(tb, J.scan, g.end_byte, s, &is_dc, &v, &zz);   // the tail of
    if (is_err(s)) return;                                                                      // a block before
    while (q < expected && state_pos(s) < g.e) {
        int comp, brow, bcol;
        block_place(J.h, g.iv, q, &comp, &brow, &bcol);
        int16_t coef[64];
        for (int k = 0; k < 64; ++k) coef[k] = 0;
        do {
            s = dstep(tb, J.scan, g.end_byte, s, &is_dc, &v, &zz);
            if (is_err(s)) {
                atomicMax(&status[img], s == kErrCoef ? kStCoefOverflow : kStBadCode);
                return;
            }
            if (is_dc) {
                pred[comp] += v;
                coef[0] = (int16_t)pred[comp];
            } else if (zz) {
                coef[natural_order(zz)] = (int16_t)v;
            }
        } while (state_k(s) != 0);
        if (state_pos(s) > g.end_byte * 8u) {
            atomicMax(&status[img], kStShortData);
            return;
        }
        uint8_t px[64];
        idct_islow(coef, J.h.qt[comp], px);
        const int64_t stride = (int64_t)J.h.comp_bw[comp] * 8;
        uint8_t* o = J.plane[comp] + (int64_t)brow * 8 * stride + bcol * 8;
        for (int y = 0; y < 8; ++y) {
            uint2 row;
            row.x = px[8 * y] | px[8 * y + 1] << 8 | px[8 * y + 2] << 16 | (uint32_t)px[8 * y + 3] << 24;
            row.y = px[8 * y + 4] | px[8 * y + 5] << 8 | px[8 * y + 6] << 16 | (uint32_t)px[8 * y + 7] << 24;
            *reinterpret_cast<uint2*>(o + y * stride) = row;     // planes are 8-byte aligned, rows a multiple of 8
        }
        ++q;
    }
}

// ---- kernel 6: one CTA per strip of output rows -----------------------------------------------------------------
__global__ void __launch_bounds__(kColorThreads)
jpeg_color_kernel(const JpegImage* __restrict__ imgs, int n, const int32_t* __restrict__ status) {
    const int img = find_image(imgs, n, blockIdx.x, true);
    const JpegImage& J = imgs[img];
    if (status[img] != kStOk) return;
    const Header& h = J.h;
    const int y0 = (blockIdx.x - J.strip_begin) * kStripRows;
    const int rows = min(kStripRows, h.H - y0);
    const int64_t npx = (int64_t)rows * h.W;
    for (int64_t p = threadIdx.x; p < npx; p += blockDim.x) {
        const int y = y0 + (int)(p / h.W), x = (int)(p % h.W);
        uint8_t* o = J.dst + ((int64_t)y * h.W + x) * 3;
        int v[kMaxComps];
        for (int c = 0; c < h.ncomp; ++c)
            v[c] = upsample_at(J.plane[c], h.comp_bw[c] * 8, h.comp_dw[c], h.comp_dh[c], h.comp_up[c], h.comp_hf[c],
                               h.comp_vf[c], x, y);
        if (h.ncomp == 1) {
            o[0] = o[1] = o[2] = (uint8_t)v[0];
        } else {
            uint8_t bgr[3];
            ycc_to_bgr(v[0], v[1], v[2], bgr);
            o[0] = bgr[0];
            o[1] = bgr[1];
            o[2] = bgr[2];
        }
    }
}

// ---- workspace layout -------------------------------------------------------------------------------------------
struct Layout {
    size_t tabs, scan, istart, wbegin, win, plane[kMaxComps], end;
    int64_t max_windows;
};

Layout layout_of(const Header& h, size_t at) {
    Layout L;
    L.max_windows = ((int64_t)h.scan_len * 8 + kWinBits - 1) / kWinBits + h.n_intervals;
    L.tabs = at;
    at = align_up(at + sizeof(HuffDerived) * 2 * kMaxComps, 16);
    L.scan = at;
    at = align_up(at + h.scan_len + 8, 16);
    L.istart = at;
    at = align_up(at + sizeof(uint32_t) * (size_t)(h.n_intervals + 1), 16);
    L.wbegin = at;
    at = align_up(at + sizeof(int32_t) * (size_t)(h.n_intervals + 1), 16);
    L.win = at;
    at = align_up(at + sizeof(Win) * (size_t)L.max_windows, 16);
    for (int c = 0; c < kMaxComps; ++c) {
        L.plane[c] = at;
        if (c < h.ncomp) at = align_up(at + (size_t)h.comp_bw[c] * 8 * h.comp_bh[c] * 8, 16);
    }
    L.end = at;
    return L;
}

size_t table_bytes(int n) { return align_up(sizeof(JpegImage) * (size_t)n, 256); }
int64_t chunks_of(const Header& h) { return (layout_of(h, 0).max_windows + kChunk - 1) / kChunk; }

}  // namespace

size_t jpeg_workspace_bytes_impl(const Header* headers, int n) {
    size_t at = table_bytes(n);
    int64_t chunks = 0;
    for (int i = 0; i < n; ++i) {
        at = layout_of(headers[i], at).end;
        chunks += chunks_of(headers[i]);
    }
    return at + sizeof(uint64_t) * (size_t)chunks;
}

// headers: the parsed, device-decodable files of images (validated by the caller); ws of
// jpeg_workspace_bytes_impl(headers, n) bytes
int launch_decode_jpeg(const attwarp_jpeg_image* images, const Header* headers, int n, void* ws, int32_t* status,
                       cudaStream_t st) {
    static thread_local std::vector<JpegImage> host;
    host.assign((size_t)n, JpegImage{});
    char* base = static_cast<char*>(ws);
    size_t at = table_bytes(n);
    int64_t chunks = 0, strips = 0;
    for (int i = 0; i < n; ++i) {
        const Header& h = headers[i];
        const Layout L = layout_of(h, at);
        at = L.end;
        JpegImage& J = host[(size_t)i];
        J.h = h;
        J.src = static_cast<const uint8_t*>(images[i].dev);
        J.dst = static_cast<uint8_t*>(images[i].dst);
        J.tabs = reinterpret_cast<HuffDerived*>(base + L.tabs);
        J.scan = reinterpret_cast<uint8_t*>(base + L.scan);
        J.istart = reinterpret_cast<uint32_t*>(base + L.istart);
        J.wbegin = reinterpret_cast<int32_t*>(base + L.wbegin);
        J.win = reinterpret_cast<Win*>(base + L.win);
        for (int c = 0; c < kMaxComps; ++c) J.plane[c] = reinterpret_cast<uint8_t*>(base + L.plane[c]);
        J.chunk_begin = (int32_t)chunks;
        J.strip_begin = (int32_t)strips;
        chunks += chunks_of(h);
        strips += (h.H + kStripRows - 1) / kStripRows;
        if (chunks > INT32_MAX || strips > INT32_MAX)
            return fail(ATTWARP_ERR_UNSUPPORTED, "decode_jpeg: the list is too large for one call");
    }
    JpegImage* d_table = reinterpret_cast<JpegImage*>(base);
    uint64_t* d_chunk_exit = reinterpret_cast<uint64_t*>(base + at);
    AW_CUDA(cudaMemcpyAsync(d_table, host.data(), sizeof(JpegImage) * (size_t)n, cudaMemcpyHostToDevice, st));
    jpeg_destuff_kernel<<<n, kDestuffThreads, 0, st>>>(d_table, status);
    int rc = check_launch("jpeg_destuff_kernel");
    if (rc != ATTWARP_OK) return rc;
    for (int second = 0; second < 2; ++second) {
        jpeg_sync_kernel<<<(unsigned)chunks, kChunk, 0, st>>>(d_table, n, status, d_chunk_exit, second != 0);
        if ((rc = check_launch("jpeg_sync_kernel")) != ATTWARP_OK) return rc;
    }
    jpeg_chain_kernel<<<(n + 63) / 64, 64, 0, st>>>(d_table, n, status);
    if ((rc = check_launch("jpeg_chain_kernel")) != ATTWARP_OK) return rc;
    jpeg_scan_kernel<<<n, kScanThreads, 0, st>>>(d_table, status);
    if ((rc = check_launch("jpeg_scan_kernel")) != ATTWARP_OK) return rc;
    jpeg_blocks_kernel<<<(unsigned)chunks, kChunk, 0, st>>>(d_table, n, status);
    if ((rc = check_launch("jpeg_blocks_kernel")) != ATTWARP_OK) return rc;
    jpeg_color_kernel<<<(unsigned)strips, kColorThreads, 0, st>>>(d_table, n, status);
    return check_launch("jpeg_color_kernel");
}

}  // namespace aw
