// png_decode.cu -- PNG decode of a list of files of mixed sizes in one launch, pixel for pixel as Pillow's
// Image.open(f).convert('RGB') gives them, written as BGR to each caller's dense [H][W][3] buffer.  Only the file
// bytes are on the device.
//
// png_decode_kernel is persistent: a fixed grid of CTAs takes whole files, biggest first, by an atomic ticket, and
// no CTA waits on another.  A file goes through these steps inside its CTA:
//   1. IDAT payloads gathered into one contiguous zlib stream; each chunk's CRC-32 checked: chunks of at most
//      kCrcSerial bytes a thread each, larger ones split across the CTA and folded with crc_combine.
//   2. Block loop.  One thread reads the block header at the known start bit and the Huffman tables are built in
//      shared memory; stored blocks are copied.  A Huffman block is cut into windows of kWinBits bits, one per
//      thread, decoded speculatively (png_inflate.h run_window: the state is the bit position at a token boundary).
//      The first window knows its entry; the others start at their first bit.  Windows whose entry changed (the
//      exit of the window before) are re-decoded until no entry changes; then every window holds its true
//      trajectory.  The first end-of-block ends the block and the windows past it are dropped; when the set of
//      kThreads windows ends before it, the next set starts from the true exit.
//   3. Byte counts of the windows, prefix-summed, give each window's output offset.
//   4. LZ77 resolution, kSeg output bytes at a time in output order.  Each window writes, for the bytes of the
//      segment its tokens produce, the literal or the position it copies from: for a match of distance d starting
//      at s, byte p copies s - d + ((p - s) mod d), so a run (d < length) points before its own start and long
//      d = 1 runs take log rounds.  Pointer jumping in the per-CTA scratch resolves every byte to a literal or to
//      a byte before the segment, which is final.  Adler-32 of the stream is folded segment by segment.
//   5. Adler-32 and the amount of data checked; filter types checked; rows unfiltered in a wavefront (row r is at
//      chunk c at step r + c, so Up, Avg and Paeth read finished bytes of the row above); then bit unpacking, the
//      palette, alpha dropping and RGB -> BGR into the caller's buffer.
// A file that fails a check gets a status code and its buffer is not written.
#include <algorithm>
#include <numeric>
#include <vector>

#include "common.cuh"
#include "png_inflate.h"

namespace aw {

namespace {

using namespace png;

constexpr int kThreads = 256;                    // a power of two: the split CRC folds as a tree (Shared::crc_op)
constexpr int kWinBits = 512;
constexpr int kSeg = 1 << 16;                    // output bytes resolved at a time (int32 scratch per CTA)
constexpr int kRing = 1 << 17;                   // >= kSeg + 32768: output past the image's rows (still Adler-summed)
constexpr int kCtasPerSm = 2;
constexpr int kPad = 1024;                       // zeros after a stream: the longest read past its end (a dynamic
                                                 // header that runs off it) stays inside
constexpr int kMinRowChunk = 16;                 // unfilter wavefront: bytes of a row a thread takes per step
constexpr uint32_t kCrcSerial = 16384;           // IDAT chunks up to this many bytes get their CRC from one thread
constexpr int32_t kWindow = 32768;               // deflate's largest distance

struct PngFile {
    const uint8_t* src;                          // the whole file
    uint8_t* dst;                                // [H][W][3] BGR
    uint8_t* stream;                             // the zlib stream, 8-byte aligned, then kPad zero bytes
    uint8_t* out;                                // [filtered] inflated rows
    const uint4* chunks;                         // per IDAT chunk: file offset of its data, length, stream offset
    int64_t filtered, row_bytes;
    uint64_t stream_bytes;
    int32_t H, W, colour, depth, bpp, nchunks;
    uint32_t plte_off, plte_entries;
};

struct Shared {
    Huff lt, dt;
    uint32_t crc[256];
    uint64_t exit[kThreads];                     // window exits of the current set
    int64_t off[kThreads];                       // inclusive prefix of the window byte counts
    uint32_t part_a[kThreads], part_b[kThreads]; // Adler-32 sums of the threads' pieces of a segment
    uint8_t pal[768];
    uint64_t pos;
    int64_t opos;
    uint32_t crc_op[8];                          // x^(8 L 2^k): folds pieces of a split chunk CRC, level k
    uint32_t adler_a, adler_b, stored_len;
    int32_t status, btype, bfinal, kend, ticket;
};

static_assert(kThreads == 256, "Shared::crc_op holds log2(kThreads) levels");

__device__ __forceinline__ void set_status(Shared& S, int s) {
    if (s != kStOk) atomicCAS(&S.status, 0, s);
}

__device__ __forceinline__ uint8_t* byte_ptr(const PngFile& F, uint8_t* ring, int64_t q) {
    return q < F.filtered ? F.out + q : ring + (q & (kRing - 1));
}

// Resolves P[0 .. e - a) (the segment [a, e) of the output: v < 0 is the byte -1 - v, v >= 0 the position
// a - kWindow + v it copies from, which fits an int32 however long the stream), writes it out and folds its Adler-32
// into S.
//
// A round updates P in place while other threads read the same slots.  That is benign: every value a slot ever
// holds is its byte or a position of the same byte value further back, an int32 store does not tear, so a read
// sees the old or the new one and both are right; the barrier between rounds publishes the progress.
__device__ void finish_segment(const PngFile& F, Shared& S, int32_t* P, uint8_t* ring, int64_t a, int64_t e) {
    const int tid = threadIdx.x;
    const int len = (int)(e - a);
    for (;;) {
        int pending = 0;
        for (int i = tid; i < len; i += kThreads) {
            const int32_t v = P[i];
            if (v >= 0) {
                // A source always lies before its byte.  Only a slot the windows never wrote (their byte counts and
                // tokens disagreeing) could hold anything else, left over from an earlier segment or file: it is
                // never followed, so the scratch is only ever read inside [0, i).
                const int32_t r = v - kWindow;           // the source relative to the segment
                const int32_t back = r >= 0 && r < i ? P[r] : -1;
#ifndef AW_PNG_BROKEN_OVERLAP
                const int32_t nv = r < 0 ? -1 - (int32_t)*byte_ptr(F, ring, max(a + r, (int64_t)0)) : back;
#else
                const int32_t nv = r < 0 ? -1 : back;           // broken build: bytes before the segment not read
#endif
                P[i] = nv;
                pending |= nv >= 0;
            }
        }
        if (!__syncthreads_or(pending)) break;
    }
    const int per = (len + kThreads - 1) / kThreads;
    const int i0 = min(tid * per, len), i1 = min(i0 + per, len);
    uint32_t sa = 0, sb = 0;
    for (int i = i0; i < i1; ++i) {
        const uint8_t v = (uint8_t)(-1 - P[i]);
        *byte_ptr(F, ring, a + i) = v;
        sa += v;
        sb += sa;
    }
    S.part_a[tid] = sa % kAdlerMod;
    S.part_b[tid] = sb % kAdlerMod;
    __syncthreads();
    if (tid == 0) {
        uint32_t aa = S.adler_a, bb = S.adler_b;
        for (int t = 0; t < kThreads; ++t) {
            const int i0t = min(t * per, len), n = min(i0t + per, len) - i0t;
            adler_combine(aa, bb, S.part_a[t], S.part_b[t], (uint32_t)n);
        }
        S.adler_a = aa;
        S.adler_b = bb;
    }
    __syncthreads();
}

// Writes the P entries of this thread's window for output bytes in [a, e).
__device__ void emit_window(const PngFile& F, Shared& S, int32_t* P, uint64_t entry, uint64_t stop, int64_t o,
                            int64_t a, int64_t e) {
    const uint64_t* w = reinterpret_cast<const uint64_t*>(F.stream);
    uint64_t pos = entry;
    while (pos < stop && o < e) {
        int x = 0, d = 0;
        const int k = decode_token(S.lt, S.dt, w, &pos, &x, &d);
        if (k == kLiteral) {
            if (o >= a) P[o - a] = -1 - x;
            ++o;
        } else if (k == kMatch) {
            if ((int64_t)d > o) {
                set_status(S, kStDistance);
                return;
            }
            const int64_t q0 = o > a ? o : a, q1 = o + x < e ? o + x : e;
            for (int64_t q = q0; q < q1; ++q)
#ifndef AW_PNG_BROKEN_OVERLAP
                P[q - a] = (int32_t)(o - d + (q - o) % d - a + kWindow);
#else
                P[q - a] = (int32_t)(q - d - a + kWindow);
#endif
            o += x;
        } else {
            return;                              // not reached on a true trajectory before `stop`
        }
    }
}

// One Huffman block from S.pos (tables in S): window sets until the first end-of-block.
__device__ void huffman_block(const PngFile& F, Shared& S, int32_t* P, uint8_t* ring) {
    const int tid = threadIdx.x;
    const uint64_t bits = F.stream_bytes * 8;
    const uint64_t* w = reinterpret_cast<const uint64_t*>(F.stream);
    for (;;) {
        const uint64_t base = S.pos;
        if (base >= bits) {
            if (tid == 0) set_status(S, kStShortStream);
            __syncthreads();
            return;
        }
        const int nwin = (int)min((uint64_t)kThreads, (bits - base + kWinBits - 1) / kWinBits);
        const bool active = tid < nwin;
        const uint64_t ws = base + (uint64_t)tid * kWinBits;
        const uint64_t we = min(ws + kWinBits, bits);
        uint64_t entry = ws;
        WinResult r{};
        if (active) {
            run_window(S.lt, S.dt, w, entry, we, &r);
            S.exit[tid] = r.exit;
        }
        __syncthreads();
        for (;;) {                               // sync rounds
            const uint64_t want = active && tid > 0 ? S.exit[tid - 1] : entry;
            const bool redo = active && tid > 0 && want != entry;
            if (!__syncthreads_or(redo)) break;
            if (redo) {
                entry = want;
                run_window(S.lt, S.dt, w, entry, we, &r);
                S.exit[tid] = r.exit;
            }
            __syncthreads();
        }
        if (tid == 0) S.kend = nwin;
        __syncthreads();
        if (active && (r.has_eob || r.bad)) atomicMin(&S.kend, tid);
        __syncthreads();
        const int kend = S.kend;
        if (tid == kend) set_status(S, r.bad ? kStBadCode : r.eob_end > bits ? kStShortStream : kStOk);
        const int last = kend < nwin ? kend : nwin - 1;
        const uint32_t mine = tid <= last ? r.bytes : 0u;
        // exclusive prefix of the byte counts (Hillis-Steele over the CTA)
        S.off[tid] = mine;
        __syncthreads();
        for (int sh = 1; sh < kThreads; sh <<= 1) {
            const int64_t v = tid >= sh ? S.off[tid - sh] : 0;
            __syncthreads();
            S.off[tid] += v;
            __syncthreads();
        }
        const int64_t total = S.off[kThreads - 1];
        const int64_t my_off = S.off[tid] - mine;
        if (S.status != kStOk) return;
        const int64_t o0 = S.opos;
        const uint64_t stop = r.has_eob ? r.eob_end : r.exit;
        for (int64_t a = o0; a < o0 + total; a += kSeg) {
            const int64_t e = min(a + kSeg, o0 + total);
            if (tid <= last && mine > 0 && o0 + my_off < e && o0 + my_off + mine > a)
                emit_window(F, S, P, entry, stop, o0 + my_off, a, e);
            if (__syncthreads_or(S.status != kStOk)) return;
            finish_segment(F, S, P, ring, a, e);
        }
        __syncthreads();                         // every thread has read S.opos and S.pos of this set
        if (tid == 0) S.opos = o0 + total;
        if (kend < nwin ? tid == kend : tid == nwin - 1) S.pos = kend < nwin ? r.eob_end : r.exit;
        __syncthreads();
        if (kend < nwin) return;
    }
}

__device__ void stored_block(const PngFile& F, Shared& S, int32_t* P, uint8_t* ring) {
    const int tid = threadIdx.x;
    const int64_t o0 = S.opos;
    const uint8_t* b = F.stream + S.pos / 8;
    const int64_t len = S.stored_len;
    for (int64_t a = o0; a < o0 + len; a += kSeg) {
        const int64_t e = min(a + kSeg, o0 + len);
        for (int64_t q = a + tid; q < e; q += kThreads) P[q - a] = -1 - (int32_t)b[q - o0];
        __syncthreads();
        finish_segment(F, S, P, ring, a, e);
    }
    __syncthreads();                             // every thread has read S.opos, S.pos and S.stored_len
    if (tid == 0) {
        S.opos = o0 + len;
        S.pos += 8 * (uint64_t)len;
    }
    __syncthreads();
}

__device__ void inflate_file(const PngFile& F, Shared& S, int32_t* P, uint8_t* ring) {
    const int tid = threadIdx.x;
    const uint64_t bits = F.stream_bytes * 8;
    const uint64_t* w = reinterpret_cast<const uint64_t*>(F.stream);
    if (tid == 0) {
        S.pos = 16;
        S.opos = 0;
        S.adler_a = 1;
        S.adler_b = 0;
    }
    // The block state tid 0 writes (S.bfinal, S.btype, S.status, S.pos, S.stored_len) is read by every thread only
    // between the barrier after the header and the barrier that opens the next header, so no thread can see the
    // next block's header while it still acts on this one.
    for (;;) {
        __syncthreads();
        if (tid == 0) {                          // block header
            uint64_t pos = S.pos;
            if (pos + 3 > bits) {
                set_status(S, kStShortStream);
            } else {
                const uint64_t v = peek64(w, pos);
                S.bfinal = (int)(v & 1);
                S.btype = (int)((v >> 1) & 3);
                pos += 3;
                if (S.btype == 3) {
                    set_status(S, kStBlockType);
                } else if (S.btype == 0) {
                    pos = (pos + 7) & ~(uint64_t)7;
                    const uint64_t h = peek64(w, pos);
                    if (pos + 32 > bits) {
                        set_status(S, kStShortStream);
                    } else if (((h & 0xFFFF) ^ 0xFFFF) != ((h >> 16) & 0xFFFF)) {
                        set_status(S, kStStoredLen);
                    } else {
                        S.stored_len = (uint32_t)(h & 0xFFFF);
                        pos += 32;
                        if (pos + 8ull * S.stored_len > bits) set_status(S, kStShortStream);
                    }
                } else {
                    uint8_t ll[288], d[32];
                    int st = kStOk;
                    if (S.btype == 1) fixed_lengths(ll, d);
                    else st = read_dynamic(w, &pos, ll, d);
                    if (st == kStOk && pos > bits) st = kStShortStream;
                    if (st == kStOk && (huff_build(&S.lt, ll, 288, kLitLen) != 0 || huff_build(&S.dt, d, 32, kDist) != 0))
                        st = kStBadCode;
                    if (st != kStOk) set_status(S, st);
                }
                S.pos = pos;
            }
        }
        __syncthreads();
        if (S.status != kStOk) return;
        if (S.btype == 0) {
            stored_block(F, S, P, ring);
        } else {
            for (int i = tid; i < (1 << kFastBits); i += kThreads) {
                S.lt.fast[i] = huff_fast_entry(S.lt, i);
                S.dt.fast[i] = huff_fast_entry(S.dt, i);
            }
            __syncthreads();
            huffman_block(F, S, P, ring);
        }
        if (S.status != kStOk) return;
        if (S.bfinal) break;
    }
    __syncthreads();
    if (tid == 0) {                              // Adler-32 trailer, then the amount of data
        const uint64_t pos = (S.pos + 7) & ~(uint64_t)7;
        if (pos + 32 > bits) set_status(S, kStShortStream);
        else if (load_be32(F.stream + pos / 8) != (S.adler_b << 16 | S.adler_a)) set_status(S, kStAdler);
        else if (S.opos < F.filtered) set_status(S, kStShortImage);
    }
    __syncthreads();
}

__device__ void gather_and_check(const PngFile& F, Shared& S) {
    const int tid = threadIdx.x;
    uint64_t* w = reinterpret_cast<uint64_t*>(F.stream);
    const uint64_t tail = F.stream_bytes / 8;
    for (int i = tid; i <= kPad / 8; i += kThreads) w[tail + i] = 0;
    __syncthreads();
    for (int k = 0; k < F.nchunks; ++k) {
        const uint4 c = F.chunks[k];
        for (uint32_t i = tid; i < c.y; i += kThreads) F.stream[c.z + i] = F.src[c.x + i];
    }
    // CRC-32 of each chunk's type and data: small chunks one thread each ...
    for (int k = tid; k < F.nchunks; k += kThreads) {
        const uint4 c = F.chunks[k];
        if (c.y > kCrcSerial) continue;
        const uint8_t* p = F.src + c.x - 4;
        if (crc32_finish(crc_raw(0, p, 0, c.y + 4, S.crc), c.y + 4) != load_be32(F.src + c.x + c.y))
            set_status(S, kStIdatCrc);
    }
    // ... larger ones split into kThreads pieces (png_inflate.h crc_piece), folded as a tree in S.part_a
    for (int k = 0; k < F.nchunks; ++k) {
        const uint4 c = F.chunks[k];
        if (c.y <= kCrcSerial) continue;
        const uint64_t n = (uint64_t)c.y + 4;
        const uint8_t* p = F.src + c.x - 4;
        uint64_t b0, b1;
        crc_piece(n, kThreads, tid, &b0, &b1);
        __syncthreads();                         // the previous chunk's fold has been read
        S.part_a[tid] = crc_raw(0, p, b0, b1, S.crc);
        if (tid == 0) {
            S.crc_op[0] = crc_shift_operator((n + kThreads - 1) / kThreads);
            for (int l = 1; l < 8; ++l) S.crc_op[l] = crc_multmodp(S.crc_op[l - 1], S.crc_op[l - 1]);
        }
        __syncthreads();
        for (int l = 0, span = 1; span < kThreads; ++l, span *= 2) {
            if (tid % (2 * span) == 0) S.part_a[tid] = crc_combine(S.part_a[tid], S.part_a[tid + span], S.crc_op[l]);
            __syncthreads();
        }
        if (tid == 0 && crc32_finish(S.part_a[0], n) != load_be32(F.src + c.x + c.y)) set_status(S, kStIdatCrc);
    }
    __syncthreads();
}

__device__ void rows_to_bgr(const PngFile& F, Shared& S) {
    const int tid = threadIdx.x;
    const int64_t stride = F.row_bytes + 1;
    for (int y = tid; y < F.H; y += kThreads)
        if (F.out[(int64_t)y * stride] > 4) set_status(S, kStFilter);
    for (int i = tid; i < 768; i += kThreads) S.pal[i] = i < 3 * (int)F.plte_entries ? F.src[F.plte_off + i] : 0;
    if (__syncthreads_or(S.status != kStOk)) return;
    // wavefront: at step s, thread t takes the row r = s - ((s - t) mod kThreads) at chunk s - r
    const int64_t chunk = max((int64_t)kMinRowChunk, (F.row_bytes + kThreads - 1) / kThreads);
    const int64_t nch = (F.row_bytes + chunk - 1) / chunk;
    for (int64_t s = 0; s < F.H + nch - 1; ++s) {
        if (s >= tid) {
            const int64_t r = s - ((s - tid) % kThreads), c = s - r;
            if (r < F.H && c < nch) {
                uint8_t* row = F.out + r * stride + 1;
                unfilter_span(row, r ? row - stride : nullptr, row[-1], F.bpp, c * chunk,
                              min((c + 1) * chunk, F.row_bytes));
            }
        }
        __syncthreads();
    }
    const int64_t npx = (int64_t)F.H * F.W;
    for (int64_t p = tid; p < npx; p += kThreads) {
        const int64_t y = p / F.W, x = p % F.W;
        expand_pixel(F.out + y * stride + 1, x, F.colour, F.depth, S.pal, F.dst + p * 3);
    }
}

__global__ void __launch_bounds__(kThreads)
png_decode_kernel(const PngFile* __restrict__ files, const int32_t* __restrict__ order, int n,
                  uint32_t* __restrict__ ticket, int32_t* __restrict__ status, int32_t* __restrict__ scratch,
                  uint8_t* __restrict__ rings) {
    __shared__ Shared S;
    const int tid = threadIdx.x;
    int32_t* P = scratch + (size_t)blockIdx.x * kSeg;
    uint8_t* ring = rings + (size_t)blockIdx.x * kRing;
    for (int i = tid; i < 256; i += kThreads) crc_table(S.crc, i);
    for (;;) {
        if (tid == 0) S.ticket = (int32_t)atomicAdd(ticket, 1u);
        __syncthreads();
        if (S.ticket >= n) return;
        const int f = order[S.ticket];
        const PngFile F = files[f];
        if (tid == 0) S.status = kStOk;
        __syncthreads();
        gather_and_check(F, S);                  // each stage ends with a barrier after its last status write;
        bool ok = S.status == kStOk;             // the status is read before the barrier that lets the next
        __syncthreads();                         // stage write it
        if (ok) inflate_file(F, S, P, ring);
        ok = S.status == kStOk;
        __syncthreads();
        if (ok) rows_to_bgr(F, S);
        __syncthreads();
        if (tid == 0) status[f] = S.status;
        __syncthreads();
    }
}

// ---- workspace layout -------------------------------------------------------------------------------------------
struct Layout {
    size_t table, order, chunks, stream0, scratch, rings, end;
    int grid;
    int64_t nchunks;
};

// The one layout the workspace-size export and the call both use: descriptor table, order, ticket and chunk table
// (uploaded together), then per file its gathered stream and its inflated rows, then per CTA the resolution
// scratch and the ring.
Layout layout_of(const Header* hs, int n, int grid) {
    Layout L;
    L.grid = grid;
    L.nchunks = 0;
    for (int i = 0; i < n; ++i) L.nchunks += hs[i].idat_chunks;
    L.table = 0;
    L.order = align_up(sizeof(PngFile) * (size_t)n, 16);
    L.chunks = align_up(L.order + sizeof(int32_t) * (size_t)n + sizeof(uint32_t), 16);
    size_t at = align_up(L.chunks + sizeof(uint4) * (size_t)L.nchunks, 256);
    L.stream0 = at;
    for (int i = 0; i < n; ++i) {
        at = align_up(at + hs[i].stream_bytes + kPad + 8, 16);
        at = align_up(at + (size_t)hs[i].filtered, 16);
    }
    L.scratch = align_up(at, 256);
    L.rings = L.scratch + sizeof(int32_t) * kSeg * (size_t)grid;
    L.end = L.rings + (size_t)kRing * grid;
    return L;
}

int grid_for(int n) { return std::min(n, kCtasPerSm * sm_count()); }

}  // namespace

size_t png_decode_workspace_bytes_impl(const Header* hs, int n) { return layout_of(hs, n, grid_for(n)).end; }

// hs: the parsed, device-decodable headers of files (validated by the caller); ws of
// png_decode_workspace_bytes_impl(hs, n) bytes
int launch_decode_png(const attwarp_png_file* files, const Header* hs, int n, void* ws, int32_t* status,
                      cudaStream_t st) {
    const Layout L = layout_of(hs, n, grid_for(n));
    static thread_local std::vector<uint8_t> host;
    host.assign(L.stream0, 0);
    PngFile* tab = reinterpret_cast<PngFile*>(host.data() + L.table);
    int32_t* order = reinterpret_cast<int32_t*>(host.data() + L.order);
    uint4* chunks = reinterpret_cast<uint4*>(host.data() + L.chunks);
    char* base = static_cast<char*>(ws);
    size_t at = L.stream0;
    int64_t ck = 0;
    for (int i = 0; i < n; ++i) {
        const Header& h = hs[i];
        PngFile& F = tab[i];
        F.src = static_cast<const uint8_t*>(files[i].dev);
        F.dst = static_cast<uint8_t*>(files[i].dst);
        F.stream = reinterpret_cast<uint8_t*>(base + at);
        at = align_up(at + h.stream_bytes + kPad + 8, 16);
        F.out = reinterpret_cast<uint8_t*>(base + at);
        at = align_up(at + (size_t)h.filtered, 16);
        F.chunks = reinterpret_cast<const uint4*>(base + L.chunks) + ck;
        F.filtered = h.filtered;
        F.row_bytes = h.row_bytes;
        F.stream_bytes = h.stream_bytes;
        F.H = h.H;
        F.W = h.W;
        F.colour = h.colour;
        F.depth = h.depth;
        F.bpp = h.bpp;
        F.nchunks = (int32_t)h.idat_chunks;
        F.plte_off = h.plte_off;
        F.plte_entries = h.plte_entries;
        uint32_t soff = 0;
        Header again;
        parse_png(static_cast<const uint8_t*>(files[i].host), files[i].nbytes, &again, [&](uint32_t off, uint32_t len) {
            chunks[ck++] = make_uint4(off, len, soff, 0);
            soff += len;
        });
    }
    std::iota(order, order + n, 0);
    std::stable_sort(order, order + n, [&](int a, int b) { return hs[a].filtered > hs[b].filtered; });
    AW_CUDA(cudaMemcpyAsync(base, host.data(), L.stream0, cudaMemcpyHostToDevice, st));
    png_decode_kernel<<<L.grid, kThreads, 0, st>>>(reinterpret_cast<const PngFile*>(base + L.table),
                                                   reinterpret_cast<const int32_t*>(base + L.order), n,
                                                   reinterpret_cast<uint32_t*>(base + L.order + sizeof(int32_t) * n),
                                                   status, reinterpret_cast<int32_t*>(base + L.scratch),
                                                   reinterpret_cast<uint8_t*>(base + L.rings));
    return check_launch("png_decode_kernel");
}

}  // namespace aw
