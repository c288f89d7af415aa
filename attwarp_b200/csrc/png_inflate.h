// png_inflate.h -- the sequential pieces of the PNG decoder (png_decode.cu): the chunk walker and header probe,
// canonical Huffman tables and the deflate block headers (RFC 1951), the token decoder, the row unfilter step and
// the expansion of a pixel to BGR.
//
// Everything here is __host__ __device__ so that tests/hostcheck can compile it with g++ and check it against zlib
// and Pillow on a machine without a GPU.  The stream is read through a 64-bit word array (bit i of the stream is
// bit i % 64 of word i / 64, deflate's LSB-first order) padded with zeros past its end (1 KiB: more than a dynamic
// header that runs off the end reads), so that one read returns the next 64 bits: enough for a whole token (at most
// 15 + 5 + 15 + 13 = 48 bits).
#pragma once

#include <stddef.h>
#include <stdint.h>

#include "png_deflate.h"

namespace aw {
namespace png {

// ---- support codes of the probe (attwarp_png_support) and per-file status codes (attwarp_png_status) ----------
enum Support { kPngOk = 0, kNotPng = 1, kTruncated = 2, kBitDepth = 3, kInterlaced = 4, kBadCritical = 5,
               kStructure = 6, kSize = 7 };
enum Status { kStOk = 0, kStBlockType = 1, kStBadCode = 2, kStDistance = 3, kStStoredLen = 4, kStShortStream = 5,
              kStAdler = 6, kStIdatCrc = 7, kStFilter = 8, kStShortImage = 9 };

constexpr int kMaxDim = 1000000;                 // libpng's default limit on either side

struct Header {
    int32_t H, W, colour, depth, support;
    int32_t bpp;                                 // bytes of one complete pixel (1 for sub-byte pixels): the filter step
    int64_t row_bytes;                           // bytes of one row without its filter byte
    int64_t filtered;                            // H * (row_bytes + 1): the inflated stream the image needs
    uint64_t stream_bytes;                       // IDAT payload bytes (the zlib stream and whatever follows it)
    uint32_t idat_chunks;
    uint32_t plte_off, plte_entries;             // file offset of the PLTE data, its entries (0: none)
};

AW_PNG_HD uint32_t load_be32(const uint8_t* p) {
    return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | (uint32_t)p[3];
}

AW_PNG_HD uint32_t crc32_bytes(const uint8_t* p, size_t n) {
    return ~crc_update_bitwise(0xFFFFFFFFu, p, (int)n);
}

// ---- CRC-32 of a chunk split into equal pieces ----------------------------------------------------------------------
// A chunk's n bytes are cut into `pieces` pieces of L = ceil(n / pieces) bytes, the first one short: the bytes are
// taken as right-aligned in pieces * L, behind leading zeros, which leave a CRC register that starts at 0 unchanged.
// Piece t covers bytes [*b0, *b1) of the chunk.  Its raw CRC (register starting at 0, no final inversion) is linear,
// so two neighbours fold as crc_combine(left, right, x^(8 * their length)); the pieces fold as a tree of equal
// halves.  crc32_finish turns the raw CRC of all n bytes into the standard CRC-32 (register starting at ~0, final
// inversion): the initial ~0 reaches the end shifted by n bytes.
AW_PNG_HD void crc_piece(uint64_t n, int pieces, int t, uint64_t* b0, uint64_t* b1) {
    const uint64_t L = (n + pieces - 1) / pieces, pad = L * pieces - n;
    const uint64_t lo = (uint64_t)t * L, hi = lo + L;
    *b0 = lo > pad ? lo - pad : 0;
    *b1 = hi > pad ? hi - pad : 0;
}

AW_PNG_HD uint32_t crc_raw(uint32_t raw, const uint8_t* p, uint64_t a, uint64_t b, const uint32_t* table) {
    for (uint64_t i = a; i < b; ++i) raw = table[(raw ^ p[i]) & 0xFF] ^ (raw >> 8);
    return raw;
}

AW_PNG_HD uint32_t crc32_finish(uint32_t raw, uint64_t n) {
    return ~(raw ^ crc_multmodp(crc_shift_operator(n), 0xFFFFFFFFu));
}

AW_PNG_HD void crc_table(uint32_t* table, int i) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ kCrcPoly : c >> 1;
    table[i] = c;
}

AW_PNG_HD int channels_of(int colour) {
    return colour == 0 || colour == 3 ? 1 : colour == 2 ? 3 : colour == 4 ? 2 : 4;
}

// Walks the chunks of f[0 .. n) and fills *h; calls on_idat(data_offset, length) for every IDAT chunk in order.
// Checks the CRCs of the critical chunks other than IDAT (those of IDAT are the decoder's); ancillary chunks are
// skipped unchecked, as libpng does.  Returns h->support.
template <typename OnIdat>
AW_PNG_HD int parse_png(const uint8_t* f, size_t n, Header* h, OnIdat&& on_idat) {
    constexpr uint8_t kSig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    *h = Header{};
    h->support = kNotPng;
    for (size_t i = 0; i < 8; ++i) {
        if (i >= n) return h->support = (i > 0 ? kTruncated : kNotPng);
        if (f[i] != kSig[i]) return h->support;
    }
    size_t off = 8;
    bool ihdr = false, idat_open = false, idat_closed = false, iend = false;
    int interlace = 0;
    uint8_t zhead[2];
    int zhave = 0;
    while (!iend) {
        if (off + 8 > n) return h->support = kTruncated;
        const uint32_t len = load_be32(f + off);
        const uint8_t* type = f + off + 4;
        if (len > 0x7FFFFFFFu) return h->support = kStructure;
        if (off + 12 + (size_t)len > n) return h->support = kTruncated;
        const uint8_t* data = f + off + 8;
        const bool critical = (type[0] & 0x20) == 0;
        const bool is_idat = type[0] == 'I' && type[1] == 'D' && type[2] == 'A' && type[3] == 'T';
        if (critical && !is_idat && crc32_bytes(type, (size_t)len + 4) != load_be32(data + len))
            return h->support = kBadCritical;
        if (!ihdr) {
            if (!(type[0] == 'I' && type[1] == 'H' && type[2] == 'D' && type[3] == 'R') || len != 13)
                return h->support = kStructure;
            ihdr = true;
            h->W = (int32_t)(load_be32(data) & 0x7FFFFFFFu);
            h->H = (int32_t)(load_be32(data + 4) & 0x7FFFFFFFu);
            if (load_be32(data) == 0 || load_be32(data + 4) == 0 || load_be32(data) > 0x7FFFFFFFu ||
                load_be32(data + 4) > 0x7FFFFFFFu)
                return h->support = kStructure;
            h->depth = data[8];
            h->colour = data[9];
            const int d = h->depth, c = h->colour;
            const bool valid = (c == 0 && (d == 1 || d == 2 || d == 4 || d == 8 || d == 16)) ||
                               (c == 3 && (d == 1 || d == 2 || d == 4 || d == 8)) ||
                               ((c == 2 || c == 4 || c == 6) && (d == 8 || d == 16));
            if (!valid || data[10] != 0 || data[11] != 0 || data[12] > 1) return h->support = kStructure;
            interlace = data[12];
        } else if (is_idat) {
            if (idat_closed) return h->support = kStructure;              // IDAT chunks that are not consecutive
            idat_open = true;
            ++h->idat_chunks;
            h->stream_bytes += len;
            for (uint32_t k = 0; k < len && zhave < 2; ++k) zhead[zhave++] = data[k];
            on_idat((uint32_t)(off + 8), len);
        } else {
            if (idat_open) idat_closed = true;
            if (type[0] == 'I' && type[1] == 'E' && type[2] == 'N' && type[3] == 'D') {
                if (len != 0) return h->support = kStructure;
                iend = true;
            } else if (type[0] == 'P' && type[1] == 'L' && type[2] == 'T' && type[3] == 'E') {
                if (idat_open || h->plte_entries != 0 || h->colour == 0 || h->colour == 4 || len == 0 ||
                    len % 3 != 0 || len > 768)
                    return h->support = kStructure;
                h->plte_off = (uint32_t)(off + 8);
                h->plte_entries = len / 3;
            } else if (critical || (type[0] == 'I' && type[1] == 'H' && type[2] == 'D' && type[3] == 'R')) {
                return h->support = kStructure;                           // unknown critical chunk, second IHDR
            }
        }
        off += 12 + (size_t)len;
    }
    if (!idat_open || (h->colour == 3 && h->plte_entries == 0)) return h->support = kStructure;
    if (zhave < 2 || (zhead[0] & 15) != 8 || (zhead[0] >> 4) > 7 || ((uint32_t)zhead[0] * 256 + zhead[1]) % 31 != 0 ||
        (zhead[1] & 0x20) != 0)
        return h->support = kStructure;
    if (h->depth == 16) return h->support = kBitDepth;
    if (interlace) return h->support = kInterlaced;
    const int64_t bits = (int64_t)h->W * channels_of(h->colour) * h->depth;
    h->row_bytes = (bits + 7) / 8;
    h->bpp = (int32_t)((channels_of(h->colour) * h->depth + 7) / 8);
    h->filtered = (int64_t)h->H * (h->row_bytes + 1);
    if (h->W > kMaxDim || h->H > kMaxDim || h->filtered > 0x7FFFFFFFLL || h->stream_bytes > 0x7FFFFFF0ull)
        return h->support = kSize;
    return h->support = kPngOk;
}

// ---- bit reading ------------------------------------------------------------------------------------------------
AW_PNG_HD uint64_t peek64(const uint64_t* w, uint64_t pos) {
    const uint64_t i = pos >> 6;
    const int sh = (int)(pos & 63);
    const uint64_t lo = w[i] >> sh;
    return sh ? lo | (w[i + 1] << (64 - sh)) : lo;
}

// ---- canonical Huffman tables (RFC 1951 section 3.2.2) --------------------------------------------------------------
constexpr int kFastBits = 9;

struct Huff {
    uint16_t count[kMaxBits + 1];                // codes of each length
    uint16_t sym[288];                           // symbols in canonical order
    uint16_t fast[1 << kFastBits];               // next kFastBits bits -> sym << 4 | length; 0: a longer code or none
};

// Which of zlib's rules (inflate_table) a code is held to: the code-length code must be complete; the literal/length
// and distance codes may also be incomplete with a single code of length 1; the distance code may also be empty (a
// block of literals only).
enum CodeKind { kCodeLengths = 0, kLitLen = 1, kDist = 2 };

// Counts and canonical symbol order of lens[0 .. n).  Returns 0 for a code `kind` allows, -1 for an over-subscribed
// or otherwise incomplete or empty one.
AW_PNG_HD int huff_build(Huff* t, const uint8_t* lens, int n, int kind) {
    uint16_t offs[kMaxBits + 2];
    for (int l = 0; l <= kMaxBits; ++l) t->count[l] = 0;
    for (int s = 0; s < n; ++s) t->count[lens[s]]++;
    t->count[0] = 0;
    int max = 0;
    for (int l = 1; l <= kMaxBits; ++l)
        if (t->count[l]) max = l;
    offs[1] = 0;
    for (int l = 1; l <= kMaxBits; ++l) offs[l + 1] = (uint16_t)(offs[l] + t->count[l]);
    for (int s = 0; s < n; ++s)
        if (lens[s]) t->sym[offs[lens[s]]++] = (uint16_t)s;
    if (max == 0) return kind == kDist ? 0 : -1;
    int left = 1;
    for (int l = 1; l <= kMaxBits; ++l) {
        left = (left << 1) - t->count[l];
        if (left < 0) return -1;
    }
    return left > 0 && (kind == kCodeLengths || max != 1) ? -1 : 0;
}

// The symbol whose code starts the LSB-first bits, by the code lengths alone (puff's decode): its length, 0 when no
// code of the table matches.
AW_PNG_HD int huff_slow(const Huff& t, uint64_t bits, int* sym) {
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= kMaxBits; ++len) {
        code |= (int)(bits & 1);
        bits >>= 1;
        const int count = t.count[len];
        if (code - first < count) {
            *sym = t.sym[index + (code - first)];
            return len;
        }
        index += count;
        first = (first + count) << 1;
        code <<= 1;
    }
    return 0;
}

// Entry i of the fast table (a CTA fills them in parallel).
AW_PNG_HD uint16_t huff_fast_entry(const Huff& t, int i) {
    int sym = 0;
    const int len = huff_slow(t, (uint64_t)i, &sym);
    return len > 0 && len <= kFastBits ? (uint16_t)(sym << 4 | len) : (uint16_t)0;
}

AW_PNG_HD int huff_decode(const Huff& t, uint64_t bits, int* sym) {
    const uint16_t e = t.fast[bits & ((1u << kFastBits) - 1)];
    if (e) {
        *sym = e >> 4;
        return e & 15;
    }
    return huff_slow(t, bits, sym);
}

AW_PNG_HD void fixed_lengths(uint8_t* ll, uint8_t* d) {
    for (int s = 0; s < 288; ++s) ll[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
    for (int s = 0; s < 32; ++s) d[s] = 5;
}

// Code lengths of a block: BTYPE 1 (fixed) or the dynamic header at bit *pos (just after BFINAL and BTYPE), which is
// advanced past it.  ll[0 .. 288), d[0 .. 32) are written in full.  Returns kStOk or kStBadCode.
AW_PNG_HD int read_dynamic(const uint64_t* w, uint64_t* pos, uint8_t* ll, uint8_t* d) {
    constexpr uint8_t kOrder[kClSymbols] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint64_t p = *pos;
    uint64_t v = peek64(w, p);
    const int nlen = (int)(v & 31) + 257, ndist = (int)((v >> 5) & 31) + 1, ncode = (int)((v >> 10) & 15) + 4;
    p += 14;
    if (nlen > 286 || ndist > 30) return kStBadCode;
    uint8_t cl[kClSymbols];
    for (int k = 0; k < kClSymbols; ++k) cl[k] = 0;
    v = peek64(w, p);
    for (int k = 0; k < ncode; ++k) cl[kOrder[k]] = (uint8_t)((v >> (3 * k)) & 7);
    p += 3 * ncode;
    Huff ct;
    if (huff_build(&ct, cl, kClSymbols, kCodeLengths) != 0) return kStBadCode;
    uint8_t lens[286 + 30];
    int k = 0;
    while (k < nlen + ndist) {
        v = peek64(w, p);
        int sym = 0;
        const int l = huff_slow(ct, v, &sym);
        if (l == 0) return kStBadCode;
        p += l;
        v >>= l;
        if (sym < 16) {
            lens[k++] = (uint8_t)sym;
            continue;
        }
        int rep, val = 0;
        if (sym == 16) {
            if (k == 0) return kStBadCode;
            val = lens[k - 1];
            rep = 3 + (int)(v & 3);
            p += 2;
        } else if (sym == 17) {
            rep = 3 + (int)(v & 7);
            p += 3;
        } else {
            rep = 11 + (int)(v & 127);
            p += 7;
        }
        if (k + rep > nlen + ndist) return kStBadCode;
        while (rep--) lens[k++] = (uint8_t)val;
    }
    if (lens[256] == 0) return kStBadCode;                                // no end-of-block code
    for (int s = 0; s < 288; ++s) ll[s] = s < nlen ? lens[s] : 0;
    for (int s = 0; s < 32; ++s) d[s] = s < ndist ? lens[nlen + s] : 0;
    *pos = p;
    return kStOk;
}

// ---- tokens -----------------------------------------------------------------------------------------------------
enum TokKind { kLiteral = 0, kMatch = 1, kEob = 2, kBad = 3 };

AW_PNG_HD int dist_base(int ds, int de) { return ds < 4 ? ds + 1 : ((2 + (ds & 1)) << de) + 1; }

// One token at bit *pos of a Huffman block: a literal (*a = the byte), a match (*a = length, *b = distance), the
// end of block, or kBad for a bit pattern that is no code, a literal/length symbol 286-287 or a distance symbol
// 30-31.  *pos is advanced past the token, and left unchanged for kBad.
AW_PNG_HD int decode_token(const Huff& lt, const Huff& dt, const uint64_t* w, uint64_t* pos, int* a, int* b) {
    uint64_t v = peek64(w, *pos);
    int sym = 0;
    int l = huff_decode(lt, v, &sym);
    if (l == 0 || sym > 285) return kBad;
    if (sym < 256) {
        *pos += l;
        *a = sym;
        return kLiteral;
    }
    if (sym == 256) {
        *pos += l;
        return kEob;
    }
    int used = l;
    v >>= l;
    const int li = sym - 257;                    // length base and extra bits, RFC 1951 section 3.2.5
    const int le = li < 8 || li == 28 ? 0 : (li >> 2) - 1;
    const int lbase = li < 8 ? 3 + li : li == 28 ? 258 : ((4 + (li & 3)) << le) + 3;
    *a = lbase + (int)(v & ((1u << le) - 1));
    v >>= le;
    used += le;
    int ds = 0;
    l = huff_decode(dt, v, &ds);
    if (l == 0 || ds > 29) return kBad;
    v >>= l;
    used += l;
    const int de = ds < 4 ? 0 : (ds >> 1) - 1;
    *b = dist_base(ds, de) + (int)(v & ((1u << de) - 1));
    used += de;
    *pos += used;
    return kMatch;
}

// ---- windows of a Huffman block ------------------------------------------------------------------------------------
// The decoder state is the bit position at a token boundary: after a complete token the next symbol is always a
// literal/length code of the block's own table, so two trajectories that reach the same position at a token
// boundary agree from there on.  A window decodes from `entry` to the first token boundary at or past `end`; a
// token that starts in the window is finished by it, distance included.  After a bad code the decode goes on from
// the next bit (a guessed entry that meets one keeps a trajectory that can still meet the true one), and an
// end-of-block code does not stop it: the exit stays a function of the entry alone.  On the true trajectory the
// first end-of-block ends the block, and a bad code before it fails the file.
struct WinResult {
    uint64_t exit, eob_end;                      // exit position; the position after the first end-of-block code
    uint32_t bytes;                              // bytes the tokens before the first end-of-block code produce
    uint8_t has_eob, bad;                        // an end-of-block code seen; a bad code before it
};

AW_PNG_HD void run_window(const Huff& lt, const Huff& dt, const uint64_t* w, uint64_t entry, uint64_t end,
                          WinResult* r) {
    uint64_t pos = entry;
    uint32_t bytes = 0;
    r->has_eob = r->bad = 0;
    r->eob_end = 0;
    while (pos < end) {
        int a = 0, b = 0;
#ifdef AW_PNG_BROKEN_SYNC_MID_TOKEN
        const uint64_t p0 = pos;
#endif
        const int k = decode_token(lt, dt, w, &pos, &a, &b);
        if (r->has_eob) {
            if (k == kBad) ++pos;
            continue;
        }
        if (k == kBad) {
            r->bad = 1;
            ++pos;
        } else if (k == kEob) {
            r->has_eob = 1;
            r->eob_end = pos;
        } else {
            bytes += k == kLiteral ? 1u : (uint32_t)a;
#ifdef AW_PNG_BROKEN_SYNC_MID_TOKEN
            if (k == kMatch && pos > end) {      // broken build: a match crossing `end` is cut before its distance
                int sym = 0;
                const int l = huff_decode(lt, peek64(w, p0), &sym), li = sym - 257;
                const uint64_t len_end = p0 + l + (li < 8 || li == 28 ? 0 : (li >> 2) - 1);
                if (len_end < end) pos = len_end;
            }
#endif
        }
    }
    r->exit = pos;
    r->bytes = bytes;
}

// ---- rows -------------------------------------------------------------------------------------------------------
AW_PNG_HD int paeth(int a, int b, int c) {
    const int p = a + b - c;
    const int pa = p > a ? p - a : a - p, pb = p > b ? p - b : b - p, pc = p > c ? p - c : c - p;
    if (pa <= pb && pa <= pc) return a;
    return pb <= pc ? b : c;
}

// Reverses filter `ft` (1-4) on row[x0 .. x1) in place; prev is the row above (already unfiltered), nullptr for
// the first row.  row[0 .. x0) must be unfiltered already.
AW_PNG_HD void unfilter_span(uint8_t* row, const uint8_t* prev, int ft, int bpp, int64_t x0, int64_t x1) {
    for (int64_t x = x0; x < x1; ++x) {
        const int a = x >= bpp ? row[x - bpp] : 0;
        const int b = prev ? prev[x] : 0;
        const int c = prev && x >= bpp ? prev[x - bpp] : 0;
        int pred;
        switch (ft) {
        case 1: pred = a; break;
        case 2: pred = b; break;
        case 3: pred = (a + b) >> 1; break;
#ifndef AW_PNG_BROKEN_PAETH_AS_UP
        case 4: pred = paeth(a, b, c); break;
#else
        case 4: pred = b; break;
#endif
        default: pred = 0; break;
        }
        row[x] = (uint8_t)(row[x] + pred);
    }
}

// Pixel x of an unfiltered row -> BGR.  pal: 256 RGB entries, zero past the file's PLTE.  Sub-byte grey is scaled
// to 8 bits as Pillow and libpng do (x 255, 85, 17); alpha is dropped.
AW_PNG_HD void expand_pixel(const uint8_t* row, int64_t x, int colour, int depth, const uint8_t* pal, uint8_t* bgr) {
    int v;
    switch (colour) {
    case 2:
        bgr[0] = row[3 * x + 2];
        bgr[1] = row[3 * x + 1];
        bgr[2] = row[3 * x];
        return;
    case 6:
        bgr[0] = row[4 * x + 2];
        bgr[1] = row[4 * x + 1];
        bgr[2] = row[4 * x];
        return;
    case 4:
        bgr[0] = bgr[1] = bgr[2] = row[2 * x];
        return;
    default:
        break;
    }
    if (depth == 8) {
        v = row[x];
    } else {
        const int64_t bit = x * depth;
        v = (row[bit >> 3] >> (8 - depth - (int)(bit & 7))) & ((1 << depth) - 1);
    }
    if (colour == 0) {
        const uint8_t g = (uint8_t)(depth == 8 ? v : v * (255 / ((1 << depth) - 1)));
        bgr[0] = bgr[1] = bgr[2] = g;
    } else {
        bgr[0] = pal[3 * v + 2];
        bgr[1] = pal[3 * v + 1];
        bgr[2] = pal[3 * v];
    }
}

}  // namespace png
}  // namespace aw
