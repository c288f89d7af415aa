// TEST-ONLY host harness: compiles attwarp_b200/csrc/png_inflate.h with g++ and runs a whole decode through it (the
// probe, block headers, Huffman tables, the window decode of png_decode.cu run one window after another, the row
// unfilter and the BGR expansion), so that the pieces the PNG kernel runs can be checked against zlib and Pillow on
// a machine without a GPU.  Matches are copied byte by byte here; the kernel's parallel LZ77 resolution is checked
// on the GPU.  Never linked into the product.
#include <stdint.h>
#include <string.h>

#include <set>
#include <vector>

#include "../../attwarp_b200/csrc/png_inflate.h"

using namespace aw::png;

namespace {

constexpr int kWinBits = 512;
constexpr int kWindows = 256;                    // windows per set, as one CTA of the kernel

struct Stream {
    std::vector<uint64_t> w;
    uint64_t bits;
};

Stream gather(const uint8_t* f, size_t n, Header* h) {
    std::vector<uint8_t> bytes;
    parse_png(f, n, h, [&](uint32_t off, uint32_t len) { bytes.insert(bytes.end(), f + off, f + off + len); });
    Stream s;
    s.bits = (uint64_t)bytes.size() * 8;
    s.w.assign((bytes.size() + 7) / 8 + 130, 0);      // 1 KiB of zeros past the end, as the kernel
    if (!bytes.empty()) memcpy(s.w.data(), bytes.data(), bytes.size());
    return s;
}

uint32_t bits_at(const Stream& s, uint64_t pos, int n) { return (uint32_t)(peek64(s.w.data(), pos) & ((1u << n) - 1)); }

void fill_fast(Huff* t) {
    for (int i = 0; i < (1 << kFastBits); ++i) t->fast[i] = huff_fast_entry(*t, i);
}

// Inflates the zlib stream of s into out; returns a Status.  stats (nullable): [0] windows with a guessed entry,
// [1] windows those guessed trajectories took to meet the true one, summed, [2] the largest such count.
int inflate(const Stream& s, std::vector<uint8_t>& out, int64_t* stats) {
    uint64_t pos = 16;
    out.clear();
    for (;;) {
        if (pos + 3 > s.bits) return kStShortStream;
        const int bfinal = (int)bits_at(s, pos, 1), btype = (int)bits_at(s, pos + 1, 2);
        pos += 3;
        if (btype == 3) return kStBlockType;
        if (btype == 0) {
            pos = (pos + 7) & ~(uint64_t)7;
            if (pos + 32 > s.bits) return kStShortStream;
            const uint32_t len = bits_at(s, pos, 16), nlen = bits_at(s, pos + 16, 16);
            if ((len ^ 0xFFFFu) != nlen) return kStStoredLen;
            pos += 32;
            if (pos + 8ull * len > s.bits) return kStShortStream;
            const uint8_t* b = reinterpret_cast<const uint8_t*>(s.w.data()) + pos / 8;
            out.insert(out.end(), b, b + len);
            pos += 8ull * len;
        } else {
            uint8_t ll[288], d[32];
            if (btype == 1) {
                fixed_lengths(ll, d);
            } else {
                if (read_dynamic(s.w.data(), &pos, ll, d) != kStOk) return kStBadCode;
                if (pos > s.bits) return kStShortStream;
            }
            Huff lt, dt;
            if (huff_build(&lt, ll, 288, kLitLen) != 0 || huff_build(&dt, d, 32, kDist) != 0) return kStBadCode;
            fill_fast(&lt);
            fill_fast(&dt);
            // the block in sets of kWindows windows, each window from the exit of the one before it (the fixed
            // point the kernel's sync rounds reach), until the first end-of-block
            bool ended = false;
            std::set<uint64_t> truth;            // token boundaries of the true trajectory in this set
            while (!ended) {
                if (pos >= s.bits) return kStShortStream;
                uint64_t entry = pos;
                std::vector<uint64_t> entries;
                for (int t = 0; t < kWindows && !ended; ++t) {
                    const uint64_t ws = pos + (uint64_t)t * kWinBits;
                    if (ws >= s.bits) break;
                    const uint64_t we = ws + kWinBits < s.bits ? ws + kWinBits : s.bits;
                    if (t > 0) entries.push_back(ws);
                    WinResult r;
                    run_window(lt, dt, s.w.data(), entry, we, &r);
                    if (r.bad) return kStBadCode;
                    // replay the window's tokens into out
                    uint64_t p = entry;
                    const uint64_t stop = r.has_eob ? r.eob_end : r.exit;
                    while (p < stop) {
                        if (stats) truth.insert(p);
                        int a = 0, b = 0;
                        const int k = decode_token(lt, dt, s.w.data(), &p, &a, &b);
                        if (k == kLiteral) {
                            out.push_back((uint8_t)a);
                        } else if (k == kMatch) {
                            if ((size_t)b > out.size()) return kStDistance;
                            const size_t from = out.size() - (size_t)b;
                            for (int q = 0; q < a; ++q) out.push_back(out[from + q]);
                        }
                    }
                    if (r.has_eob) {
                        if (r.eob_end > s.bits) return kStShortStream;
                        ended = true;
                        pos = r.eob_end;
                    }
                    entry = r.exit;
                }
                if (stats && !truth.empty()) {
                    const uint64_t hi = *truth.rbegin();
                    for (uint64_t g : entries) {     // a guessed entry at a window start: follow it to the truth
                        uint64_t p = g;
                        while (!truth.count(p) && p < hi) {
                            int a = 0, b = 0;
                            if (decode_token(lt, dt, s.w.data(), &p, &a, &b) == kBad) ++p;
                        }
                        if (!truth.count(p)) continue;   // meets it only past this set
                        const int64_t wins = (int64_t)((p - g) / kWinBits) + 1;
                        stats[0] += 1;
                        stats[1] += wins;
                        if (wins > stats[2]) stats[2] = wins;
                    }
                    truth.clear();
                }
                if (!ended) pos = entry;
            }
        }
        if (bfinal) break;
    }
    pos = (pos + 7) & ~(uint64_t)7;
    if (pos + 32 > s.bits) return kStShortStream;
    uint32_t a = 1, b = 0;
    for (uint8_t v : out) {
        a = (a + v) % kAdlerMod;
        b = (b + a) % kAdlerMod;
    }
    const uint8_t* t = reinterpret_cast<const uint8_t*>(s.w.data()) + pos / 8;
    if (load_be32(t) != (b << 16 | a)) return kStAdler;
    return kStOk;
}

}  // namespace

extern "C" {

// info[0..4] = H, W, colour type, bit depth, support code
int hc_png_probe(const uint8_t* f, size_t n, int32_t* info) {
    Header h;
    parse_png(f, n, &h, [](uint32_t, uint32_t) {});
    info[0] = h.H;
    info[1] = h.W;
    info[2] = h.colour;
    info[3] = h.depth;
    info[4] = h.support;
    return h.support;
}

// The inflated zlib stream of the file's IDAT chunks into out (cap bytes); *n_out its length.  Returns the negated
// Status (< 0) of a malformed stream, 0 on success.  stats: see inflate().
int hc_png_inflate(const uint8_t* f, size_t n, uint8_t* out, int64_t cap, int64_t* n_out, int64_t* stats) {
    Header h;
    const Stream s = gather(f, n, &h);
    std::vector<uint8_t> o;
    const int st = inflate(s, o, stats);
    if (st != kStOk) return -st;
    *n_out = (int64_t)o.size();
    if ((int64_t)o.size() <= cap) memcpy(out, o.data(), o.size());
    return 0;
}

// Whole decode into out (H * W * 3 BGR).  Returns the support code (> 0) of a file outside the subset, the negated
// Status (< 0) of a malformed one, 0 on success.
int hc_png_decode(const uint8_t* f, size_t n, uint8_t* out) {
    Header h;
    const Stream s = gather(f, n, &h);
    if (h.support != kPngOk) return h.support;
    std::vector<uint8_t> o;
    int st = inflate(s, o, nullptr);
    if (st != kStOk) return -st;
    if ((int64_t)o.size() < h.filtered) return -kStShortImage;
    const int64_t stride = h.row_bytes + 1;
    for (int y = 0; y < h.H; ++y)
        if (o[(size_t)(y * stride)] > 4) return -kStFilter;
    for (int y = 0; y < h.H; ++y) {
        uint8_t* row = o.data() + y * stride + 1;
        unfilter_span(row, y ? row - stride : nullptr, o[(size_t)(y * stride)], h.bpp, 0, h.row_bytes);
    }
    uint8_t pal[768];
    memset(pal, 0, sizeof(pal));
    if (h.plte_entries) memcpy(pal, f + h.plte_off, 3 * h.plte_entries);
    for (int y = 0; y < h.H; ++y)
        for (int x = 0; x < h.W; ++x)
            expand_pixel(o.data() + y * stride + 1, x, h.colour, h.depth, pal, out + ((size_t)y * h.W + x) * 3);
    return 0;
}

// CRC-32 of p[0 .. n) computed as the kernel splits a chunk: `pieces` pieces, each a raw CRC, folded as a tree.
uint32_t hc_crc32_split(const uint8_t* p, uint64_t n, int pieces) {
    uint32_t table[256];
    for (int i = 0; i < 256; ++i) crc_table(table, i);
    std::vector<uint32_t> raw((size_t)pieces);
    for (int t = 0; t < pieces; ++t) {
        uint64_t b0, b1;
        crc_piece(n, pieces, t, &b0, &b1);
        raw[(size_t)t] = crc_raw(0, p, b0, b1, table);
    }
    const uint64_t L = (n + pieces - 1) / pieces;
    uint32_t op = crc_shift_operator(L);
    for (int span = 1; span < pieces; span *= 2, op = crc_multmodp(op, op))
        for (int t = 0; t + span < pieces; t += 2 * span) raw[(size_t)t] = crc_combine(raw[(size_t)t], raw[(size_t)(t + span)], op);
    return crc32_finish(raw[0], n);
}

// huff_build's verdict (0 or -1) on lens[0 .. n) for a code kind (0 code lengths, 1 literal/length, 2 distance).
int hc_huff_build(const uint8_t* lens, int n, int kind) {
    Huff t;
    return huff_build(&t, lens, n, kind);
}

}  // extern "C"
