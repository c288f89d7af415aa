// png_deflate.h -- the sequential pieces of the PNG encoder (png.cu): length-limited Huffman code lengths,
// canonical codes, the dynamic-block header (RFC 1951 section 3.2.7), the greedy distance-1 tokeniser and the
// CRC-32 arithmetic.
//
// Everything here is __host__ __device__ so that tests/hostcheck can compile it with g++ and check it against
// zlib on a machine without a GPU.  One thread of a CTA runs the Huffman and header code; the tokeniser is run by
// every thread over its own chunk of the segment.
#pragma once

#include <stdint.h>

#if defined(__CUDACC__)
#define AW_PNG_HD __host__ __device__ __forceinline__
#else
#define AW_PNG_HD inline
#endif

namespace aw {
namespace png {

constexpr int kLitLenSymbols = 286;     // 0-255 literals, 256 end of block, 257-285 lengths
constexpr int kClSymbols = 19;          // code-length alphabet
constexpr int kMaxBits = 15;            // longest literal/length code
constexpr int kMaxClBits = 7;           // longest code-length code

// ---- Huffman code lengths --------------------------------------------------------------------------------------
// sorted[0..m): the symbols of non-zero count in ascending (count, symbol) order.  Insertion sort (host and the
// 19-symbol code-length alphabet; png.cu ranks the literal/length alphabet in parallel instead).
AW_PNG_HD int huff_sort(const uint32_t* freq, int n, uint16_t* sorted) {
    int m = 0;
    for (int s = 0; s < n; ++s) {
        if (freq[s] == 0) continue;
        int j = m++;
        while (j > 0 && freq[sorted[j - 1]] > freq[s]) {
            sorted[j] = sorted[j - 1];
            --j;
        }
        sorted[j] = (uint16_t)s;
    }
    return m;
}

// Code lengths of the symbols in `sorted` (m of n, ascending count) limited to max_bits; lens[0..n) is written in
// full (0 = unused symbol).  Fewer than two used symbols get two codes of length 1 (the lowest unused symbol fills
// in), so that the code is always complete.  work: >= m uint32.
//
// Minimum-redundancy lengths by Moffat and Katajainen's in-place algorithm ("In-place calculation of
// minimum-redundancy codes", 1995), then the length limit: the counts of codes longer than max_bits are moved to
// max_bits and the Kraft sum is brought back to 1 by lengthening the longest codes that are still shorter than
// max_bits.  The lengths go back to the symbols in count order, the longest to the rarest.
AW_PNG_HD void huff_lengths_sorted(const uint32_t* freq, const uint16_t* sorted, int m, int n, int max_bits,
                                   uint8_t* lens, uint32_t* work) {
    for (int s = 0; s < n; ++s) lens[s] = 0;
    if (m < 2) {
        int a = m == 1 ? sorted[0] : -1, filled = 0;
        if (a >= 0) lens[a] = 1, ++filled;
        for (int s = 0; s < n && filled < 2; ++s)
            if (s != a) lens[s] = 1, ++filled;
        return;
    }
    uint32_t* A = work;
    for (int i = 0; i < m; ++i) A[i] = freq[sorted[i]];
    // phase 1: internal node weights, parents as indices
    A[0] += A[1];
    int root = 0, leaf = 2;
    for (int next = 1; next < m - 1; ++next) {
        if (leaf >= m || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = (uint32_t)next; }
        else A[next] = A[leaf++];
        if (leaf >= m || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = (uint32_t)next; }
        else A[next] += A[leaf++];
    }
    // phase 2: internal node depths
    A[m - 2] = 0;
    for (int next = m - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
    // phase 3: leaf depths, A[0] the longest
    int avbl = 1, used = 0, dpth = 0, next = m - 1;
    root = m - 2;
    while (avbl > 0) {
        while (root >= 0 && (int)A[root] == dpth) { ++used; --root; }
        while (avbl > used) { A[next--] = (uint32_t)dpth; --avbl; }
        avbl = 2 * used;
        ++dpth;
        used = 0;
    }
    // length limit
    int count[kMaxBits + 1];
    for (int l = 0; l <= max_bits; ++l) count[l] = 0;
    for (int i = 0; i < m; ++i) count[A[i] > (uint32_t)max_bits ? max_bits : A[i]]++;
    uint32_t total = 0;
    for (int l = 1; l <= max_bits; ++l) total += (uint32_t)count[l] << (max_bits - l);
    while (total != (1u << max_bits)) {
        count[max_bits]--;
        for (int l = max_bits - 1; l > 0; --l)
            if (count[l] != 0) {
                count[l]--;
                count[l + 1] += 2;
                break;
            }
        total--;
    }
    int i = 0;
    for (int l = max_bits; l > 0; --l)
        for (int k = 0; k < count[l]; ++k) lens[sorted[i++]] = (uint8_t)l;
}

// Canonical codes (RFC 1951 section 3.2.2), bit-reversed: deflate sends Huffman codes most significant bit first
// into an LSB-first stream.
AW_PNG_HD void huff_codes(const uint8_t* lens, int n, uint16_t* rev_codes) {
    int bl_count[kMaxBits + 1], next_code[kMaxBits + 1];
    for (int l = 0; l <= kMaxBits; ++l) bl_count[l] = 0;
    for (int s = 0; s < n; ++s) bl_count[lens[s]]++;
    bl_count[0] = 0;
    int code = 0;
    for (int l = 1; l <= kMaxBits; ++l) {
        code = (code + bl_count[l - 1]) << 1;
        next_code[l] = code;
    }
    for (int s = 0; s < n; ++s) {
        const int l = lens[s];
        uint32_t c = l ? (uint32_t)next_code[l]++ : 0u, r = 0;
        for (int b = 0; b < l; ++b, c >>= 1) r = (r << 1) | (c & 1u);
        rev_codes[s] = (uint16_t)r;
    }
}

// ---- bit writer (LSB first, whole bytes) ------------------------------------------------------------------------
struct BitWriter {
    uint8_t* out;
    uint64_t acc;
    int nacc;
    int bytes;
    AW_PNG_HD void put(uint32_t v, int n) {
        acc |= (uint64_t)v << nacc;
        nacc += n;
        while (nacc >= 8) {
            out[bytes++] = (uint8_t)acc;
            acc >>= 8;
            nacc -= 8;
        }
    }
    AW_PNG_HD int bits() const { return bytes * 8 + nacc; }
    AW_PNG_HD void flush_partial() {          // the pending bits as one last (zero-padded) byte; bits() unchanged
        if (nacc > 0) out[bytes] = (uint8_t)acc;
    }
};

// ---- dynamic block header ---------------------------------------------------------------------------------------
// Calls emit(symbol, extra_value, extra_bits) for the run-length coding of the concatenated code lengths
// ll_lens[0..n_ll) ++ d_lens[0..n_d) with the code-length alphabet (16: repeat the previous length 3-6 times,
// 17: 3-10 zeros, 18: 11-138 zeros).
template <typename Emit>
AW_PNG_HD void cl_tokens(const uint8_t* ll_lens, int n_ll, const uint8_t* d_lens, int n_d, Emit&& emit) {
    const int total = n_ll + n_d;
    int i = 0;
    while (i < total) {
        const int v = i < n_ll ? ll_lens[i] : d_lens[i - n_ll];
        int r = 1;
        while (i + r < total && (i + r < n_ll ? ll_lens[i + r] : d_lens[i + r - n_ll]) == v) ++r;
        i += r;
        if (v == 0) {
            while (r >= 11) {
                const int k = r < 138 ? r : 138;
                emit(18, k - 11, 7);
                r -= k;
            }
            if (r >= 3) {
                emit(17, r - 3, 3);
                r = 0;
            }
            for (; r > 0; --r) emit(0, 0, 0);
        } else {
            emit(v, 0, 0);
            --r;
            while (r >= 3) {
                const int k = r < 6 ? r : 6;
                emit(16, k - 3, 2);
                r -= k;
            }
            for (; r > 0; --r) emit(v, 0, 0);
        }
    }
}

// Writes the block header of a dynamic-Huffman block -- BFINAL, BTYPE = 2, HLIT, HDIST, HCLEN, the code-length
// code and the run-length coded literal/length and distance code lengths -- into bw.  ll_lens: 286 entries,
// d_lens: n_d >= 1 entries.  HLIT is trimmed to the last used literal/length symbol (at least 257).
AW_PNG_HD void write_dynamic_header(BitWriter& bw, int bfinal, const uint8_t* ll_lens, const uint8_t* d_lens, int n_d) {
    constexpr uint8_t kOrder[kClSymbols] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    int n_ll = kLitLenSymbols;
    while (n_ll > 257 && ll_lens[n_ll - 1] == 0) --n_ll;
    uint32_t cl_freq[kClSymbols];
    for (int s = 0; s < kClSymbols; ++s) cl_freq[s] = 0;
    cl_tokens(ll_lens, n_ll, d_lens, n_d, [&](int sym, int, int) { cl_freq[sym]++; });
    uint16_t sorted[kClSymbols];
    uint32_t work[kClSymbols];
    uint8_t cl_lens[kClSymbols];
    uint16_t cl_codes[kClSymbols];
    const int m = huff_sort(cl_freq, kClSymbols, sorted);
    huff_lengths_sorted(cl_freq, sorted, m, kClSymbols, kMaxClBits, cl_lens, work);
    huff_codes(cl_lens, kClSymbols, cl_codes);
    int hclen = kClSymbols;
    while (hclen > 4 && cl_lens[kOrder[hclen - 1]] == 0) --hclen;
    bw.put((uint32_t)bfinal, 1);
    bw.put(2u, 2);
    bw.put((uint32_t)(n_ll - 257), 5);
    bw.put((uint32_t)(n_d - 1), 5);
    bw.put((uint32_t)(hclen - 4), 4);
    for (int k = 0; k < hclen; ++k) bw.put(cl_lens[kOrder[k]], 3);
    cl_tokens(ll_lens, n_ll, d_lens, n_d, [&](int sym, int extra, int nextra) {
        bw.put(cl_codes[sym], cl_lens[sym]);
        if (nextra) bw.put((uint32_t)extra, nextra);
    });
}

// ---- tokens -----------------------------------------------------------------------------------------------------
// Match length 3..258 -> literal/length symbol and its extra bits (RFC 1951 section 3.2.5).
AW_PNG_HD void length_symbol(int len, int& sym, int& extra, int& nextra) {
    if (len == 258) { sym = 285; extra = 0; nextra = 0; return; }
    const int v = len - 3;
    if (v < 8) { sym = 257 + v; extra = 0; nextra = 0; return; }
    int lg = 3;
    while ((v >> (lg + 1)) != 0) ++lg;
    nextra = lg - 2;
    sym = 261 + 4 * nextra + ((v >> nextra) - 4);
    extra = v & ((1 << nextra) - 1);
}

// Greedy distance-1 tokens of buf[0..n) (one deflate block: nothing refers to bytes before buf[0]), restricted to
// the token starts that fall in [a, b).  Position i "continues a run" when i > 0 and buf[i] == buf[i-1].  A maximal
// stretch of R such positions starting at s is coded as floor(R / 258) matches of 258 bytes, then one match of
// the remaining r bytes when r >= 3 or r literals when r < 3; every other byte is a literal.  This is what a left
// to right greedy parser with matches at distance 1 only produces, decided from local information so that each
// thread can tokenise its own chunk:
//   prev_break  the largest position < a that does not continue a run (-1 when a == 0: position 0 never does)
//   next_break  the smallest position >= b that does not continue a run (n when there is none)
// emit(literal_byte, -1) for a literal, emit(-1, length) for a match.
template <typename Emit>
AW_PNG_HD void rle_tokens(const uint8_t* buf, int n, int a, int b, int prev_break, int next_break, Emit&& emit) {
    int i = a;
    int brk = prev_break;                       // last position <= i - 1 that does not continue a run
    while (i < b) {
        if (i == 0 || buf[i] != buf[i - 1]) {
            emit((int)buf[i], -1);
            brk = i;
            ++i;
            continue;
        }
        const int s = brk + 1;                  // this stretch of run positions starts at s (s <= i)
        int e = i + 1;
        while (e < b && buf[e] == buf[e - 1]) ++e;
        if (e == b) e = next_break > b ? next_break : b;   // the stretch may go on past the chunk
        const int R = e - s, full = R / 258 * 258, r = R - full;
        const int stop = e < b ? e : b;
        for (int k = i - s; s + k < stop;) {    // token starts inside [i, stop)
            if (k < full) {
                if (k % 258 == 0) { emit(-1, 258); k += 258; }
                else k += 258 - k % 258;        // inside a match that started before a
            } else if (r >= 3) {
                if (k == full) emit(-1, r);
                break;                          // the rest is covered by that match
            } else {
                emit((int)buf[s + k], -1);
                ++k;
            }
        }
        i = stop;                               // no break inside [i, stop): brk stays
    }
}

// ---- Adler-32 ---------------------------------------------------------------------------------------------------
constexpr uint32_t kAdlerMod = 65521;

// Folds a piece of `len` bytes into the running Adler-32 sums (a, b) (a starts at 1, b at 0): seg_a = sum of its
// bytes b_k, seg_b = sum of (len - k) b_k, both mod 65521.
AW_PNG_HD void adler_combine(uint32_t& a, uint32_t& b, uint32_t seg_a, uint32_t seg_b, uint32_t len) {
    b = (uint32_t)(((uint64_t)b + (uint64_t)a * len + seg_b) % kAdlerMod);
    a = (a + seg_a) % kAdlerMod;
}

// ---- CRC-32 (ISO-HDLC, reflected polynomial 0xEDB88320) -------------------------------------------------------------
constexpr uint32_t kCrcPoly = 0xEDB88320u;

// a * b modulo the CRC polynomial, both as reflected polynomials (x^0 is 0x80000000).
AW_PNG_HD uint32_t crc_multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ kCrcPoly : b >> 1;
    }
    return p;
}

// x^(8 * bytes) modulo the polynomial: the operator that moves a CRC past `bytes` zero bytes.
AW_PNG_HD uint32_t crc_shift_operator(uint64_t bytes) {
    uint32_t p = 1u << 31, sq = 1u << 30;       // x^0, x^1
    for (int k = 0; k < 3; ++k) sq = crc_multmodp(sq, sq);   // x^8
    for (; bytes != 0; bytes >>= 1) {
        if (bytes & 1) p = crc_multmodp(sq, p);
        sq = crc_multmodp(sq, sq);
    }
    return p;
}

// crc32(A ++ B) from crc32(A), crc32(B) and the operator of len(B).
AW_PNG_HD uint32_t crc_combine(uint32_t crc_a, uint32_t crc_b, uint32_t op_len_b) {
    return crc_multmodp(op_len_b, crc_a) ^ crc_b;
}

AW_PNG_HD uint32_t crc_update_bitwise(uint32_t crc, const uint8_t* p, int n) {   // crc: running value, ~ applied
    for (int i = 0; i < n; ++i) {
        crc ^= p[i];
        for (int k = 0; k < 8; ++k) crc = (crc & 1) ? (crc >> 1) ^ kCrcPoly : crc >> 1;
    }
    return crc;
}

}  // namespace png
}  // namespace aw
