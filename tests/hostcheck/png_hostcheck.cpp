// TEST-ONLY host harness: compiles attwarp_b200/csrc/png_deflate.h with g++ so that the Huffman builder, the
// dynamic-block header, the chunked tokeniser and the CRC combination the PNG kernels run can be checked against
// zlib on a machine without a GPU.  Never linked into the product.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../attwarp_b200/csrc/png_deflate.h"

using namespace aw::png;

extern "C" {

void hc_huff_lengths(const uint32_t* freq, int n, int max_bits, uint8_t* lens) {
    std::vector<uint16_t> sorted(n);
    std::vector<uint32_t> work(n);
    const int m = huff_sort(freq, n, sorted.data());
    huff_lengths_sorted(freq, sorted.data(), m, n, max_bits, lens, work.data());
}

// One final dynamic-Huffman block of data[0..n) as the kernel builds it, with the tokeniser run over `nchunks`
// equal chunks (the break positions either side of each chunk found the way png.cu finds them).  Returns the
// block's length in bytes; out holds >= 2 n + 1024 bytes.
int hc_deflate_block(const uint8_t* data, int n, int nchunks, uint8_t* out) {
    auto is_break = [&](int i) { return i == 0 || data[i] != data[i - 1]; };
    const int per = (n + nchunks - 1) / nchunks;
    std::vector<int> prev_brk(nchunks), next_brk(nchunks);
    for (int c = 0; c < nchunks; ++c) {
        const int a = c * per < n ? c * per : n, b = a + per < n ? a + per : n;
        int p = a - 1;
        while (p >= 0 && !is_break(p)) --p;
        int q = b;
        while (q < n && !is_break(q)) ++q;
        prev_brk[c] = p;
        next_brk[c] = q;
    }
    uint32_t freq[kLitLenSymbols] = {0};
    auto run_all = [&](auto&& emit) {
        for (int c = 0; c < nchunks; ++c) {
            const int a = c * per < n ? c * per : n, b = a + per < n ? a + per : n;
            rle_tokens(data, n, a, b, prev_brk[c], next_brk[c], emit);
        }
    };
    run_all([&](int lit, int len) {
        if (lit >= 0) {
            freq[lit]++;
        } else {
            int sym, extra, nextra;
            length_symbol(len, sym, extra, nextra);
            freq[sym]++;
        }
    });
    freq[256] = 1;
    uint8_t ll_lens[kLitLenSymbols];
    uint16_t ll_codes[kLitLenSymbols];
    hc_huff_lengths(freq, kLitLenSymbols, kMaxBits, ll_lens);
    huff_codes(ll_lens, kLitLenSymbols, ll_codes);
    const uint8_t d_lens[2] = {1, 1};
    BitWriter bw{out, 0, 0, 0};
    write_dynamic_header(bw, 1, ll_lens, d_lens, 2);
    run_all([&](int lit, int len) {
        if (lit >= 0) {
            bw.put(ll_codes[lit], ll_lens[lit]);
        } else {
            int sym, extra, nextra;
            length_symbol(len, sym, extra, nextra);
            bw.put(ll_codes[sym], ll_lens[sym]);
            if (nextra) bw.put((uint32_t)extra, nextra);
            bw.put(0u, 1);                      // distance code 0 (distance 1)
        }
    });
    bw.put(ll_codes[256], ll_lens[256]);
    bw.flush_partial();
    return (bw.bits() + 7) / 8;
}

// crc32 of data[0..n) from the CRCs of `nchunks` chunks, combined like png.cu combines its threads' CRCs.
uint32_t hc_crc32_chunked(const uint8_t* data, int n, int nchunks) {
    const int per = (n + nchunks - 1) / nchunks;
    uint32_t crc = 0;
    for (int c = 0; c < nchunks; ++c) {
        const int a = c * per < n ? c * per : n, b = a + per < n ? a + per : n;
        const uint32_t part = ~crc_update_bitwise(0xFFFFFFFFu, data + a, b - a);
        crc = crc_combine(crc, part, crc_shift_operator((uint64_t)(b - a)));
    }
    return crc;
}

}  // extern "C"
