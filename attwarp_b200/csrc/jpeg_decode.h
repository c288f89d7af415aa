// jpeg_decode.h -- the sequential pieces of the baseline JPEG decoder (jpeg.cu), __host__ __device__ so that g++
// checks them on a CPU (tests/hostcheck/jpeg_hostcheck.cpp).  The target is libjpeg-turbo as Pillow calls it
// (Image.open(path).convert('RGB')): JDCT_ISLOW, do_fancy_upsampling = TRUE, so never the merged up-sampler.
//
//   parse_header       marker parser (host): a file -> Header, with a support code (attwarp_jpeg_support)
//   build_derived      BITS/HUFFVAL -> canonical decode tables + a 9-bit lookahead (jdhuff.c's derived table)
//   peek32 / step      one Huffman symbol of the entropy decoder; the decoder state is (bit position, block of
//                      the MCU, coefficient index) -- all three decide what the next bits mean
//   idct_islow         jpeg_idct_islow (jidctint.c) with libjpeg's post-IDCT range-limit table
//   upsample_at        one output sample of a component: jdsample.c's fancy h2v1 / h2v2 / h1v2, int_upsample
//   ycc_to_bgr         ycc_rgb_convert (jdcolor.c): SCALEBITS 16 fixed point
#pragma once

#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define AW_HD __host__ __device__ __forceinline__
#else
#define AW_HD inline
#endif

namespace aw {
namespace jpeg {

constexpr int kMaxComps = 3;
constexpr int kMaxBlocksPerMcu = 10;
constexpr int kLookBits = 9;
constexpr uint64_t kErrState = ~0ull;           // decoder state after an invalid code or a coefficient past 63

// support codes (attwarp_jpeg_support in include/attwarp.h)
enum Support {
    kOk = 0, kNotJpeg = 1, kTruncated = 2, kProgressive = 3, kArithmetic = 4, kOtherProcess = 5, kPrecision = 6,
    kColour = 7, kSampling = 8, kStructure = 9, kBadTable = 10, kSize = 11
};
// per-image device status (attwarp_decode_jpeg's status_out)
// (ordered: the larger code is the cause -- a bad code leaves its interval short of blocks)
enum Status { kStOk = 0, kStShortData = 1, kStBadCode = 2, kStCoefOverflow = 3, kStRestart = 4, kStMarker = 5 };

AW_HD int natural_order(int k) {
    constexpr uint8_t z[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                               41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                               30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return z[k];
}

// ---- file descriptor ------------------------------------------------------------------------------------------
enum Upsample : int8_t { kFull = 0, kH2V1Fancy = 1, kH2V2Fancy = 2, kH1V2Fancy = 3, kReplicate = 4 };

struct Header {
    int32_t support;
    int32_t H, W, ncomp;
    int32_t hmax, vmax;
    int32_t mcus_x, mcus_y;                     // MCU grid (one component: the component's blocks)
    int32_t bpm;                                // blocks per MCU
    int32_t restart;                            // restart interval in MCUs; 0 = none
    int32_t n_intervals;                        // restart intervals in the scan (1 without restart markers)
    uint32_t scan_off, scan_len;                // entropy-coded data: file bytes [scan_off, scan_off + scan_len)
    int32_t comp_h[kMaxComps], comp_v[kMaxComps];
    int32_t comp_dw[kMaxComps], comp_dh[kMaxComps];   // downsampled_width / _height
    int32_t comp_bw[kMaxComps], comp_bh[kMaxComps];   // component plane in blocks
    int32_t comp_q[kMaxComps], comp_dc[kMaxComps], comp_ac[kMaxComps];
    int8_t comp_up[kMaxComps], comp_hf[kMaxComps], comp_vf[kMaxComps];   // up-sampling method and factors
    int8_t blk_comp[kMaxBlocksPerMcu], blk_dx[kMaxBlocksPerMcu], blk_dy[kMaxBlocksPerMcu];
    uint8_t pad_[2];
    uint16_t qt[kMaxComps][64];                  // each component's quantisation table, natural order
    uint8_t hbits[2 * kMaxComps][17];            // the scan's tables: DC of component c at c, AC at kMaxComps + c
    uint8_t hval[2 * kMaxComps][256];
};

// ---- Huffman --------------------------------------------------------------------------------------------------
struct HuffDerived {
    int32_t maxcode[18];                         // largest code of length l, -1 if none; [17] sentinel
    int32_t valoffset[18];
    uint16_t look[1 << kLookBits];               // (length << 8) | symbol for codes of <= kLookBits bits, else 0
    uint8_t huffval[256];
};

// jpeg_make_d_derived_tbl: false for a table libjpeg rejects (over-subscribed, > 256 symbols, DC symbol > 15)
AW_HD bool build_derived(const uint8_t* bits, const uint8_t* vals, bool is_dc, HuffDerived* d) {
    int count = 0;
    for (int l = 1; l <= 16; ++l) count += bits[l];
    if (count > 256) return false;
    int32_t code = 0, p = 0;
    for (int l = 1; l <= 16; ++l) {
        if (bits[l]) {
            d->valoffset[l] = p - code;
            code += bits[l];
            p += bits[l];
            d->maxcode[l] = code - 1;
            if (code >= (1 << l)) return false;         // no code may be all ones
        } else {
            d->maxcode[l] = -1;
            d->valoffset[l] = 0;
        }
        code <<= 1;
    }
    d->maxcode[0] = -1;
    d->valoffset[0] = d->valoffset[17] = 0;
    d->maxcode[17] = 0xFFFFF;
    for (int i = 0; i < 256; ++i) d->huffval[i] = i < count ? vals[i] : 0;
    if (is_dc)
        for (int i = 0; i < count; ++i)
            if (vals[i] > 15) return false;
    for (int e = 0; e < (1 << kLookBits); ++e) {
        uint16_t v = 0;
        for (int l = 1; l <= kLookBits; ++l) {
            const int32_t c = e >> (kLookBits - l);
            if (c <= d->maxcode[l]) {
                v = (uint16_t)((l << 8) | d->huffval[(c + d->valoffset[l]) & 255]);
                break;
            }
        }
        d->look[e] = v;
    }
    return true;
}

// the symbol at the top of `v` (32 bits): its length in bits, 0 for an invalid code
AW_HD int huff_decode(const HuffDerived* d, uint32_t v, int* sym) {
    const uint16_t e = d->look[v >> (32 - kLookBits)];
    if (e) {
        *sym = e & 255;
        return e >> 8;
    }
    for (int l = kLookBits + 1; l <= 16; ++l) {
        const int32_t c = (int32_t)(v >> (32 - l));
        if (c <= d->maxcode[l]) {
            *sym = d->huffval[(c + d->valoffset[l]) & 255];
            return l;
        }
    }
    return 0;
}

// HUFF_EXTEND
AW_HD int extend(int r, int s) { return r < (1 << (s - 1)) ? r + (int)(~0u << s) + 1 : r; }

// 32 bits of the de-stuffed stream from bit `pos`; the bytes from `end_byte` on read as zero
AW_HD uint32_t peek32(const uint8_t* d, uint32_t pos, uint32_t end_byte) {
    const uint32_t b = pos >> 3;
    uint64_t w = 0;
    for (int j = 0; j < 5; ++j) w = (w << 8) | (b + j < end_byte ? d[b + j] : 0u);
    return (uint32_t)(w >> (8 - (pos & 7)));
}

// decoder state: bit position, block of the MCU, coefficient index (0 = the next symbol is a DC difference)
AW_HD uint64_t pack_state(uint32_t pos, int blk, int k) { return ((uint64_t)pos << 16) | ((uint64_t)blk << 8) | (uint64_t)k; }
AW_HD uint32_t state_pos(uint64_t s) { return (uint32_t)(s >> 16); }
AW_HD int state_blk(uint64_t s) { return (int)((s >> 8) & 255); }
AW_HD int state_k(uint64_t s) { return (int)(s & 255); }

// the tables of one scan: per block of the MCU, its DC and AC table
struct ScanTables {
    const HuffDerived* dc[kMaxBlocksPerMcu];
    const HuffDerived* ac[kMaxBlocksPerMcu];
    int bpm;
};

// One Huffman symbol (plus its extra bits) from state s.  Returns the next state, kErrState on an invalid code or
// a coefficient index past 63.  *is_dc / *value / *zz describe what was decoded: a DC difference, or the AC value
// at zig-zag index *zz (value 0 for EOB / ZRL).
AW_HD uint64_t step(const ScanTables& t, const uint8_t* d, uint32_t end_byte, uint64_t s, bool* is_dc, int* value,
                    int* zz) {
    uint32_t pos = state_pos(s);
    int blk = state_blk(s), k = state_k(s);
    const uint32_t v = peek32(d, pos, end_byte);
    int sym = 0;
    *value = 0;
    if (k == 0) {
        const int len = huff_decode(t.dc[blk], v, &sym);
        if (len == 0) return kErrState;
        *is_dc = true;
        *zz = 0;
        if (sym) *value = extend((int)((v << len) >> (32 - sym)), sym);
        pos += len + sym;
        k = 1;
    } else {
        const int len = huff_decode(t.ac[blk], v, &sym);
        if (len == 0) return kErrState;
        *is_dc = false;
        const int r = sym >> 4, sz = sym & 15;
        *zz = 0;
        if (sz) {
            k += r;
            if (k > 63) return kErrState;
            *value = extend((int)((v << len) >> (32 - sz)), sz);
            *zz = k;
            ++k;
            pos += len + sz;
        } else if (r == 15) {
            k += 16;
            if (k > 64) return kErrState;
            pos += len;
        } else {
            k = 64;                                 // EOB
            pos += len;
        }
        if (k == 64) {
            k = 0;
            blk = blk + 1 == t.bpm ? 0 : blk + 1;
        }
    }
    return pack_state(pos, blk, k);
}

// ---- IDCT -----------------------------------------------------------------------------------------------------
// post-IDCT range limit (jdmaster.c prepare_range_limit_table, indexed by x & RANGE_MASK, CENTERJSAMPLE added)
AW_HD uint8_t idct_limit(int x) {
    const int m = x & 1023;
    return (uint8_t)(m < 128 ? m + 128 : m < 512 ? 255 : m < 896 ? 0 : m - 896);
}

// jpeg_idct_islow: coef in natural order, q the quantisation table in natural order; out[8 * r + c]
AW_HD void idct_islow(const int16_t* coef, const uint16_t* q, uint8_t* out) {
    constexpr int CB = 13, P1 = 2;
    constexpr int32_t F0298 = 2446, F0390 = 3196, F0541 = 4433, F0765 = 6270, F0899 = 7373, F1175 = 9633,
                      F1501 = 12299, F1847 = 15137, F1961 = 16069, F2053 = 16819, F2562 = 20995, F3072 = 25172;
    int32_t ws[64];
    for (int c = 0; c < 8; ++c) {
        int32_t z2 = (int32_t)coef[16 + c] * q[16 + c], z3 = (int32_t)coef[48 + c] * q[48 + c];
        int32_t z1 = (z2 + z3) * F0541;
        const int32_t t2 = z1 - z3 * F1847, t3 = z1 + z2 * F0765;
        z2 = (int32_t)coef[c] * q[c];
        z3 = (int32_t)coef[32 + c] * q[32 + c];
        int32_t t0 = (int32_t)((uint32_t)(z2 + z3) << CB), t1 = (int32_t)((uint32_t)(z2 - z3) << CB);
        const int32_t t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
        t0 = (int32_t)coef[56 + c] * q[56 + c];
        t1 = (int32_t)coef[40 + c] * q[40 + c];
        int32_t u2 = (int32_t)coef[24 + c] * q[24 + c], u3 = (int32_t)coef[8 + c] * q[8 + c];
        z1 = t0 + u3;
        z2 = t1 + u2;
        z3 = t0 + u2;
        int32_t z4 = t1 + u3;
        const int32_t z5 = (z3 + z4) * F1175;
        t0 *= F0298;
        t1 *= F2053;
        u2 *= F3072;
        u3 *= F1501;
        z1 *= -F0899;
        z2 *= -F2562;
        z3 = z3 * -F1961 + z5;
        z4 = z4 * -F0390 + z5;
        t0 += z1 + z3;
        t1 += z2 + z4;
        u2 += z2 + z3;
        u3 += z1 + z4;
        constexpr int sh = CB - P1;
        constexpr int32_t rnd = 1 << (sh - 1);
        ws[c] = (t10 + u3 + rnd) >> sh;
        ws[56 + c] = (t10 - u3 + rnd) >> sh;
        ws[8 + c] = (t11 + u2 + rnd) >> sh;
        ws[48 + c] = (t11 - u2 + rnd) >> sh;
        ws[16 + c] = (t12 + t1 + rnd) >> sh;
        ws[40 + c] = (t12 - t1 + rnd) >> sh;
        ws[24 + c] = (t13 + t0 + rnd) >> sh;
        ws[32 + c] = (t13 - t0 + rnd) >> sh;
    }
    for (int r = 0; r < 8; ++r) {
        const int32_t* w = ws + 8 * r;
        int32_t z2 = w[2], z3 = w[6];
        int32_t z1 = (z2 + z3) * F0541;
        const int32_t t2 = z1 - z3 * F1847, t3 = z1 + z2 * F0765;
        int32_t t0 = (int32_t)((uint32_t)(w[0] + w[4]) << CB), t1 = (int32_t)((uint32_t)(w[0] - w[4]) << CB);
        const int32_t t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
        t0 = w[7];
        t1 = w[5];
        int32_t u2 = w[3], u3 = w[1];
        z1 = t0 + u3;
        z2 = t1 + u2;
        z3 = t0 + u2;
        int32_t z4 = t1 + u3;
        const int32_t z5 = (z3 + z4) * F1175;
        t0 *= F0298;
        t1 *= F2053;
        u2 *= F3072;
        u3 *= F1501;
        z1 *= -F0899;
        z2 *= -F2562;
        z3 = z3 * -F1961 + z5;
        z4 = z4 * -F0390 + z5;
        t0 += z1 + z3;
        t1 += z2 + z4;
        u2 += z2 + z3;
        u3 += z1 + z4;
        constexpr int sh = CB + P1 + 3;
        constexpr int32_t rnd = 1 << (sh - 1);
        uint8_t* o = out + 8 * r;
        o[0] = idct_limit((t10 + u3 + rnd) >> sh);
        o[7] = idct_limit((t10 - u3 + rnd) >> sh);
        o[1] = idct_limit((t11 + u2 + rnd) >> sh);
        o[6] = idct_limit((t11 - u2 + rnd) >> sh);
        o[2] = idct_limit((t12 + t1 + rnd) >> sh);
        o[5] = idct_limit((t12 - t1 + rnd) >> sh);
        o[3] = idct_limit((t13 + t0 + rnd) >> sh);
        o[4] = idct_limit((t13 - t0 + rnd) >> sh);
    }
}

// ---- up-sampling and colour -----------------------------------------------------------------------------------
// Output sample (x, y) of a component whose plane (row stride `stride`) holds dw x dh real samples.  The context
// row above row 0 and below row dh - 1 replicates that row; the right edge is at dw, not at the block width.
AW_HD int upsample_at(const uint8_t* p, int stride, int dw, int dh, int mode, int hf, int vf, int x, int y) {
    switch (mode) {
    case kFull:
        return p[(int64_t)y * stride + x];
    case kH2V1Fancy: {
        const uint8_t* r = p + (int64_t)y * stride;
        const int i = x >> 1;
        if ((x & 1) == 0) return i == 0 ? r[0] : (3 * r[i] + r[i - 1] + 1) >> 2;
        return i == dw - 1 ? r[i] : (3 * r[i] + r[i + 1] + 2) >> 2;
    }
    case kH1V2Fancy: {
        const int ry = y >> 1, v = y & 1;
        const int ny = v == 0 ? (ry > 0 ? ry - 1 : 0) : (ry + 1 < dh ? ry + 1 : dh - 1);
        return (3 * p[(int64_t)ry * stride + x] + p[(int64_t)ny * stride + x] + (v == 0 ? 1 : 2)) >> 2;
    }
    case kH2V2Fancy: {
        const int ry = y >> 1, v = y & 1;
        const int ny = v == 0 ? (ry > 0 ? ry - 1 : 0) : (ry + 1 < dh ? ry + 1 : dh - 1);
        const uint8_t* r0 = p + (int64_t)ry * stride;
        const uint8_t* r1 = p + (int64_t)ny * stride;
        const int i = x >> 1;
        const int cs = 3 * r0[i] + r1[i];
        if ((x & 1) == 0) return i == 0 ? (cs * 4 + 8) >> 4 : (cs * 3 + 3 * r0[i - 1] + r1[i - 1] + 8) >> 4;
        return i == dw - 1 ? (cs * 4 + 7) >> 4 : (cs * 3 + 3 * r0[i + 1] + r1[i + 1] + 7) >> 4;
    }
    default:
        return p[(int64_t)(y / vf) * stride + x / hf];
    }
}

AW_HD uint8_t clamp255(int v) { return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v); }

// ycc_rgb_convert; writes B, G, R
AW_HD void ycc_to_bgr(int y, int cb, int cr, uint8_t* bgr) {
    constexpr int SB = 16;
    constexpr int64_t half = (int64_t)1 << (SB - 1);
    constexpr int64_t f1402 = 91881, f1772 = 116130, f0714 = 46802, f0344 = 22554;   // FIX(x) = x * 2^16 + 0.5
    const int64_t xr = cr - 128, xb = cb - 128;
    const int r_off = (int)((f1402 * xr + half) >> SB);
    const int b_off = (int)((f1772 * xb + half) >> SB);
    const int g_off = (int)((-f0714 * xr + -f0344 * xb + half) >> SB);
    bgr[0] = clamp255(y + b_off);
    bgr[1] = clamp255(y + g_off);
    bgr[2] = clamp255(y + r_off);
}

// ---- marker parser (host) -------------------------------------------------------------------------------------
// The entropy-coded data must run to an EOI that ends the file: everything after the scan header up to the last
// two bytes.  A second scan or DNL inside it is found by the device (status kStMarker).
inline int parse_header(const uint8_t* f, size_t n, Header* h) {
    memset(h, 0, sizeof(*h));
    if (n < 4 || f[0] != 0xFF || f[1] != 0xD8) return h->support = kNotJpeg;
    if (n >= ((size_t)1 << 29)) return h->support = kSize;
    uint8_t qdef[4] = {0, 0, 0, 0}, qtab[4][64];
    uint8_t hdef[8] = {0}, hbits[8][17], hval[8][256];
    int comp_id[kMaxComps] = {0}, comp_qsel[kMaxComps] = {0};
    bool sof = false, jfif = false, adobe = false;
    size_t p = 2;
    for (;;) {
        if (p + 2 > n) return h->support = kTruncated;
        if (f[p] != 0xFF) return h->support = kStructure;
        while (p < n && f[p] == 0xFF) ++p;               // fill bytes
        if (p + 3 > n) return h->support = kTruncated;
        const int m = f[p++];
        if (m == 0xD8 || m == 0xD9 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) return h->support = kStructure;
        const size_t len = ((size_t)f[p] << 8) | f[p + 1];
        if (len < 2 || p + len > n) return h->support = kTruncated;
        const uint8_t* s = f + p + 2;
        const size_t sl = len - 2;
        if (m == 0xC0 || m == 0xC1) {
            if (sof || sl < 6) return h->support = sof ? kStructure : kTruncated;
            sof = true;
            if (s[0] != 8) return h->support = kPrecision;
            h->H = (s[1] << 8) | s[2];
            h->W = (s[3] << 8) | s[4];
            h->ncomp = s[5];
            if (h->H == 0 || h->W == 0) return h->support = kSize;      // 0 lines: a DNL marker gives them
            if (h->ncomp != 1 && h->ncomp != 3) return h->support = kColour;
            if (sl < 6 + 3 * (size_t)h->ncomp) return h->support = kTruncated;
            for (int c = 0; c < h->ncomp; ++c) {
                comp_id[c] = s[6 + 3 * c];
                h->comp_h[c] = s[7 + 3 * c] >> 4;
                h->comp_v[c] = s[7 + 3 * c] & 15;
                comp_qsel[c] = s[8 + 3 * c];
                if (h->comp_h[c] < 1 || h->comp_h[c] > 4 || h->comp_v[c] < 1 || h->comp_v[c] > 4 || comp_qsel[c] > 3)
                    return h->support = kBadTable;
            }
        } else if (m == 0xC2 || m == 0xC6 || m == 0xCA || m == 0xCE) {
            return h->support = kProgressive;
        } else if ((m >= 0xC9 && m <= 0xCF) || m == 0xCC) {
            return h->support = kArithmetic;
        } else if (m == 0xC3 || m == 0xC5 || m == 0xC7 || m == 0xDE || m == 0xDF) {
            return h->support = kOtherProcess;
        } else if (m == 0xC4) {
            size_t q = 0;
            while (q < sl) {
                if (q + 17 > sl) return h->support = kTruncated;
                const int tc = s[q] >> 4, th = s[q] & 15;
                if (tc > 1 || th > 3) return h->support = kBadTable;
                const int slot = tc * 4 + th;
                hbits[slot][0] = 0;
                int cnt = 0;
                for (int l = 1; l <= 16; ++l) cnt += hbits[slot][l] = s[q + l];
                if (cnt > 256 || q + 17 + cnt > sl) return h->support = cnt > 256 ? kBadTable : kTruncated;
                memcpy(hval[slot], s + q + 17, (size_t)cnt);
                hdef[slot] = 1;
                q += 17 + cnt;
            }
        } else if (m == 0xDB) {
            size_t q = 0;
            while (q < sl) {
                const int pq = s[q] >> 4, tq = s[q] & 15;
                if (pq != 0) return h->support = kPrecision;
                if (tq > 3) return h->support = kBadTable;
                if (q + 65 > sl) return h->support = kTruncated;
                for (int k = 0; k < 64; ++k) qtab[tq][natural_order(k)] = s[q + 1 + k];
                qdef[tq] = 1;
                q += 65;
            }
        } else if (m == 0xDD) {
            if (sl < 2) return h->support = kTruncated;
            h->restart = (s[0] << 8) | s[1];
        } else if (m == 0xE0) {
            if (sl >= 5 && memcmp(s, "JFIF\0", 5) == 0) jfif = true;
        } else if (m == 0xEE) {
            if (sl >= 5 && memcmp(s, "Adobe", 5) == 0) adobe = true;
        } else if ((m >= 0xE1 && m <= 0xEF) || m == 0xFE) {
            // APPn / COM: skipped
        } else if (m == 0xDA) {
            if (!sof) return h->support = kStructure;
            if (sl < 1 || sl < 1 + 2 * (size_t)s[0] + 3) return h->support = kTruncated;
            const int ns = s[0];
            if (ns != h->ncomp) return h->support = kStructure;          // one scan holding every component
            for (int j = 0; j < ns; ++j) {
                const int c = j;
                if (s[1 + 2 * j] != comp_id[c]) return h->support = kStructure;
                const int td = s[2 + 2 * j] >> 4, ta = s[2 + 2 * j] & 15;
                if (td > 3 || ta > 3 || !hdef[td] || !hdef[4 + ta]) return h->support = kBadTable;
                h->comp_dc[c] = td;
                h->comp_ac[c] = ta;
                memcpy(h->hbits[c], hbits[td], 17);
                memcpy(h->hval[c], hval[td], 256);
                memcpy(h->hbits[kMaxComps + c], hbits[4 + ta], 17);
                memcpy(h->hval[kMaxComps + c], hval[4 + ta], 256);
            }
            const uint8_t* e = s + 1 + 2 * ns;
            if (e[0] != 0 || e[1] != 63 || e[2] != 0) return h->support = kProgressive;
            h->scan_off = (uint32_t)(p + len);
            break;
        } else {
            return h->support = kStructure;                            // DNL, DHP, EXP, JPGn, ...
        }
        p += len;
    }
    if (n < h->scan_off + 2 || f[n - 2] != 0xFF || f[n - 1] != 0xD9) return h->support = kStructure;
    h->scan_len = (uint32_t)(n - 2 - h->scan_off);
    for (int c = 0; c < h->ncomp; ++c) {
        if (!qdef[comp_qsel[c]]) return h->support = kBadTable;
        h->comp_q[c] = comp_qsel[c];
        for (int k = 0; k < 64; ++k) h->qt[c][k] = qtab[comp_qsel[c]][k];
    }
    for (int c = 0; c < h->ncomp; ++c) {
        HuffDerived d;
        if (!build_derived(h->hbits[c], h->hval[c], true, &d) ||
            !build_derived(h->hbits[kMaxComps + c], h->hval[kMaxComps + c], false, &d))
            return h->support = kBadTable;
    }
    if (h->ncomp == 3) {
        if (!jfif && (adobe || comp_id[0] != 1 || comp_id[1] != 2 || comp_id[2] != 3)) return h->support = kColour;
        const int lh = h->comp_h[0], lv = h->comp_v[0];
        const bool ok = h->comp_h[1] == 1 && h->comp_v[1] == 1 && h->comp_h[2] == 1 && h->comp_v[2] == 1 &&
                        ((lh == 1 && lv == 1) || (lh == 2 && lv == 1) || (lh == 2 && lv == 2) ||
                         (lh == 1 && lv == 2) || (lh == 4 && lv == 1));
        if (!ok) return h->support = kSampling;
        h->hmax = lh;
        h->vmax = lv;
        h->mcus_x = (h->W + 8 * lh - 1) / (8 * lh);
        h->mcus_y = (h->H + 8 * lv - 1) / (8 * lv);
        int b = 0;
        for (int c = 0; c < 3; ++c) {
            h->comp_dw[c] = (h->W * h->comp_h[c] + lh - 1) / lh;
            h->comp_dh[c] = (h->H * h->comp_v[c] + lv - 1) / lv;
            h->comp_bw[c] = h->mcus_x * h->comp_h[c];
            h->comp_bh[c] = h->mcus_y * h->comp_v[c];
            for (int dy = 0; dy < h->comp_v[c]; ++dy)
                for (int dx = 0; dx < h->comp_h[c]; ++dx, ++b) {
                    h->blk_comp[b] = (int8_t)c;
                    h->blk_dx[b] = (int8_t)dx;
                    h->blk_dy[b] = (int8_t)dy;
                }
            const int hf = lh / h->comp_h[c], vf = lv / h->comp_v[c];
            h->comp_hf[c] = (int8_t)hf;
            h->comp_vf[c] = (int8_t)vf;
            // jdsample.c: fancy h2v1 / h2v2 only for downsampled_width > 2, else plain replication
            h->comp_up[c] = hf == 1 && vf == 1                        ? kFull
                            : hf == 2 && vf == 1 && h->comp_dw[c] > 2 ? kH2V1Fancy
                            : hf == 2 && vf == 2 && h->comp_dw[c] > 2 ? kH2V2Fancy
                            : hf == 1 && vf == 2                      ? kH1V2Fancy
                                                                      : kReplicate;
        }
        h->bpm = b;
    } else {                                                           // one component: non-interleaved, 1 block MCUs
        h->hmax = h->vmax = 1;
        h->comp_h[0] = h->comp_v[0] = 1;
        h->comp_dw[0] = h->W;
        h->comp_dh[0] = h->H;
        h->mcus_x = h->comp_bw[0] = (h->W + 7) / 8;
        h->mcus_y = h->comp_bh[0] = (h->H + 7) / 8;
        h->comp_up[0] = kFull;
        h->comp_hf[0] = h->comp_vf[0] = 1;
        h->bpm = 1;
    }
    const int64_t mcus = (int64_t)h->mcus_x * h->mcus_y;
    h->n_intervals = h->restart ? (int32_t)((mcus + h->restart - 1) / h->restart) : 1;
    return h->support = kOk;
}

// MCUs of restart interval i
AW_HD int64_t interval_mcus(const Header& h, int64_t i) {
    const int64_t mcus = (int64_t)h.mcus_x * h.mcus_y;
    if (!h.restart) return mcus;
    const int64_t rest = mcus - i * h.restart;
    return rest < h.restart ? rest : h.restart;
}

// plane position of block q (in decode order) of restart interval i: component, block row, block column
AW_HD void block_place(const Header& h, int64_t i, int64_t q, int* comp, int* brow, int* bcol) {
    const int64_t mcu = i * (h.restart ? h.restart : 0) + q / h.bpm;
    const int b = (int)(q % h.bpm);
    const int mr = (int)(mcu / h.mcus_x), mc = (int)(mcu % h.mcus_x);
    const int c = h.blk_comp[b];
    *comp = c;
    *brow = mr * h.comp_v[c] + h.blk_dy[b];
    *bcol = mc * h.comp_h[c] + h.blk_dx[b];
}

}  // namespace jpeg
}  // namespace aw
