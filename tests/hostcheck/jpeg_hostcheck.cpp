// TEST-ONLY host harness: compiles attwarp_b200/csrc/jpeg_decode.h with g++ and runs a whole sequential decode
// through it (parser, Huffman tables and symbol steps, ISLOW IDCT, up-sampling, colour conversion), so that the
// pieces the JPEG kernels run can be checked against Pillow on a machine without a GPU.  De-stuffing and the RSTn
// split are done here sequentially.  Never linked into the product.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../attwarp_b200/csrc/jpeg_decode.h"

using namespace aw::jpeg;

extern "C" {

// info[0..3] = H, W, components, support code
int hc_jpeg_probe(const uint8_t* f, size_t n, int32_t* info) {
    Header h;
    const int s = parse_header(f, n, &h);
    info[0] = h.H;
    info[1] = h.W;
    info[2] = h.ncomp;
    info[3] = s;
    return s;
}

// Sequential decode into out (H * W * 3 BGR).  Returns the support code (> 0) of an unsupported file, the negated
// device status code (< 0) of malformed entropy data, 0 on success.  max_dequant (nullable) receives the largest
// |coefficient x quantisation step| of the file.
int hc_jpeg_decode(const uint8_t* f, size_t n, uint8_t* out, int32_t* max_dequant) {
    if (max_dequant) *max_dequant = 0;
    Header h;
    if (parse_header(f, n, &h) != kOk) return h.support;
    // de-stuff, split at RSTn
    std::vector<uint8_t> d;
    std::vector<uint32_t> starts{0};
    const uint8_t* s = f + h.scan_off;
    for (uint32_t i = 0; i < h.scan_len; ++i) {
        const uint8_t b = s[i];
        const int next = i + 1 < h.scan_len ? s[i + 1] : 0xFF;
        if (b == 0xFF) {
            if (next == 0x00) {
                d.push_back(0xFF);
                ++i;
            } else if (next >= 0xD0 && next <= 0xD7) {
                if ((int)starts.size() >= h.n_intervals || next - 0xD0 != (int)((starts.size() - 1) & 7))
                    return -kStRestart;
                starts.push_back((uint32_t)d.size());
                ++i;
            } else if (next != 0xFF) {
                return -kStMarker;
            }
        } else {
            d.push_back(b);
        }
    }
    if ((int)starts.size() != h.n_intervals) return -kStRestart;
    starts.push_back((uint32_t)d.size());
    d.resize(d.size() + 8, 0);

    HuffDerived tabs[2 * kMaxComps];
    for (int c = 0; c < h.ncomp; ++c) {
        build_derived(h.hbits[c], h.hval[c], true, &tabs[c]);
        build_derived(h.hbits[kMaxComps + c], h.hval[kMaxComps + c], false, &tabs[kMaxComps + c]);
    }
    ScanTables st;
    st.bpm = h.bpm;
    for (int b = 0; b < h.bpm; ++b) {
        st.dc[b] = &tabs[h.blk_comp[b]];
        st.ac[b] = &tabs[kMaxComps + h.blk_comp[b]];
    }
    std::vector<std::vector<uint8_t>> planes(h.ncomp);
    for (int c = 0; c < h.ncomp; ++c) planes[c].assign((size_t)h.comp_bw[c] * 8 * h.comp_bh[c] * 8, 0);
    for (int iv = 0; iv < h.n_intervals; ++iv) {
        const uint32_t end_byte = starts[iv + 1];
        uint64_t state = pack_state(starts[iv] * 8, 0, 0);
        int pred[kMaxComps] = {0, 0, 0};
        const int64_t nblk = interval_mcus(h, iv) * h.bpm;
        for (int64_t q = 0; q < nblk; ++q) {
            int16_t coef[64];
            memset(coef, 0, sizeof(coef));
            int comp, brow, bcol;
            block_place(h, iv, q, &comp, &brow, &bcol);
            do {
                bool is_dc;
                int value, zz;
                state = step(st, d.data(), end_byte, state, &is_dc, &value, &zz);
                if (state == kErrState) return -kStBadCode;
                if (is_dc) {
                    pred[comp] += value;
                    coef[0] = (int16_t)pred[comp];
                } else if (zz) {
                    coef[natural_order(zz)] = (int16_t)value;
                }
            } while (state_k(state) != 0);
            if (state_pos(state) > end_byte * 8) return -kStShortData;
            if (max_dequant)
                for (int k = 0; k < 64; ++k) {
                    const int32_t v = coef[k] * (int32_t)h.qt[comp][k];
                    if ((v < 0 ? -v : v) > *max_dequant) *max_dequant = v < 0 ? -v : v;
                }
            uint8_t px[64];
            idct_islow(coef, h.qt[comp], px);
            const int stride = h.comp_bw[comp] * 8;
            for (int r = 0; r < 8; ++r)
                memcpy(&planes[comp][(size_t)(brow * 8 + r) * stride + bcol * 8], px + 8 * r, 8);
        }
    }
    for (int y = 0; y < h.H; ++y)
        for (int x = 0; x < h.W; ++x) {
            uint8_t* o = out + ((size_t)y * h.W + x) * 3;
            int v[kMaxComps];
            for (int c = 0; c < h.ncomp; ++c)
                v[c] = upsample_at(planes[c].data(), h.comp_bw[c] * 8, h.comp_dw[c], h.comp_dh[c], h.comp_up[c],
                                   h.comp_hf[c], h.comp_vf[c], x, y);
            if (h.ncomp == 1)
                o[0] = o[1] = o[2] = (uint8_t)v[0];
            else
                ycc_to_bgr(v[0], v[1], v[2], o);
        }
    return 0;
}

}  // extern "C"
