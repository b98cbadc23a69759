// jpeg_color_enc_emul.cpp -- CPU emulation of the colour JPEG encoder kernels (csrc/dmc_jpeg_color_enc.cu): the same
// phases, built from the same host/device primitives of csrc/dmc_jpeg_color_enc_core.h and csrc/dmc_jpeg_enc_core.h, with
// a CTA's lanes executed one after the other and the barriers turned into loop boundaries.  Test infrastructure: it lets
// the CPU test suite confirm the colour rules (conversion, downsampling, edges, dummy blocks, interleaved MCUs with two
// table sets) and the lanes' MCU runs against cv2.imencode without a GPU.  Built by tests/test_jpeg_color_enc_emul.py.
#include "../../depthmapcompression_b200/csrc/dmc_jpeg_color_enc_core.h"

#include <algorithm>
#include <vector>

using namespace dmcjpeg;

namespace {
const uint32_t kUntouched = 0xA5A5A5A5u;
}

// Encodes one rows x cols 8UC3 BGR image with `lanes` emulated lanes.  Returns the stream length, or a negative number:
// -1 an ownership violation of the packed words, -2 the stream does not fit into `cap`, -3 more bits than the bound
// allows, -4 a stream over the bound, -5 an unknown sampling.
extern "C" long long jpeg_color_enc_emul(const uint8_t* img, int rows, int cols, int quality, int sampling, int lanes, uint8_t* out, unsigned long long cap) {
    int hy, vy;
    if (!color_sampling_factors(sampling, &hy, &vy)) return -5;
    EncColorTables t;
    make_enc_color_tables(quality, rows, cols, hy, vy, &t);
    const ColorEncGeom g = color_enc_geom(rows, cols, hy, vy);
    const uint32_t nb = color_enc_blocks(g), bpm = (uint32_t)g.bpm, nm = nb / bpm;
    auto px = [img, cols](int x, int y, int* B, int* G, int* R) {
        const uint8_t* p = img + ((size_t)y * cols + x) * 3;
        *B = p[0]; *G = p[1]; *R = p[2];
    };
    // transform: one "thread" per block in scan order
    std::vector<int16_t> coefs((size_t)nb * 64);
    std::vector<EncBlock> info(nb);
    for (uint32_t b = 0; b < nb; b++) info[b] = color_transform_block(g, px, b, t.qmul, t.qhalf, t.ac, &coefs[(size_t)b * 64]);

    // entropy stage: lane j codes MCUs [j * per, (j + 1) * per); its predictors start from the previous MCU's blocks
    const uint32_t per = (nm + lanes - 1) / lanes;
    auto preds = [&](uint32_t m0, int* p) {
        for (int c = 0; c < 3; c++) p[c] = m0 > 0 ? info[m0 * bpm - 3 + c].dc : 0;
    };
    std::vector<uint32_t> bits(lanes, 0), start(lanes, 0);
    for (int j = 0; j < lanes; j++) {
        const uint32_t m0 = std::min(j * per, nm), m1 = std::min(m0 + per, nm);
        int pred[3]; preds(m0, pred);
        for (uint32_t b = m0 * bpm, pos = 0; b < m1 * bpm; b++, pos = pos + 1 == bpm ? 0 : pos + 1) {
            const int c = pos < (uint32_t)g.ny ? 0 : (int)(pos - g.ny) + 1;
            bits[j] += info[b].ac_bits + block_dc_bits(info[b].dc - pred[c], t.dc[c > 0]);
            pred[c] = info[b].dc;
        }
    }
    uint32_t T = 0;
    for (int j = 0; j < lanes; j++) { start[j] = T; T += bits[j]; }
    const uint64_t max_bits = (uint64_t)nb * kColorEncMaxBlockBits;
    if (T > max_bits) return -3;
    std::vector<uint32_t> words(max_bits / 32 + 2, kUntouched);
    for (int j = 0; j < lanes; j++) {
        const uint32_t B = start[j], E = B + bits[j];
        if (B & 31) words[B >> 5] = 0;
        if (E & 31) words[E >> 5] = 0;
    }
    bool violation = false;
    for (int j = 0; j < lanes; j++) {
        const uint32_t m0 = std::min(j * per, nm), m1 = std::min(m0 + per, nm);
        auto sink = [&](uint32_t wi, uint32_t v, bool partial) {
            if (partial) { if (words[wi] == kUntouched) violation = true; words[wi] |= v; }
            else { if (words[wi] != kUntouched) violation = true; words[wi] = v; }
        };
        auto w = bw_start(start[j], sink);
        int pred[3]; preds(m0, pred);
        for (uint32_t b = m0 * bpm, pos = 0; b < m1 * bpm; b++, pos = pos + 1 == bpm ? 0 : pos + 1) {
            const int c = pos < (uint32_t)g.ny ? 0 : (int)(pos - g.ny) + 1, k = c > 0;
            const int16_t* zz = &coefs[(size_t)b * 64];
            emit_block(w, info[b].dc - pred[c], info[b].nz, [zz](int i) { return (int)zz[i]; }, t.dc[k], t.ac[k]);
            pred[c] = info[b].dc;
        }
        bw_finish(w);
    }
    if (violation) return -1;
    pad_scan(words.data(), T);

    // stuffing: tiles of 16 bytes per lane, exclusive scan of the 0xFF counts
    const uint32_t L = (T + 7) / 8;
    std::vector<uint8_t> scan;
    uint64_t out_base = 0;
    for (uint64_t t0 = 0; t0 < L; t0 += 16ull * lanes) {
        std::vector<uint32_t> off(lanes);
        uint32_t tile_total = 0;
        for (int j = 0; j < lanes; j++) {
            const uint32_t i0 = (uint32_t)(t0 + 16ull * j); uint32_t wv[4];
            stuff_load(words.data(), L, i0, wv);
            off[j] = tile_total; tile_total += i0 < L ? stuff_count(wv, L, i0) : 0;
        }
        scan.resize(scan.size() + std::min<uint64_t>(16ull * lanes, L - t0) + tile_total);
        for (int j = 0; j < lanes; j++) {
            const uint32_t i0 = (uint32_t)(t0 + 16ull * j); uint32_t wv[4];
            if (i0 >= L) continue;
            stuff_load(words.data(), L, i0, wv);
            stuff_write(wv, L, i0, scan.data() + i0 + out_base + off[j]);
        }
        out_base += tile_total;
    }
    const uint64_t len = (uint64_t)kColorEncHeaderBytes + scan.size() + 2;
    if (len > jpeg_encode_color_bound(rows, cols, hy, vy)) return -4;
    if (len > cap) return -2;
    memcpy(out, t.header, kColorEncHeaderBytes);
    memcpy(out + kColorEncHeaderBytes, scan.data(), scan.size());
    out[len - 2] = 0xFF; out[len - 1] = 0xD9;
    return (long long)len;
}

// Worst-case stream bytes, 0 for an unknown sampling.
extern "C" unsigned long long jpeg_color_enc_bound(int rows, int cols, int sampling) {
    int hy, vy;
    return color_sampling_factors(sampling, &hy, &vy) ? jpeg_encode_color_bound(rows, cols, hy, vy) : 0;
}

// The header bytes (kColorEncHeaderBytes) into out; returns their count, or -5 for an unknown sampling.
extern "C" int jpeg_color_enc_header(int quality, int rows, int cols, int sampling, uint8_t* out) {
    int hy, vy;
    if (!color_sampling_factors(sampling, &hy, &vy)) return -5;
    EncColorTables t;
    make_enc_color_tables(quality, rows, cols, hy, vy, &t);
    memcpy(out, t.header, kColorEncHeaderBytes);
    return kColorEncHeaderBytes;
}
