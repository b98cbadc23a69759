// jpeg_enc_emul.cpp -- CPU emulation of the JPEG encoder kernels (csrc/dmc_jpeg_enc.cu): the same phases, built from the
// same host/device primitives of csrc/dmc_jpeg_enc_core.h, with a CTA's lanes executed one after the other and the
// barriers turned into loop boundaries.  Test infrastructure: it lets the CPU test suite check the transform, the bit
// offsets of the lanes, the word packing with shared boundary words and the byte stuffing against cv2.imencode without a
// GPU.  Built by tests/test_jpeg_enc_emul.py with g++.
#include "../../depthmapcompression_b200/csrc/dmc_jpeg_enc_core.h"

#include <algorithm>
#include <vector>

using namespace dmcjpeg;

namespace {

// jpeg_enc_transform_kernel for one block
EncBlock transform_block(const uint8_t* img, int rows, int cols, int bx, int by, const EncTables& t, int16_t* zz) {
    int d[64];
    for (int r = 0; r < 8; r++) {
        const uint8_t* row = img + (size_t)std::min(by * 8 + r, rows - 1) * cols;
        for (int c = 0; c < 8; c++) d[r * 8 + c] = (int)row[std::min(bx * 8 + c, cols - 1)] - 128;
    }
    fdct_islow(d);
    EncBlock e;
    e.nz = quantize_zigzag(d, t.qmul, t.qhalf, zz);
    e.ac_bits = block_ac_bits(zz, t.ac);
    e.dc = zz[0];
    return e;
}

const uint32_t kUntouched = 0xA5A5A5A5u;

}  // namespace

// Encodes one rows x cols 8UC1 image with `lanes` emulated lanes.  Returns the stream length, or a negative number on an
// ownership violation of the packed words (-1) or when the stream does not fit into `cap` bytes (-2).
extern "C" long long jpeg_enc_emul(const uint8_t* img, int rows, int cols, int quality, int lanes, uint8_t* out, unsigned long long cap) {
    EncTables t;
    make_enc_tables(quality, rows, cols, &t);
    const int bw = (cols + 7) / 8, nb = bw * ((rows + 7) / 8);
    std::vector<int16_t> coefs((size_t)nb * 64);
    std::vector<EncBlock> info(nb);
    for (int b = 0; b < nb; b++) info[b] = transform_block(img, rows, cols, b % bw, b / bw, t, &coefs[(size_t)b * 64]);

    // entropy stage: lane j codes blocks [j * per, (j + 1) * per)
    const int per = (nb + lanes - 1) / lanes;
    std::vector<uint32_t> bits(lanes, 0), start(lanes, 0);
    for (int j = 0; j < lanes; j++) {
        const int b0 = std::min(j * per, nb), b1 = std::min(b0 + per, nb);
        int prev = b0 > 0 ? info[b0 - 1].dc : 0;
        for (int b = b0; b < b1; b++) { bits[j] += info[b].ac_bits + block_dc_bits(info[b].dc - prev, t.dc); prev = info[b].dc; }
    }
    uint32_t T = 0;
    for (int j = 0; j < lanes; j++) { start[j] = T; T += bits[j]; }
    const uint64_t max_bits = (uint64_t)nb * kEncMaxBlockBits;
    if (T > max_bits) return -3;
    std::vector<uint32_t> words(max_bits / 32 + 2, kUntouched);
    for (int j = 0; j < lanes; j++) {                   // zero the words a lane shares with its neighbours
        const uint32_t B = start[j], E = B + bits[j];
        if (B & 31) words[B >> 5] = 0;
        if (E & 31) words[E >> 5] = 0;
    }
    bool violation = false;
    for (int j = 0; j < lanes; j++) {
        const int b0 = std::min(j * per, nb), b1 = std::min(b0 + per, nb);
        auto sink = [&](uint32_t wi, uint32_t v, bool partial) {
            if (partial) { if (words[wi] == kUntouched) violation = true; words[wi] |= v; }
            else { if (words[wi] != kUntouched) violation = true; words[wi] = v; }
        };
        auto w = bw_start(start[j], sink);
        int prev = b0 > 0 ? info[b0 - 1].dc : 0;
        for (int b = b0; b < b1; b++) {
            const int16_t* zz = &coefs[(size_t)b * 64];
            emit_block(w, info[b].dc - prev, info[b].nz, [zz](int k) { return (int)zz[k]; }, t.dc, t.ac);
            prev = info[b].dc;
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
        std::vector<uint32_t> cnt(lanes), off(lanes);
        uint32_t tile_total = 0;
        for (int j = 0; j < lanes; j++) {
            const uint32_t i0 = (uint32_t)(t0 + 16ull * j); uint32_t wv[4];
            stuff_load(words.data(), L, i0, wv);
            cnt[j] = i0 < L ? stuff_count(wv, L, i0) : 0;
            off[j] = tile_total; tile_total += cnt[j];
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
    const uint64_t len = (uint64_t)kEncHeaderBytes + scan.size() + 2;
    if (len > jpeg_encode_bound(rows, cols)) return -4;
    if (len > cap) return -2;
    memcpy(out, t.header, kEncHeaderBytes);
    memcpy(out + kEncHeaderBytes, scan.data(), scan.size());
    out[len - 2] = 0xFF; out[len - 1] = 0xD9;
    return (long long)len;
}

extern "C" unsigned long long jpeg_enc_bound(int rows, int cols) { return jpeg_encode_bound(rows, cols); }

// Quantiser proof: the multiply-high of quant_div against the division, for every |x| < 2^15 and every Q in 1..255.
// Returns the number of mismatches.
extern "C" long long jpeg_enc_check_quant(void) {
    long long bad = 0;
    for (int q = 1; q <= 255; q++) {
        uint32_t qmul, qhalf;
        quant_recip((uint32_t)q, &qmul, &qhalf);
        for (int x = -32767; x <= 32767; x++) {
            const int a = x < 0 ? -x : x, want = (x < 0 ? -1 : 1) * (int)((a + 4 * q) / (8 * q));
            if (quant_div(x, qmul, qhalf) != want) bad++;
        }
    }
    return bad;
}
