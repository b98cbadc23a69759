// jpeg_color_emul.cpp -- CPU emulation of the colour JPEG decoder (csrc/dmc_jpeg_color.cu): jpeg_color_frame_kernel's
// phases with the CTA's lanes executed one after the other and the barriers turned into loop boundaries, the one-lane
// decode of restart-interval streams, and the upsampling / colour conversion kernel, all built from the primitives of
// csrc/dmc_jpeg_color_core.h that the kernels use.  Test infrastructure: tests/test_jpeg_color_emul.py checks it against
// cv2.imdecode(buf, IMREAD_COLOR) without a GPU and reads the synchronisation rounds from it.
#include "../../depthmapcompression_b200/csrc/dmc_jpeg_parse.h"

#include <algorithm>

using namespace dmcjpeg;

namespace {

void set_err(char* err, size_t err_len, const std::string& why) {
    if (err && err_len) { strncpy(err, why.c_str(), err_len - 1); err[err_len - 1] = 0; }
}

// Decodes the scan of `stream` into the component planes (color_planes layout); *rounds: synchronisation rounds (0 for
// the restart-interval path).
int decode_planes(const uint8_t* stream, size_t len, int rows, int cols, int lanes, ColorFrameDesc& d, std::vector<uint8_t>& planes, int* rounds_out,
                  char* err, size_t err_len) {
    dmc::JpegTablePools pools;
    std::string why = dmc::jpeg_parse_color_frame(stream, len, 0, rows, cols, pools, &d);
    if (!why.empty()) { set_err(err, err_len, why); return -1; }
    HuffTable tabs[6]; int quant[3][64];
    for (int c = 0; c < 3; c++) {
        tabs[2 * c] = pools.h.items[d.dc[c]]; tabs[2 * c + 1] = pools.h.items[d.ac[c]];
        for (int i = 0; i < 64; i++) quant[c][i] = pools.q.items[d.qt[c]].q[i];
    }
    planes.assign(color_plane_bytes(d), 0xAB);
    const uint32_t nblocks = color_blocks(d);
    const int bpm = color_blocks_per_mcu(d), ny = color_luma_blocks(d);
    auto emit_block = [&](uint32_t blk, int* cf, uint64_t mask) {
        int comp, stride; const uint64_t o = color_block_origin(d, blk, &comp, &stride);
        idct_islow_inplace([cf](int i) -> int& { return cf[i]; }, quant[comp], mask, [&](int r, const uint8_t* row) {
            memcpy(&planes[o + (size_t)r * stride], row, 8);
        });
    };
    if (rounds_out) *rounds_out = 0;
    if (d.restart_interval) {                 // jpeg_color_huff_kernel + jpeg_color_idct_kernel
        std::vector<int16_t> coefs((size_t)nblocks * 64, 0);
        color_decode_serial(stream, d, tabs, coefs.data());
        for (uint32_t b = 0; b < nblocks; b++) {
            int comp, stride; const uint64_t o = color_block_origin(d, b, &comp, &stride);
            uint8_t px[64];
            idct_islow_block(&coefs[(size_t)b * 64], pools.q.items[d.qt[comp]].q, px);
            for (int r = 0; r < 8; r++) memcpy(&planes[o + (size_t)r * stride], px + 8 * r, 8);
        }
        return 0;
    }
    // phase 0: de-stuff up to the first marker, zero padding, big-endian words
    const uint8_t* raw = stream + d.scan_offset; const uint64_t raw_len = d.scan_end - d.scan_offset;
    std::vector<uint8_t> ds;
    for (uint64_t i = 0; i < raw_len; i++) {
        if (raw[i] == 0xFF) { const uint8_t nx = i + 1 < raw_len ? raw[i + 1] : 0xD9; if (nx != 0) break; ds.push_back(0xFF); i++; }
        else ds.push_back(raw[i]);
    }
    const uint32_t L = (uint32_t)ds.size(), last_word = (L + 3) / 4;
    ds.resize(4 * (last_word + 2), 0);
    std::vector<uint32_t> words(last_word + 2);
    for (uint32_t i = 0; i < last_word + 2; i++) words[i] = ((uint32_t)ds[4 * i] << 24) | ((uint32_t)ds[4 * i + 1] << 16) | ((uint32_t)ds[4 * i + 2] << 8) | ds[4 * i + 3];
    // phases 1 and 2
    const uint32_t total_bits = L * 8, S = scan_subseq_bits(total_bits, (uint32_t)lanes);
    const uint32_t nsub = total_bits ? (total_bits + S - 1) / S : 1;
    std::vector<ColorScanState> rec(nsub), st(nsub); std::vector<uint32_t> rec_nb(nsub); std::vector<int32_t> rec_dc(3 * (size_t)nsub);
    std::vector<char> active(nsub, 0);
    for (uint32_t j = 0; j < nsub; j++) {
        st[j].p = j * S; st[j].k = 0; st[j].m = 0;
        color_scan_count(words.data(), last_word, tabs, ny, bpm, st[j], std::min((j + 1) * S, total_bits), &rec_nb[j], &rec_dc[3 * j]);
        rec[j] = st[j];
        active[j] = j + 1 < nsub;
    }
    int rounds = 0;
    for (uint32_t r = 1; std::any_of(active.begin(), active.end(), [](char a) { return a != 0; }); r++, rounds++) {
        for (uint32_t j = 0; j < nsub; j++) {
            if (!active[j]) continue;
            const uint32_t tgt = j + r;
            color_scan_count(words.data(), last_word, tabs, ny, bpm, st[j], std::min((tgt + 1) * S, total_bits), &rec_nb[tgt], &rec_dc[3 * tgt]);
            const bool met = rec[tgt].p == st[j].p && rec[tgt].k == st[j].k && rec[tgt].m == st[j].m;
            rec[tgt] = st[j];
            if (met || tgt + 1 >= nsub) active[j] = 0;
        }
    }
    if (rounds_out) *rounds_out = rounds;
    // phases 3 and 4
    uint32_t blk0 = 0; int32_t pred0[3] = {0, 0, 0};
    for (uint32_t j = 0; j < nsub; j++) {
        ColorScanState s; if (j == 0) { s.p = 0; s.k = 0; s.m = 0; } else s = rec[j - 1];
        const uint32_t hi = j + 1 == nsub ? 0xFFFFFFFFu : (j + 1) * S;
        uint32_t blk = blk0; int pred[3] = {pred0[0], pred0[1], pred0[2]}; int kz, comp;
        int cf[64]; for (int i = 0; i < 64; i++) cf[i] = 0;
        while (s.k != 0 && s.p < hi) color_scan_symbol(words.data(), last_word, tabs, ny, bpm, s, &kz, &comp);
        while (s.k == 0 && s.p < hi && blk < nblocks) {
            const int v = color_scan_symbol(words.data(), last_word, tabs, ny, bpm, s, &kz, &comp);
            pred[comp] += v;
            cf[0] = (int)(int16_t)pred[comp];
            uint64_t mask = 0;
            while (s.k != 0) {
                const int a = color_scan_symbol(words.data(), last_word, tabs, ny, bpm, s, &kz, &comp);
                if (kz > 0) { const int nat = zigzag_to_natural(kz); cf[nat] = a; mask |= 1ull << nat; }
            }
            emit_block(blk, cf, mask);
            if (mask & ~1ull) for (int i = 1; i < 64; i++) cf[i] = 0;
            blk++;
        }
        blk0 += rec_nb[j];
        for (int c = 0; c < 3; c++) pred0[c] += rec_dc[3 * j + c];
    }
    return 0;
}

}  // namespace

// Decodes one stream to rows x cols BGR (out: 3 * rows * cols bytes).  Returns 0, or < 0 with the reason in err.
extern "C" int jpeg_color_emul_decode(const uint8_t* stream, size_t len, int rows, int cols, uint8_t* out, int lanes, int* rounds_out, char* err, size_t err_len) {
    ColorFrameDesc d; std::vector<uint8_t> planes;
    const int rc = decode_planes(stream, len, rows, cols, lanes, d, planes, rounds_out, err, err_len);
    if (rc) return rc;
    YccTables t; make_ycc_tables(&t);
    for (int y = 0; y < rows; y++)
        for (int x = 0; x < cols; x++) color_pixel_bgr(d, planes.data(), t, rows, cols, x, y, out + 3 * ((size_t)y * cols + x));
    return 0;
}

// The component planes of one stream before upsampling: geom = {nc, hy, vy, yw, yh, cw, ch}; planes receives
// yw*yh (+ 2*cw*ch) bytes when cap allows.  Returns the byte count, or < 0 with the reason in err.
extern "C" long jpeg_color_emul_planes(const uint8_t* stream, size_t len, int rows, int cols, uint8_t* planes, size_t cap, int* geom, char* err, size_t err_len) {
    ColorFrameDesc d; std::vector<uint8_t> p; int rounds;
    const int rc = decode_planes(stream, len, rows, cols, 768, d, p, &rounds, err, err_len);
    if (rc) return rc;
    const ColorPlanes pl = color_planes(d);
    const int g[7] = {d.nc, d.hy, d.vy, pl.yw, pl.yh, pl.cw, pl.ch};
    memcpy(geom, g, sizeof g);
    if (p.size() <= cap) memcpy(planes, p.data(), p.size());
    return (long)p.size();
}

// The host restatement of upsampling and conversion applied to given planes (geom as jpeg_color_emul_planes reports it).
extern "C" void jpeg_color_emul_convert(const uint8_t* planes, const int* geom, int rows, int cols, uint8_t* out) {
    ColorFrameDesc d; memset(&d, 0, sizeof d);
    d.nc = geom[0]; d.hy = geom[1]; d.vy = geom[2]; d.mcus_x = geom[5] / 8; d.mcus_y = geom[6] / 8;
    if (d.nc == 1) { d.mcus_x = geom[3] / 8; d.mcus_y = geom[4] / 8; }
    YccTables t; make_ycc_tables(&t);
    for (int y = 0; y < rows; y++)
        for (int x = 0; x < cols; x++) color_pixel_bgr(d, planes, t, rows, cols, x, y, out + 3 * ((size_t)y * cols + x));
}

extern "C" int jpeg_color_emul_probe(const uint8_t* stream, size_t len, int* rows, int* cols, int* nc, char* err, size_t err_len) {
    dmc::JpegTablePools pools; ColorFrameDesc d; int r = 0, c = 0, n = 0;
    std::string why = dmc::jpeg_parse_color_frame(stream, len, 0, -1, -1, pools, &d, &r, &c, &n);
    if (rows) *rows = r;
    if (cols) *cols = c;
    if (nc) *nc = n;
    set_err(err, err_len, why);
    return why.empty() ? 0 : -1;
}

extern "C" void jpeg_color_emul_ycc_tables(int32_t* out /*4 x 256: cr_r, cb_b, cr_g, cb_g*/) {
    YccTables t; make_ycc_tables(&t);
    memcpy(out, &t, sizeof t);
}
