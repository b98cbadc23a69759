// dmc_jpeg_color_enc_core.h -- baseline colour JPEG ENCODING primitives shared by the CUDA kernels of dmc_jpeg_color_enc.cu
// and by their lane-by-lane CPU emulation (tests/cpp/jpeg_color_enc_emul.cpp): sampling factors and block geometry, the
// 623-byte header, colour conversion and chroma downsampling, and the samples of one block of the interleaved scan.  The
// transform, quantiser, bit counts, bit packing and byte stuffing are the gray encoder's (dmc_jpeg_enc_core.h).
//
// The target is byte equality with cv2.imencode(".jpg", img, [IMWRITE_JPEG_QUALITY, q, IMWRITE_JPEG_SAMPLING_FACTOR, s])
// of an 8UC3 BGR image (libjpeg-turbo 3.1.2 in cv2 4.13, single-pass coding, no restart intervals).  On top of the gray
// rules, that encoder is fully determined by these (confirmed against cv2 by tests/test_jpeg_color_enc_emul.py):
//   1. Colour conversion (jccolor.c rgb_ycc_convert, BGR input as cv2 passes JCS_EXT_BGR; the SIMD paths give the same
//      bits), FIX(x) = round(x * 2^16):
//        Y  = ( 19595 R + 38470 G +  7471 B + 32768) >> 16
//        Cb = (-11059 R - 21709 G + 32768 B + (128 << 16) + 32767) >> 16
//        Cr = ( 32768 R - 27439 G -  5329 B + (128 << 16) + 32767) >> 16
//   2. Downsampling of Cb and Cr by the luma factors hy x vy (jcsample.c, no smoothing), output column cx:
//        1x1 copies; 2x1 (p0 + p1 + (cx & 1)) >> 1; 2x2 (p00 + p01 + p10 + p11 + 1 + (cx & 1)) >> 2;
//        1x2 and 4x1 (int_downsample) (sum + n / 2) / n.
//   3. Edges.  A component of factors (h, v) is comp_w = ceil(cols h / hy) x comp_h = ceil(rows v / vy) samples, coded in
//      width_in_blocks = ceil(comp_w / 8) x height_in_blocks = ceil(comp_h / 8) blocks.  Horizontally, jcsample.c's
//      expand_right_edge replicates the last INPUT column to width_in_blocks * 8 * (hy / h) columns before downsampling, so
//      every column of a block reads input columns clamped to cols - 1.  Vertically, jcprepct.c replicates the last input
//      row only inside the last row group (vy rows), and below it copies the last DOWNSAMPLED row down to the iMCU height.
//      So a chroma sample (cx, cy) is the downsampling of the input pixels (clamp(hy cx + i, cols - 1),
//      clamp(vy min(cy, comp_h - 1) + j, rows - 1)): reading the input at clamped coordinates alone would be wrong below
//      an even last row pair (the bias depends only on cx, so nothing else differs).  Luma (h = hy, v = vy) reduces to
//      clamped coordinates.
//   4. Block geometry: mcus_x = ceil(cols / (8 hy)) x mcus_y = ceil(rows / (8 vy)) MCUs, each the hy x vy luma blocks in
//      raster order, then one Cb and one Cr block (chroma width_in_blocks = mcus_x, so chroma blocks are always real).
//      Every component has its own DC predictor starting at 0, dummy blocks included; Y codes with tables 0 (K.1, K.3,
//      K.5), Cb and Cr with tables 1 (K.2, K.4, K.6), the quantisation tables scaled by the gray rule.
//   5. Dummy blocks (jccoefct.c compress_data): luma blocks of an MCU at or beyond width_in_blocks / height_in_blocks are
//      not transformed; their AC is zero and their quantised DC is copied, at the right edge from the block to their left,
//      in a bottom dummy row from the MCU's block just before that row.  Both chains end at the same real block: the MCU's
//      last real column in row min(by, height_in_blocks - 1).
//   6. Bound: K.4 has an 11-bit code for DC category 11, so a chroma block takes at most (11 + 11) + 63 (16 + 10) = 1660
//      bits (1658 for luma); a stream is at most 623 + 2 + 2 ceil(blocks 1660 / 8) bytes, dummy blocks included.
// The header (623 bytes) depends only on size, quality and sampling: SOI, APP0, DQT 0 (K.1), DQT 1 (K.2), SOF0 with
// components (1, hy vy, 0) (2, 0x11, 1) (3, 0x11, 1), DHT DC0, AC0, DC1, AC1, SOS.
#pragma once
#include "dmc_jpeg_enc_core.h"

namespace dmcjpeg {

constexpr int kColorEncHeaderBytes = 623;
constexpr uint32_t kColorEncMaxBlockBits = (11 + 11) + 63 * (16 + 10);

// cv2's IMWRITE_JPEG_SAMPLING_FACTOR values -> luma factors (chroma is 1x1); false for any other value.
inline bool color_sampling_factors(int sampling, int* hy, int* vy) {
    switch (sampling) {
        case 0x111111: *hy = 1; *vy = 1; return true;
        case 0x211111: *hy = 2; *vy = 1; return true;
        case 0x221111: *hy = 2; *vy = 2; return true;
        case 0x121111: *hy = 1; *vy = 2; return true;
        case 0x411111: *hy = 4; *vy = 1; return true;
        default: return false;
    }
}

struct ColorEncGeom {
    int rows, cols, hy, vy;
    int mcus_x, mcus_y, ny, bpm;     // MCUs; luma blocks and all blocks per MCU
    int ybw, ybh;                    // luma width_in_blocks / height_in_blocks
    int ch;                          // chroma comp_h
};

DMC_HD ColorEncGeom color_enc_geom(int rows, int cols, int hy, int vy) {
    ColorEncGeom g;
    g.rows = rows; g.cols = cols; g.hy = hy; g.vy = vy;
    g.mcus_x = (cols + 8 * hy - 1) / (8 * hy); g.mcus_y = (rows + 8 * vy - 1) / (8 * vy);
    g.ny = hy * vy; g.bpm = g.ny + 2;
    g.ybw = (cols + 7) / 8; g.ybh = (rows + 7) / 8;
    g.ch = (rows + vy - 1) / vy;
    return g;
}

DMC_HD uint32_t color_enc_blocks(const ColorEncGeom& g) { return (uint32_t)g.mcus_x * (uint32_t)g.mcus_y * (uint32_t)g.bpm; }

inline uint64_t jpeg_encode_color_bound(int rows, int cols, int hy, int vy) {
    const uint64_t blocks = color_enc_blocks(color_enc_geom(rows, cols, hy, vy));
    return (uint64_t)kColorEncHeaderBytes + 2 + 2 * ((blocks * kColorEncMaxBlockBits + 7) / 8);
}

// Tables of both classes (0: Y, 1: Cb and Cr) and the header.
struct EncColorTables {
    uint32_t dc[2][16];
    uint32_t ac[2][256];
    uint32_t qmul[2][64];
    uint32_t qhalf[2][64];
    uint8_t header[kColorEncHeaderBytes];
};

// ---- tables and header (host) -----------------------------------------------------------------------------------------
inline const uint8_t* std_chrominance_quant() {        // ITU T.81 K.2, natural order
    static const uint8_t t[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99,
                                  47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                  99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
    return t;
}
static const uint8_t kStdChromaDcBits[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};            // K.4
static const uint8_t kStdChromaAcBits[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};         // K.6
static const uint8_t kStdChromaAcVals[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08, 0x14, 0x42,
    0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19,
    0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55,
    0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83,
    0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8,
    0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4,
    0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9,
    0xfa};

// The 623 header bytes cv2.imencode writes for an 8UC3 image with luma factors hy x vy.
inline void build_color_header(const uint8_t qy[64], const uint8_t qc[64], int rows, int cols, int hy, int vy, uint8_t* h) {
    uint8_t* p = h;
    memcpy(p, kSoiApp0, 20); p += 20;
    for (int t = 0; t < 2; t++) {
        const uint8_t* q = t ? qc : qy;
        *p++ = 0xFF; *p++ = 0xDB; *p++ = 0x00; *p++ = 0x43; *p++ = (uint8_t)t;
        for (int k = 0; k < 64; k++) *p++ = q[zigzag_to_natural(k)];
    }
    const uint8_t sof[19] = {0xFF, 0xC0, 0x00, 0x11, 0x08, (uint8_t)(rows >> 8), (uint8_t)rows, (uint8_t)(cols >> 8), (uint8_t)cols, 0x03,
                             0x01, (uint8_t)((hy << 4) | vy), 0x00, 0x02, 0x11, 0x01, 0x03, 0x11, 0x01};
    memcpy(p, sof, 19); p += 19;
    for (int t = 0; t < 2; t++) {
        *p++ = 0xFF; *p++ = 0xC4; *p++ = 0x00; *p++ = 0x1F; *p++ = (uint8_t)t;
        memcpy(p, t ? kStdChromaDcBits : kStdDcBits, 16); p += 16; memcpy(p, kStdDcVals, 12); p += 12;
        *p++ = 0xFF; *p++ = 0xC4; *p++ = 0x00; *p++ = 0xB5; *p++ = (uint8_t)(0x10 | t);
        memcpy(p, t ? kStdChromaAcBits : kStdAcBits, 16); p += 16; memcpy(p, t ? kStdChromaAcVals : kStdAcVals, 162); p += 162;
    }
    const uint8_t sos[14] = {0xFF, 0xDA, 0x00, 0x0C, 0x03, 0x01, 0x00, 0x02, 0x11, 0x03, 0x11, 0x00, 0x3F, 0x00};
    memcpy(p, sos, 14);
}

inline void make_enc_color_tables(int quality, int rows, int cols, int hy, int vy, EncColorTables* t) {
    uint8_t qy[64], qc[64];
    scale_quant_table(std_luminance_quant(), quality, qy);
    scale_quant_table(std_chrominance_quant(), quality, qc);
    make_code_table(kStdDcBits, kStdDcVals, t->dc[0], 16);
    make_code_table(kStdAcBits, kStdAcVals, t->ac[0], 256);
    make_code_table(kStdChromaDcBits, kStdDcVals, t->dc[1], 16);
    make_code_table(kStdChromaAcBits, kStdChromaAcVals, t->ac[1], 256);
    for (int i = 0; i < 64; i++) { quant_recip(qy[i], &t->qmul[0][i], &t->qhalf[0][i]); quant_recip(qc[i], &t->qmul[1][i], &t->qhalf[1][i]); }
    build_color_header(qy, qc, rows, cols, hy, vy, t->header);
}

// ---- colour conversion and block samples ------------------------------------------------------------------------------
DMC_HD int enc_min(int a, int b) { return a < b ? a : b; }

// Component c (0 Y, 1 Cb, 2 Cr) of one B, G, R pixel (rule 1; every sum is non-negative, so >> is a floor).
DMC_HD int rgb_to_ycc(int c, int b, int g, int r) {
    if (c == 0) return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
    if (c == 1) return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
    return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

// Block b of the scan (MCU order): its component (the return value), whether it is a dummy block, and the block (bx, by)
// of the component's block grid whose samples it codes -- for a dummy block, the real block its DC is copied from (rule 5).
DMC_HD int color_enc_block(const ColorEncGeom& g, uint32_t b, int* bx, int* by, bool* dummy) {
    const uint32_t mcu = b / (uint32_t)g.bpm, pos = b - mcu * (uint32_t)g.bpm;
    const int mx = (int)(mcu % (uint32_t)g.mcus_x), my = (int)(mcu / (uint32_t)g.mcus_x);
    if (pos >= (uint32_t)g.ny) { *bx = mx; *by = my; *dummy = false; return (int)(pos - (uint32_t)g.ny) + 1; }
    const int x = mx * g.hy + (int)pos % g.hy, y = my * g.vy + (int)pos / g.hy;
    *dummy = x >= g.ybw || y >= g.ybh;
    const int last_real_x = enc_min(mx * g.hy + g.hy - 1, g.ybw - 1);
    *bx = y >= g.ybh ? last_real_x : enc_min(x, g.ybw - 1);
    *by = enc_min(y, g.ybh - 1);
    return 0;
}

// The 64 centred samples (row-major) of block (bx, by) of component c.  px(x, y, &b, &g, &r) reads the input pixel at
// 0 <= x < cols, 0 <= y < rows.
template <class Px>
DMC_HD void color_block_samples(const ColorEncGeom& g, Px px, int c, int bx, int by, int* d) {
    if (c == 0) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const int y = enc_min(by * 8 + r, g.rows - 1);
#pragma unroll
            for (int k = 0; k < 8; k++) {
                int B, G, R;
                px(enc_min(bx * 8 + k, g.cols - 1), y, &B, &G, &R);
                d[r * 8 + k] = rgb_to_ycc(0, B, G, R) - 128;
            }
        }
        return;
    }
    const int n = g.hy * g.vy;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int cy = enc_min(by * 8 + r, g.ch - 1);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int cx = bx * 8 + k;
            int sum = 0;
            for (int j = 0; j < g.vy; j++) {
                const int y = enc_min(cy * g.vy + j, g.rows - 1);
                for (int i = 0; i < g.hy; i++) {
                    int B, G, R;
                    px(enc_min(cx * g.hy + i, g.cols - 1), y, &B, &G, &R);
                    sum += rgb_to_ycc(c, B, G, R);
                }
            }
            int v;
            if (n == 1) v = sum;
            else if (g.vy == 1 && g.hy == 2) v = (sum + (cx & 1)) >> 1;
            else if (g.vy == 2 && g.hy == 2) v = (sum + 1 + (cx & 1)) >> 2;
            else v = (sum + n / 2) / n;
            d[r * 8 + k] = v - 128;
        }
    }
}

// The transform of block b of the scan: samples, islow FDCT, quantisation with the component's table into zz (zigzag
// order) and the block record with the AC bits counted with the component's table.  A dummy block transforms its source
// block, keeps only that block's quantised DC and codes an EOB.  Tables are indexed by class (0 Y, 1 Cb / Cr).
template <class Px>
DMC_HD EncBlock color_transform_block(const ColorEncGeom& g, Px px, uint32_t b, const uint32_t (*qmul)[64], const uint32_t (*qhalf)[64],
                                      const uint32_t (*ac)[256], int16_t* zz) {
    int bx, by; bool dummy;
    const int c = color_enc_block(g, b, &bx, &by, &dummy), t = c > 0 ? 1 : 0;
    int d[64];
    color_block_samples(g, px, c, bx, by, d);
    fdct_islow(d);
    EncBlock e;
    e.nz = quantize_zigzag(d, qmul[t], qhalf[t], zz);
    e.dc = zz[0];
    if (dummy) {
        e.nz = 0; e.ac_bits = code_len(ac[t][0x00]);
#pragma unroll
        for (int k = 1; k < 64; k++) zz[k] = 0;
    } else {
        e.ac_bits = block_ac_bits(zz, ac[t]);
    }
    return e;
}

}  // namespace dmcjpeg
