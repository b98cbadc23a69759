// dmc_jpeg_color_core.h -- baseline colour JPEG decoding primitives shared by the CUDA kernels of dmc_jpeg_color.cu and by
// the CPU emulation of tests/cpp/jpeg_color_emul.cpp: the frame descriptor and its MCU geometry, the interleaved-MCU
// extension of the self-synchronising scan decoder of dmc_jpeg_core.h, the one-lane decode of restart-interval streams,
// and libjpeg-turbo's fancy upsampling (jdsample.c) and YCbCr -> BGR conversion (jdcolor.c) as cv2.imdecode(buf,
// IMREAD_COLOR) runs them.  The rules were confirmed against cv2 4.13 (libjpeg-turbo 3.1.2) by the emulation tests.
#pragma once
#include "dmc_jpeg_core.h"

namespace dmcjpeg {

// One colour (or one-component) frame.  Components are Y, Cb, Cr in frame order; chroma is sampled 1x1 and luma hy x vy
// (1x1, 2x1, 2x2, 1x2 or 4x1).  A one-component frame has nc = 1 and hy = vy = 1 (its MCU is one block whatever its
// sampling factors say, as in libjpeg's non-interleaved scans).
struct ColorFrameDesc {
    uint64_t scan_offset;    // offset of the entropy-coded segment inside the blob
    uint64_t scan_end;       // one past the last byte of this frame's stream
    uint64_t ds_offset;      // de-stuffed copy of the scan inside the scan scratch (16-aligned)
    uint64_t plane_offset;   // component planes (Y, then Cb and Cr) inside the plane scratch (64-aligned)
    uint64_t coef_offset;    // restart-interval frames: first block of the frame inside the coefficient scratch
    int32_t restart_interval;
    int32_t nc, hy, vy;
    int32_t mcus_x, mcus_y;
    int32_t qt[3], dc[3], ac[3];   // per component: indices into the de-duplicated table arrays
    int32_t pad;
};

// libjpeg's ycc_rgb_convert tables (jdcolor.c build_ycc_rgb_table, SCALEBITS 16), indexed by the chroma sample.
struct YccTables { int32_t cr_r[256], cb_b[256], cr_g[256], cb_g[256]; };

inline void make_ycc_tables(YccTables* t) {
    auto fix = [](double x) { return (int32_t)(x * 65536.0 + 0.5); };
    for (int i = 0; i < 256; i++) {
        const int32_t x = i - 128;
        t->cr_r[i] = (fix(1.40200) * x + (1 << 15)) >> 16;
        t->cb_b[i] = (fix(1.77200) * x + (1 << 15)) >> 16;
        t->cr_g[i] = -fix(0.71414) * x;
        t->cb_g[i] = -fix(0.34414) * x + (1 << 15);
    }
}

DMC_HD int color_luma_blocks(const ColorFrameDesc& d) { return d.hy * d.vy; }
DMC_HD int color_blocks_per_mcu(const ColorFrameDesc& d) { return d.nc == 1 ? 1 : d.hy * d.vy + 2; }
DMC_HD uint32_t color_blocks(const ColorFrameDesc& d) { return (uint32_t)d.mcus_x * (uint32_t)d.mcus_y * (uint32_t)color_blocks_per_mcu(d); }

// Plane geometry: every plane is padded to the MCU grid.  Y is (mcus_y*vy*8) x (mcus_x*hy*8), Cb and Cr (mcus_y*8) x (mcus_x*8).
struct ColorPlanes { int yw, yh, cw, ch; };
DMC_HD ColorPlanes color_planes(const ColorFrameDesc& d) {
    ColorPlanes p; p.yw = d.mcus_x * d.hy * 8; p.yh = d.mcus_y * d.vy * 8; p.cw = d.mcus_x * 8; p.ch = d.mcus_y * 8;
    return p;
}
DMC_HD uint64_t color_plane_bytes(const ColorFrameDesc& d) {
    const ColorPlanes p = color_planes(d);
    return (uint64_t)p.yw * p.yh + (d.nc == 3 ? 2ull * p.cw * p.ch : 0ull);
}

// Block `blk` of the scan (MCU order, the blocks of each MCU in component order, luma blocks row by row): its component and
// the offset of its top-left sample from the frame's plane base; *stride = the row pitch of that plane.
DMC_HD uint64_t color_block_origin(const ColorFrameDesc& d, uint32_t blk, int* comp, int* stride) {
    const ColorPlanes pl = color_planes(d);
    const uint32_t bpm = (uint32_t)color_blocks_per_mcu(d), ny = (uint32_t)color_luma_blocks(d);
    const uint32_t mcu = blk / bpm, pos = blk - mcu * bpm;
    const uint32_t mx = mcu % (uint32_t)d.mcus_x, my = mcu / (uint32_t)d.mcus_x;
    if (pos < ny) {
        const uint32_t bx = mx * (uint32_t)d.hy + pos % (uint32_t)d.hy, by = my * (uint32_t)d.vy + pos / (uint32_t)d.hy;
        *comp = 0; *stride = pl.yw;
        return (uint64_t)by * 8u * pl.yw + bx * 8u;
    }
    const int c = (int)(pos - ny) + 1;
    *comp = c; *stride = pl.cw;
    return (uint64_t)pl.yw * pl.yh + (uint64_t)(c - 1) * pl.cw * pl.ch + (uint64_t)my * 8u * pl.cw + mx * 8u;
}

// ---- parallel entropy decoding of interleaved MCUs -------------------------------------------------------------------
// The synchronisation state of dmc_jpeg_core.h's scan decoder plus the block's position inside the MCU, which selects the
// component and so the Huffman tables.  Two decoders agree only when bit position, zigzag index and MCU position agree.
// tabs[2c] / tabs[2c + 1] are the DC / AC tables of component c.
struct ColorScanState { uint32_t p; int k; int m; };

DMC_HD int color_scan_symbol(const uint32_t* words, uint32_t last_word, const HuffTable* tabs, int ny, int bpm, ColorScanState& st, int* kz, int* comp) {
    const int c = st.m < ny ? 0 : st.m - ny + 1;
    ScanState s; s.p = st.p; s.k = st.k;
    const int v = scan_symbol(words, last_word, tabs[2 * c], tabs[2 * c + 1], s, kz);
    if (st.k != 0 && s.k == 0) st.m = st.m + 1 == bpm ? 0 : st.m + 1;       // block complete: the next one of the MCU
    st.p = s.p; st.k = s.k;
    *comp = c;
    return v;
}

// Counting pass over one sub-sequence: symbols that START in [st.p, hi).  nb = blocks whose DC code starts here,
// dcsum[c] = the sum of the DC differences of component c among them.
DMC_HD void color_scan_count(const uint32_t* words, uint32_t last_word, const HuffTable* tabs, int ny, int bpm, ColorScanState& st, uint32_t hi,
                             uint32_t* nb, int32_t* dcsum) {
    uint32_t n = 0; int32_t s0 = 0, s1 = 0, s2 = 0;
    while (st.p < hi) {
        int kz, c; const int v = color_scan_symbol(words, last_word, tabs, ny, bpm, st, &kz, &c);
        if (kz == 0) { n++; if (c == 0) s0 += v; else if (c == 1) s1 += v; else s2 += v; }
    }
    *nb = n; dcsum[0] = s0; dcsum[1] = s1; dcsum[2] = s2;
}

// ---- one lane per frame: streams with restart intervals ----------------------------------------------------------
// Decodes every block of the frame into coefs (64 int16 per block in scan order, natural order, not dequantised; zero on
// entry).  An MCU counter drives the restarts; every RSTn resets all DC predictors (jdhuff.c process_restart).
DMC_HD void color_decode_serial(const uint8_t* blob, const ColorFrameDesc& d, const HuffTable* tabs, int16_t* coefs) {
    BitReader br; br_init(br, blob, d.scan_offset, d.scan_end);
    int pred[3] = {0, 0, 0}, until_restart = d.restart_interval;
    const int bpm = color_blocks_per_mcu(d), ny = color_luma_blocks(d);
    const uint32_t nmcu = (uint32_t)d.mcus_x * (uint32_t)d.mcus_y;
    for (uint32_t u = 0; u < nmcu; u++) {
        if (d.restart_interval) {
            if (until_restart == 0) {       // byte-align, consume RSTn, reset the predictors
                if (!br.marker) { br.nbits = 0; br_fill(br); }
                if (br.marker >= 0xD0 && br.marker <= 0xD7) br.pos += 2;
                br.acc = 0; br.nbits = 0; br.marker = 0; pred[0] = pred[1] = pred[2] = 0; until_restart = d.restart_interval;
            }
            until_restart--;
        }
        for (int m = 0; m < bpm; m++, coefs += 64) {
            const int c = m < ny ? 0 : m - ny + 1;
            decode_block(br, tabs[2 * c], tabs[2 * c + 1], pred[c], coefs);
        }
    }
}

// ---- upsampling and colour conversion ------------------------------------------------------------------------------
// Chroma sample of output pixel (x, y), upsampled as libjpeg-turbo's jdsample.c does with fancy upsampling on (its default;
// merged upsampling runs only without it).  c: the plane, pitch cw; dw x dh: the real downsampled size,
// ceil(cols / hy) x ceil(rows / vy), whose last column and row are the edges (not the padded IDCT output).
//   2x1, dw > 2: h2v1_fancy_upsample   (3 this + left + 1) >> 2, (3 this + right + 2) >> 2, edge columns copied
//   1x2:         h1v2_fancy_upsample   (3 this + above + 1) >> 2, (3 this + below + 2) >> 2
//   2x2, dw > 2: h2v2_fancy_upsample   column sums 3 this + above / below, then (3 s + s_left + 8) >> 4 and
//                (3 s + s_right + 7) >> 4, edge columns (4 s + 8) >> 4 and (4 s + 7) >> 4
//   otherwise (4x1, or 2x1 / 2x2 with dw <= 2): replication (h2v1_upsample, h2v2_upsample, int_upsample)
// The rows above the first and below the last real chroma row are copies of those rows (jdmainct.c context rows).
DMC_HD int color_chroma_sample(const uint8_t* c, int cw, int dw, int dh, int hy, int vy, int x, int y) {
    if (hy == 1 && vy == 1) return c[(size_t)y * cw + x];
    if (hy == 1 && vy == 2) {
        const int cy = y >> 1, ny = (y & 1) ? (cy + 1 < dh ? cy + 1 : cy) : (cy > 0 ? cy - 1 : 0);
        return (3 * c[(size_t)cy * cw + x] + c[(size_t)ny * cw + x] + ((y & 1) ? 2 : 1)) >> 2;
    }
    if (hy == 2 && vy == 1 && dw > 2) {
        const uint8_t* r = c + (size_t)y * cw;
        const int cx = x >> 1, v = r[cx];
        if (x & 1) return cx == dw - 1 ? v : (3 * v + r[cx + 1] + 2) >> 2;
        return cx == 0 ? v : (3 * v + r[cx - 1] + 1) >> 2;
    }
    if (hy == 2 && vy == 2 && dw > 2) {
        const int cy = y >> 1, ny = (y & 1) ? (cy + 1 < dh ? cy + 1 : cy) : (cy > 0 ? cy - 1 : 0);
        const uint8_t* r0 = c + (size_t)cy * cw; const uint8_t* r1 = c + (size_t)ny * cw;
        const int cx = x >> 1, s = 3 * r0[cx] + r1[cx];
        if (x & 1) return cx == dw - 1 ? (4 * s + 7) >> 4 : (3 * s + 3 * r0[cx + 1] + r1[cx + 1] + 7) >> 4;
        return cx == 0 ? (4 * s + 8) >> 4 : (3 * s + 3 * r0[cx - 1] + r1[cx - 1] + 8) >> 4;
    }
    return c[(size_t)(y / vy) * cw + x / hy];
}

DMC_HD uint8_t color_clamp(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

// Output pixel (x, y) of the frame whose planes start at `planes`, as B, G, R (one-component frames: B = G = R = Y).
DMC_HD void color_pixel_bgr(const ColorFrameDesc& d, const uint8_t* planes, const YccTables& t, int rows, int cols, int x, int y, uint8_t* bgr) {
    const ColorPlanes pl = color_planes(d);
    const int Y = planes[(size_t)y * pl.yw + x];
    if (d.nc == 1) { bgr[0] = bgr[1] = bgr[2] = (uint8_t)Y; return; }
    const int dw = (cols + d.hy - 1) / d.hy, dh = (rows + d.vy - 1) / d.vy;
    const uint8_t* cbp = planes + (size_t)pl.yw * pl.yh;
    const uint8_t* crp = cbp + (size_t)pl.cw * pl.ch;
    const int cb = color_chroma_sample(cbp, pl.cw, dw, dh, d.hy, d.vy, x, y);
    const int cr = color_chroma_sample(crp, pl.cw, dw, dh, d.hy, d.vy, x, y);
    bgr[0] = color_clamp(Y + t.cb_b[cb]);
    bgr[1] = color_clamp(Y + ((t.cb_g[cb] + t.cr_g[cr]) >> 16));
    bgr[2] = color_clamp(Y + t.cr_r[cr]);
}

}  // namespace dmcjpeg
