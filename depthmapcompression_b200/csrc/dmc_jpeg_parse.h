// dmc_jpeg_parse.h -- host-side marker parsing of baseline grayscale JPEG streams (DQT / SOF0 / DHT / DRI / SOS), table
// validation and de-duplication (the derivation itself, derive_table, is in dmc_jpeg_core.h), and the colour parse of the
// colour decoder (jpeg_parse_color_frame).  Host only; shared by dmc_capi.cu and by the CPU emulation harnesses of the
// parallel decoders (tests/cpp/jpeg_emul.cpp, tests/cpp/jpeg_color_emul.cpp).  Reference
// counterpart: libjpeg's jdmarker.c / jdhuff.c as reached through cv::imdecode(buf, 0) (main.cpp:284, :521) and jpeg_decode() (jpegTurboDemo.cpp:217-271).
#pragma once
#include "dmc_jpeg_core.h"
#include "dmc_jpeg_color_core.h"
#include <string.h>
#include <string>
#include <unordered_map>
#include <vector>

namespace dmc {

using namespace dmcjpeg;

// ---- host: marker parsing ----------------------------------------------------------------------------------------
// De-duplicated table pool: the distinct tables in first-occurrence order, found again by a hash of their bytes (equal
// hashes are confirmed with memcmp), so that interning is linear in the number of tables -- a batch of streams with
// optimised Huffman tables brings two distinct tables per frame.
template <class T> struct TablePool {
    std::vector<T> items;
    std::unordered_multimap<uint64_t, int> index;
    static uint64_t hash(const T& v) {
        static_assert(sizeof(T) % 8 == 0, "tables are hashed as 64-bit words");
        uint64_t w[sizeof(T) / 8], h = 0x9E3779B97F4A7C15ull;
        memcpy(w, &v, sizeof w);
        for (uint64_t x : w) { h ^= x; h *= 0xFF51AFD7ED558CCDull; h ^= h >> 32; }
        return h;
    }
    int find(const T& v, uint64_t h) const {
        auto r = index.equal_range(h);
        for (auto it = r.first; it != r.second; ++it) if (memcmp(&items[it->second], &v, sizeof(T)) == 0) return it->second;
        return -1;
    }
    int intern(const T& v) {
        const uint64_t h = hash(v);
        const int i = find(v, h);
        if (i >= 0) return i;
        items.push_back(v);
        index.emplace(h, (int)items.size() - 1);
        return (int)items.size() - 1;
    }
    void assign(const std::vector<T>& v) {         // takes v as the pool; equal entries resolve to the first of them
        clear();
        items = v;
        for (size_t i = 0; i < items.size(); i++) { const uint64_t h = hash(items[i]); if (find(items[i], h) < 0) index.emplace(h, (int)i); }
    }
    void clear() { items.clear(); index.clear(); }
};
struct JpegTablePools { TablePool<QuantTable> q; TablePool<HuffTable> h; };

// Parses one stream [p, p+len).  Returns an empty string on success, else the reason it is not supported.
// rows < 0: any frame size is accepted (reported through out_rows / out_cols).
// The frame's tables are interned into `pools` (FrameDesc::qt / dc / ac index pools.q.items / pools.h.items).
inline std::string jpeg_parse_frame(const uint8_t* p, uint64_t len, uint64_t blob_offset, int rows, int cols,
                                    JpegTablePools& pools, FrameDesc* d, int* out_rows = nullptr, int* out_cols = nullptr) {
    QuantTable qt[4]; bool have_q[4] = {false, false, false, false};
    HuffTable dc[4], ac[4]; bool have_dc[4] = {false, false, false, false}, have_ac[4] = {false, false, false, false};
    int comp_tq = -1, restart = 0; bool have_sof = false;
    if (len < 4 || p[0] != 0xFF || p[1] != 0xD8) return "no SOI marker";
    uint64_t i = 2;
    while (i + 4 <= len) {
        if (p[i] != 0xFF) return "marker expected";
        uint8_t m = p[i + 1];
        if (m == 0xFF) { i++; continue; }                       // fill byte
        if (m == 0x01 || (m >= 0xD0 && m <= 0xD7)) { i += 2; continue; }     // TEM / RSTn: stand-alone markers without a length
        uint64_t seg = ((uint64_t)p[i + 2] << 8) | p[i + 3];    // includes the two length bytes
        if (seg < 2) return "bad segment length";
        if (i + 2 + seg > len) return "truncated segment";
        const uint8_t* s = p + i + 4; uint64_t sl = seg - 2;
        if (m == 0xDB) {                                        // DQT
            uint64_t k = 0;
            while (k < sl) {
                int pq = s[k] >> 4, tq = s[k] & 15; k++;
                if (tq > 3 || pq > 1) return "bad DQT";
                if (k + (pq ? 128u : 64u) > sl) return "truncated DQT";
                for (int z = 0; z < 64; z++) {
                    int v = pq ? ((s[k] << 8) | s[k + 1]) : s[k]; k += pq ? 2 : 1;
                    qt[tq].q[zigzag_to_natural(z)] = (uint16_t)v;
                }
                have_q[tq] = true;
            }
        } else if (m == 0xC4) {                                 // DHT
            uint64_t k = 0;
            while (k < sl) {
                if (k + 17 > sl) return "truncated DHT";
                int tc = s[k] >> 4, th = s[k] & 15; k++;
                if (th > 3 || tc > 1) return "bad DHT";
                uint8_t bits[17]; bits[0] = 0; int n = 0;
                for (int l = 1; l <= 16; l++) { bits[l] = s[k++]; n += bits[l]; }
                if (n > 256 || k + n > sl) return "bad DHT";
                if (tc == 0) for (int v = 0; v < n; v++) if (s[k + v] > 15) return "bad DHT (DC category > 15)";      // jdhuff.c rejects these too
                if (!derive_table(bits, s + k, n, tc ? &ac[th] : &dc[th])) return "bad DHT (code lengths do not form a prefix code)";
                k += n;
                (tc ? have_ac : have_dc)[th] = true;
            }
        } else if (m == 0xC0 || m == 0xC1) {                    // SOF0 / SOF1 (sequential Huffman)
            if (sl < 9 || s[0] != 8) return "only 8-bit precision is supported";
            int h = (s[1] << 8) | s[2], w = (s[3] << 8) | s[4];
            if (s[5] != 1) return "only single-component (grayscale) JPEG is supported";
            if (s[7] != 0x11) return "unexpected sampling factors";
            if (h == 0 || w == 0) return "empty frame (DNL-defined height is not supported)";
            if (out_rows) *out_rows = h;
            if (out_cols) *out_cols = w;
            if (rows >= 0 && (h != rows || w != cols)) return "frame size differs from the batch size";
            comp_tq = s[8]; have_sof = true;
        } else if (m == 0xC2 || (m >= 0xC5 && m <= 0xCF && m != 0xC8 && m != 0xCC)) {
            return "progressive / lossless / arithmetic JPEG is not supported";
        } else if (m == 0xDD) {                                 // DRI
            if (sl < 2) return "truncated DRI";
            restart = (s[0] << 8) | s[1];
        } else if (m == 0xDA) {                                 // SOS: entropy-coded data follows
            if (!have_sof) return "SOS before SOF";
            if (sl < 6) return "truncated SOS";
            if (s[0] != 1) return "only single-component scans are supported";
            int td = s[2] >> 4, ta = s[2] & 15;
            if (td > 3 || ta > 3 || comp_tq < 0 || comp_tq > 3 || !have_dc[td] || !have_ac[ta] || !have_q[comp_tq]) return "scan refers to a missing table";
            d->scan_offset = blob_offset + i + 2 + seg; d->scan_end = blob_offset + len; d->restart_interval = restart;
            d->qt = pools.q.intern(qt[comp_tq]);
            d->dc = pools.h.intern(dc[td]); d->ac = pools.h.intern(ac[ta]);
            return "";
        }
        i += 2 + seg;
    }
    return "no SOS marker";
}

// The same with plain vectors as the pools (tables already in them are found again, the first of equal ones first).
inline std::string jpeg_parse_frame(const uint8_t* p, uint64_t len, uint64_t blob_offset, int rows, int cols,
                                    std::vector<QuantTable>& qpool, std::vector<HuffTable>& hpool, FrameDesc* d, int* out_rows = nullptr, int* out_cols = nullptr) {
    JpegTablePools pools;
    pools.q.assign(qpool); pools.h.assign(hpool);
    std::string why = jpeg_parse_frame(p, len, blob_offset, rows, cols, pools, d, out_rows, out_cols);
    qpool.swap(pools.q.items); hpool.swap(pools.h.items);
    return why;
}

// ---- colour streams (dmc_jpeg_color.cu) -------------------------------------------------------------------------------
// Parses one stream for the colour decoder: baseline / extended sequential Huffman, 8-bit, one component or three in one
// interleaved scan that libjpeg would treat as YCbCr, chroma sampled 1x1 and luma 1x1, 2x1, 2x2, 1x2 or 4x1.  Returns an
// empty string on success, else the reason.  rows < 0: any frame size; out_nc receives the component count.  The tables
// of the frame are interned into `pools`; d->ds_offset, plane_offset and coef_offset are left to the caller.
inline std::string jpeg_parse_color_frame(const uint8_t* p, uint64_t len, uint64_t blob_offset, int rows, int cols, JpegTablePools& pools,
                                          ColorFrameDesc* d, int* out_rows = nullptr, int* out_cols = nullptr, int* out_nc = nullptr) {
    QuantTable qt[4]; bool have_q[4] = {false, false, false, false};
    HuffTable dc[4], ac[4]; bool have_dc[4] = {false, false, false, false}, have_ac[4] = {false, false, false, false};
    int restart = 0, nc = 0, frame_h = 0, frame_w = 0, comp_id[3] = {0, 0, 0}, comp_tq[3] = {0, 0, 0}, samp[3] = {0, 0, 0};
    bool have_sof = false, jfif = false, adobe = false; int adobe_transform = -1;
    if (len < 4 || p[0] != 0xFF || p[1] != 0xD8) return "no SOI marker";
    uint64_t i = 2;
    while (i + 4 <= len) {
        if (p[i] != 0xFF) return "marker expected";
        uint8_t m = p[i + 1];
        if (m == 0xFF) { i++; continue; }
        if (m == 0x01 || (m >= 0xD0 && m <= 0xD7)) { i += 2; continue; }
        uint64_t seg = ((uint64_t)p[i + 2] << 8) | p[i + 3];
        if (seg < 2) return "bad segment length";
        if (i + 2 + seg > len) return "truncated segment";
        const uint8_t* s = p + i + 4; uint64_t sl = seg - 2;
        if (m == 0xE0) {                                        // APP0: JFIF implies YCbCr (jdmarker.c examine_app0)
            if (sl >= 14 && memcmp(s, "JFIF\0", 5) == 0) jfif = true;
        } else if (m == 0xEE) {                                 // APP14: Adobe colour transform (examine_app14)
            if (sl >= 12 && memcmp(s, "Adobe", 5) == 0) { adobe = true; adobe_transform = s[11]; }
        } else if (m == 0xDB) {
            uint64_t k = 0;
            while (k < sl) {
                int pq = s[k] >> 4, tq = s[k] & 15; k++;
                if (tq > 3 || pq > 1) return "bad DQT";
                if (k + (pq ? 128u : 64u) > sl) return "truncated DQT";
                for (int z = 0; z < 64; z++) {
                    int v = pq ? ((s[k] << 8) | s[k + 1]) : s[k]; k += pq ? 2 : 1;
                    qt[tq].q[zigzag_to_natural(z)] = (uint16_t)v;
                }
                have_q[tq] = true;
            }
        } else if (m == 0xC4) {
            uint64_t k = 0;
            while (k < sl) {
                if (k + 17 > sl) return "truncated DHT";
                int tc = s[k] >> 4, th = s[k] & 15; k++;
                if (th > 3 || tc > 1) return "bad DHT";
                uint8_t bits[17]; bits[0] = 0; int n = 0;
                for (int l = 1; l <= 16; l++) { bits[l] = s[k++]; n += bits[l]; }
                if (n > 256 || k + n > sl) return "bad DHT";
                if (tc == 0) for (int v = 0; v < n; v++) if (s[k + v] > 15) return "bad DHT (DC category > 15)";
                if (!derive_table(bits, s + k, n, tc ? &ac[th] : &dc[th])) return "bad DHT (code lengths do not form a prefix code)";
                k += n;
                (tc ? have_ac : have_dc)[th] = true;
            }
        } else if (m == 0xC0 || m == 0xC1) {                    // SOF0 / SOF1
            if (have_sof) return "more than one SOF marker";
            if (sl < 6 || s[0] != 8) return "only 8-bit precision is supported";
            frame_h = (s[1] << 8) | s[2]; frame_w = (s[3] << 8) | s[4]; nc = s[5];
            if (nc == 4) return "CMYK / YCCK JPEG is not supported";
            if (nc != 1 && nc != 3) return "only one- or three-component JPEG is supported";
            if (sl < 6 + 3u * nc) return "truncated SOF";
            for (int c = 0; c < nc; c++) {
                comp_id[c] = s[6 + 3 * c]; samp[c] = s[7 + 3 * c]; comp_tq[c] = s[8 + 3 * c];
                const int h = samp[c] >> 4, v = samp[c] & 15;
                if (h < 1 || h > 4 || v < 1 || v > 4) return "bad sampling factors";
                if (comp_tq[c] > 3) return "bad quantisation table index";
            }
            if (nc == 3) {
                const int y = samp[0];
                if (samp[1] != 0x11 || samp[2] != 0x11 || (y != 0x11 && y != 0x21 && y != 0x22 && y != 0x12 && y != 0x41))
                    return "unsupported sampling factors (luma 1x1, 2x1, 2x2, 1x2 or 4x1 with 1x1 chroma are supported)";
            }
            if (frame_h == 0 || frame_w == 0) return "empty frame (DNL-defined height is not supported)";
            if (out_rows) *out_rows = frame_h;
            if (out_cols) *out_cols = frame_w;
            if (out_nc) *out_nc = nc;
            if (rows >= 0 && (frame_h != rows || frame_w != cols)) return "frame size differs from the batch size";
            have_sof = true;
        } else if (m == 0xC2 || m == 0xC3 || (m >= 0xC5 && m <= 0xCF && m != 0xC8 && m != 0xCC)) {
            return "progressive / lossless / arithmetic JPEG is not supported";
        } else if (m == 0xDD) {
            if (sl < 2) return "truncated DRI";
            restart = (s[0] << 8) | s[1];
        } else if (m == 0xDA) {
            if (!have_sof) return "SOS before SOF";
            if (sl < 1 || sl < 4u + 2u * s[0]) return "truncated SOS";
            if (nc == 3) {                                      // libjpeg's default_decompress_parms: JFIF, then Adobe, then the IDs
                if (!jfif && adobe && adobe_transform == 0) return "RGB JPEG (Adobe transform 0) is not supported";
                if (!jfif && !adobe && comp_id[0] == 'R' && comp_id[1] == 'G' && comp_id[2] == 'B') return "RGB JPEG (component IDs R G B) is not supported";
            }
            if (s[0] != nc) return nc == 3 ? "non-interleaved (multi-scan) colour JPEG is not supported" : "bad SOS component count";
            for (int c = 0; c < nc; c++) {
                if (s[1 + 2 * c] != comp_id[c]) return "scan components differ from the frame's components or their order";
                const int td = s[2 + 2 * c] >> 4, ta = s[2 + 2 * c] & 15;
                if (td > 3 || ta > 3 || !have_dc[td] || !have_ac[ta] || !have_q[comp_tq[c]]) return "scan refers to a missing table";
                d->qt[c] = pools.q.intern(qt[comp_tq[c]]);
                d->dc[c] = pools.h.intern(dc[td]); d->ac[c] = pools.h.intern(ac[ta]);
            }
            for (int c = nc; c < 3; c++) { d->qt[c] = d->qt[0]; d->dc[c] = d->dc[0]; d->ac[c] = d->ac[0]; }
            d->nc = nc;
            d->hy = nc == 3 ? samp[0] >> 4 : 1; d->vy = nc == 3 ? samp[0] & 15 : 1;
            d->mcus_x = (frame_w + 8 * d->hy - 1) / (8 * d->hy); d->mcus_y = (frame_h + 8 * d->vy - 1) / (8 * d->vy);
            d->scan_offset = blob_offset + i + 2 + seg; d->scan_end = blob_offset + len; d->restart_interval = restart;
            d->ds_offset = d->plane_offset = d->coef_offset = 0; d->pad = 0;
            return "";
        }
        i += 2 + seg;
    }
    return "no SOS marker";
}

}  // namespace dmc
