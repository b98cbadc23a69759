// dmc_jpeg_parse.h -- host-side marker parsing of baseline grayscale JPEG streams (DQT / SOF0 / DHT / DRI / SOS), table
// validation and de-duplication (the derivation itself, derive_table, is in dmc_jpeg_core.h).  Host only; shared by
// dmc_jpeg.cu and by the CPU emulation harness of the parallel decoder (tests/cpp/jpeg_emul.cpp).  Reference
// counterpart: libjpeg's jdmarker.c / jdhuff.c as reached through cv::imdecode(buf, 0) (main.cpp:284, :521) and jpeg_decode() (jpegTurboDemo.cpp:217-271).
#pragma once
#include "dmc_jpeg_core.h"
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

}  // namespace dmc
