// jpeg_enc_opt_emul.cpp -- CPU emulation of the JPEG encoder kernels in optimised-table mode (csrc/dmc_jpeg_enc.cu with
// DMC_JPEG_OPTIMIZE_HUFFMAN): the AC symbol counts of the transform, the DC category counts and the warp-parallel table
// builder of the table kernel (32 lanes executed one after the other, the warp reductions turned into loops), the header
// with the frame's DHT segments, and the entropy stage with the frame's tables.  Everything is built from the primitives
// of csrc/dmc_jpeg_enc_core.h.  Also a serial restatement of libjpeg's jpeg_gen_optimal_table (jchuff.c) that the
// builder is compared with, and a check of the parser's table de-duplication against a linear scan.  Built by
// tests/test_jpeg_enc_opt_emul.py with g++.
#include "../../depthmapcompression_b200/csrc/dmc_jpeg_enc_core.h"
#include "../../depthmapcompression_b200/csrc/dmc_jpeg_parse.h"

#include <algorithm>
#include <vector>

using namespace dmcjpeg;

namespace {

// jchuff.c jpeg_gen_optimal_table, serially (freq[0..256], freq[256] is set to 1 here).  Returns the number of symbols,
// -1 where libjpeg fails with JERR_HUFF_CLEN_OVERFLOW.
int gen_optimal_table_serial(const uint32_t* hist, int nsym, uint8_t bits_out[16], uint8_t vals[256]) {
    const int MAX_CLEN = 32;
    long freq[257];
    for (int i = 0; i < 257; i++) freq[i] = i < nsym ? (long)hist[i] : 0;
    int bits[MAX_CLEN + 1] = {0}, codesize[257] = {0}, others[257];
    for (int i = 0; i < 257; i++) others[i] = -1;
    freq[256] = 1;
    for (;;) {
        int c1 = -1, c2 = -1;
        long v = 1000000000L;
        for (int i = 0; i <= 256; i++) if (freq[i] && freq[i] <= v) { v = freq[i]; c1 = i; }
        v = 1000000000L;
        for (int i = 0; i <= 256; i++) if (freq[i] && freq[i] <= v && i != c1) { v = freq[i]; c2 = i; }
        if (c2 < 0) break;
        freq[c1] += freq[c2];
        freq[c2] = 0;
        codesize[c1]++;
        while (others[c1] >= 0) { c1 = others[c1]; codesize[c1]++; }
        others[c1] = c2;
        codesize[c2]++;
        while (others[c2] >= 0) { c2 = others[c2]; codesize[c2]++; }
    }
    for (int i = 0; i <= 256; i++)
        if (codesize[i]) {
            if (codesize[i] > MAX_CLEN) return -1;
            bits[codesize[i]]++;
        }
    int i;
    for (i = MAX_CLEN; i > 16; i--)
        while (bits[i] > 0) {
            int j = i - 2;
            while (bits[j] == 0) j--;
            bits[i] -= 2; bits[i - 1]++; bits[j + 1] += 2; bits[j]--;
        }
    while (bits[i] == 0) i--;
    bits[i]--;
    int n = 0;
    for (int l = 1; l <= 16; l++) { bits_out[l - 1] = (uint8_t)bits[l]; n += bits[l]; }
    int p = 0;
    for (int l = 1; l <= MAX_CLEN; l++)
        for (int j = 0; j <= 255; j++) if (codesize[j] == l) vals[p++] = (uint8_t)j;
    return n;
}

// build_opt_table of dmc_jpeg_enc.cu with the warp's 32 lanes emulated.  *folded: a code length over 16 was folded.
int build_opt_table_emul(const uint32_t* hist, int nsym, uint8_t bits[16], uint8_t vals[256], uint32_t code[256], bool* folded) {
    OptLane L[32];
    for (int lane = 0; lane < 32; lane++) opt_lane_init(L[lane], hist, nsym, lane);
    for (;;) {
        uint32_t f[32]; int s[32];
        auto search = [&](int excl, uint32_t* fmin, int* c) {
            for (int lane = 0; lane < 32; lane++) opt_lane_min(L[lane], lane, excl, &f[lane], &s[lane]);
            *fmin = 0xFFFFFFFFu; *c = -1;
            for (int lane = 0; lane < 32; lane++) *fmin = std::min(*fmin, f[lane]);                    // __reduce_min_sync
            for (int lane = 0; lane < 32; lane++) if (f[lane] == *fmin) *c = std::max(*c, s[lane]);     // __reduce_max_sync
        };
        uint32_t f1, f2; int c1, c2;
        search(-1, &f1, &c1);
        search(c1, &f2, &c2);
        if (c2 < 0) break;
        for (int lane = 0; lane < 32; lane++) opt_lane_merge(L[lane], lane, c1, c2, f2);
    }
    uint32_t cnt[kOptMaxLen + 1] = {0}, start[kOptMaxLen + 1];
    int longest = 0;
    for (int lane = 0; lane < 32; lane++)
        for (int k = 0; k < kOptPer; k++)
            if (L[lane].cs[k]) {
                if (L[lane].cs[k] > kOptMaxLen) return -1;
                cnt[L[lane].cs[k]]++; longest = std::max(longest, (int)L[lane].cs[k]);
            }
    *folded = longest > 16;
    uint32_t acc = 0;
    for (int c = 0; c <= kOptMaxLen; c++) { start[c] = acc; acc += cnt[c] - (c == L[0].cs[8] ? 1u : 0u); }
    for (int k = 0; k < 8; k++) {
        unsigned same[32];
        for (int lane = 0; lane < 32; lane++) {                                                       // __match_any_sync
            same[lane] = 0;
            for (int o = 0; o < 32; o++) if (L[o].cs[k] == L[lane].cs[k]) same[lane] |= 1u << o;
        }
        for (int lane = 0; lane < 32; lane++) {
            const int c = L[lane].cs[k];
            if (c) vals[start[c] + __builtin_popcount(same[lane] & ((1u << lane) - 1u))] = (uint8_t)(32 * k + lane);
        }
        for (int lane = 0; lane < 32; lane++) {
            const int c = L[lane].cs[k];
            if (c && lane == __builtin_ctz(same[lane])) start[c] += __builtin_popcount(same[lane]);
        }
    }
    const int n = opt_fold(cnt, bits);
    memset(code, 0, 256 * sizeof(uint32_t));
    for (int p = 0; p < n; p++) code[vals[p]] = opt_code(bits, p);
    return n;
}

const uint32_t kUntouched = 0xA5A5A5A5u;

}  // namespace

// Encodes one rows x cols 8UC1 image with optimised tables and `lanes` emulated entropy lanes.  Returns the stream length,
// or a negative number: -1 an ownership violation of the packed words, -2 the stream does not fit into `cap` bytes,
// -3 / -4 the scan / stream exceeds the optimised bound, -5 a table the decoder's derive_table refuses, -6 a table
// builder failure.  *folded: a code length over 16 was folded back in one of the two tables.
extern "C" long long jpeg_enc_opt_emul(const uint8_t* img, int rows, int cols, int quality, int lanes, uint8_t* out, unsigned long long cap, int* folded) {
    EncTables t;
    make_enc_tables(quality, rows, cols, &t);
    const int bw = (cols + 7) / 8, nb = bw * ((rows + 7) / 8);
    std::vector<int16_t> coefs((size_t)nb * 64);
    std::vector<EncBlock> info(nb);
    uint32_t hist[2][256] = {};
    // transform (jpeg_enc_transform_kernel<true>): AC symbol counts
    for (int b = 0; b < nb; b++) {
        const int bx = b % bw, by = b / bw;
        int d[64];
        for (int r = 0; r < 8; r++) {
            const uint8_t* row = img + (size_t)std::min(by * 8 + r, rows - 1) * cols;
            for (int c = 0; c < 8; c++) d[r * 8 + c] = (int)row[std::min(bx * 8 + c, cols - 1)] - 128;
        }
        fdct_islow(d);
        int16_t* zz = &coefs[(size_t)b * 64];
        info[b].nz = quantize_zigzag(d, t.qmul, t.qhalf, zz);
        block_ac_symbols(zz, [&](int sym, int c) { hist[1][sym] += (uint32_t)c; });
        info[b].ac_bits = 0;
        info[b].dc = zz[0];
    }
    // table kernel: DC categories, the two tables, the header, the decoder's tables
    for (int b = 0; b < nb; b++) hist[0][bit_length((uint32_t)std::abs(info[b].dc - (b > 0 ? info[b - 1].dc : 0)))]++;
    EncFrameCode fc;
    uint8_t bits[2][16], vals[2][256];
    int n[2];
    bool fold[2];
    uint32_t dc_code[256];
    n[0] = build_opt_table_emul(hist[0], 16, bits[0], vals[0], dc_code, &fold[0]);
    n[1] = build_opt_table_emul(hist[1], 256, bits[1], vals[1], fc.ac, &fold[1]);
    if (n[0] < 0 || n[1] < 0) return -6;
    memcpy(fc.dc, dc_code, sizeof fc.dc);
    *folded = (fold[0] ? 1 : 0) | (fold[1] ? 2 : 0);
    for (int c = 0; c < 2; c++) {
        uint8_t b17[17]; b17[0] = 0;
        memcpy(b17 + 1, bits[c], 16);
        HuffTable ht;
        if (!derive_table(b17, vals[c], n[c], &ht)) return -5;
    }
    memcpy(fc.header, t.header, kEncHeaderDhtAt);
    int h = kEncHeaderDhtAt;
    h += opt_write_dht(fc.header + h, 0, bits[0], vals[0], n[0]);
    h += opt_write_dht(fc.header + h, 1, bits[1], vals[1], n[1]);
    memcpy(fc.header + h, t.header + kEncHeaderBytes - kEncSosBytes, kEncSosBytes);
    fc.header_bytes = (uint32_t)(h + kEncSosBytes);

    // entropy stage (jpeg_enc_entropy_kernel<true>): lane j codes blocks [j * per, (j + 1) * per)
    const int per = (nb + lanes - 1) / lanes;
    std::vector<uint32_t> lbits(lanes, 0), start(lanes, 0);
    for (int j = 0; j < lanes; j++) {
        const int b0 = std::min(j * per, nb), b1 = std::min(b0 + per, nb);
        int prev = b0 > 0 ? info[b0 - 1].dc : 0;
        for (int b = b0; b < b1; b++) {
            const int16_t* zz = &coefs[(size_t)b * 64];
            lbits[j] += block_ac_bits_sparse(info[b].nz, [zz](int k) { return (int)zz[k]; }, fc.ac) + block_dc_bits(info[b].dc - prev, fc.dc);
            prev = info[b].dc;
        }
    }
    uint32_t T = 0;
    for (int j = 0; j < lanes; j++) { start[j] = T; T += lbits[j]; }
    const uint64_t max_bits = (uint64_t)nb * kEncMaxBlockBitsOpt;
    if (T > max_bits) return -3;
    std::vector<uint32_t> words(max_bits / 32 + 2, kUntouched);
    for (int j = 0; j < lanes; j++) {
        const uint32_t B = start[j], E = B + lbits[j];
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
            emit_block(w, info[b].dc - prev, info[b].nz, [zz](int k) { return (int)zz[k]; }, fc.dc, fc.ac);
            prev = info[b].dc;
        }
        bw_finish(w);
    }
    if (violation) return -1;
    pad_scan(words.data(), T);
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
    const uint64_t len = (uint64_t)fc.header_bytes + scan.size() + 2;
    if (len > jpeg_encode_bound(rows, cols, true)) return -4;
    if (len > cap) return -2;
    memcpy(out, fc.header, fc.header_bytes);
    memcpy(out + fc.header_bytes, scan.data(), scan.size());
    out[len - 2] = 0xFF; out[len - 1] = 0xD9;
    return (long long)len;
}

extern "C" unsigned long long jpeg_enc_opt_bound(int rows, int cols, int optimize) { return jpeg_encode_bound(rows, cols, optimize != 0); }

// The emulated warp builder against the serial jpeg_gen_optimal_table on one histogram of nsym counts.  Returns the
// number of symbols when BITS, HUFFVAL and the code table agree, -1 when they differ, -2 when the serial one fails.
extern "C" int jpeg_opt_table_check(const uint32_t* hist, int nsym) {
    uint8_t bits[16], vals[256], sbits[16], svals[256];
    uint32_t code[256], scode[256];
    bool folded;
    const int ns = gen_optimal_table_serial(hist, nsym, sbits, svals);
    if (ns < 0) return -2;
    const int n = build_opt_table_emul(hist, nsym, bits, vals, code, &folded);
    make_code_table(sbits, svals, scode, 256);
    if (n != ns || memcmp(bits, sbits, 16) != 0 || memcmp(vals, svals, (size_t)n) != 0 || memcmp(code, scode, sizeof code) != 0) return -1;
    return n;
}

// Parses n streams (blob + offsets[i] .. offsets[i + 1]) into one set of pools, as a decode group does, and compares
// the pools and the FrameDesc indices with those of the linear first-occurrence scan.  Returns the number of distinct
// Huffman tables, -1 on a difference, -2 on a parse error.
extern "C" int jpeg_dedup_check(const uint8_t* blob, const unsigned long long* offsets, int n, int* n_quant) {
    dmc::JpegTablePools pools;
    std::vector<QuantTable> lq; std::vector<HuffTable> lh;
    auto linear = [](auto& pool, const auto& v) {
        for (size_t i = 0; i < pool.size(); i++) if (memcmp(&pool[i], &v, sizeof v) == 0) return (int)i;
        pool.push_back(v); return (int)pool.size() - 1;
    };
    for (int i = 0; i < n; i++) {
        FrameDesc d, one;
        std::vector<QuantTable> q1; std::vector<HuffTable> h1;
        if (!dmc::jpeg_parse_frame(blob + offsets[i], offsets[i + 1] - offsets[i], 0, -1, -1, pools, &d).empty()) return -2;
        if (!dmc::jpeg_parse_frame(blob + offsets[i], offsets[i + 1] - offsets[i], 0, -1, -1, q1, h1, &one).empty()) return -2;
        if (d.qt != linear(lq, q1[one.qt]) || d.dc != linear(lh, h1[one.dc]) || d.ac != linear(lh, h1[one.ac])) return -1;
    }
    if (pools.q.items.size() != lq.size() || pools.h.items.size() != lh.size()) return -1;
    if (memcmp(pools.q.items.data(), lq.data(), lq.size() * sizeof(QuantTable)) != 0) return -1;
    if (memcmp(pools.h.items.data(), lh.data(), lh.size() * sizeof(HuffTable)) != 0) return -1;
    *n_quant = (int)lq.size();
    return (int)lh.size();
}
