// dmc_jpeg_enc_core.h -- baseline-JPEG (SOF0, 8-bit, single component) ENCODING primitives shared by the CUDA kernels of
// dmc_jpeg_enc.cu and by their lane-by-lane CPU emulation (tests/cpp/jpeg_enc_emul.cpp): quality -> quantisation table,
// the stream header, the IJG "islow" forward DCT, quantisation + zigzag, the bit count of one block and the emission of
// one block's codes at a given bit offset, and the byte-stuffing pass.
//
// The target is byte equality with cv2.imencode(img, [IMWRITE_JPEG_QUALITY, q]) of an 8UC1 image (libjpeg-turbo with
// OpenCV's settings: JFIF 1.1 APP0, one DQT, the standard luminance Huffman tables of ITU T.81 K.3 / K.5, no restart
// intervals).  That encoder is fully determined by these rules:
//   * quality: q clamped to [1, 100]; scale = q < 50 ? 5000 / q : 200 - 2q; entry = clamp((std * scale + 50) / 100, 1, 255)
//     (jcparam.c jpeg_quality_scaling / jpeg_add_quant_table with force_baseline);
//   * the last column and row are replicated to a multiple of 8 (jccoefct.c / jcsample.c edge expansion);
//   * forward DCT: jfdctint.c on x - 128 in 32-bit ints, the same 13-bit constants as idct_1d of dmc_jpeg_core.h;
//   * quantisation: sign(x) * ((|x| + 4Q) / (8Q)) -- jcdctmgr.c's reciprocal quantiser computes exactly this;
//   * Huffman coding in raster block order, one DC predictor starting at 0, 0xF0 (ZRL) before a non-zero coefficient
//     preceded by 16 or more zeros, 0x00 (EOB) after the last non-zero one; MSB-first bits, 0x00 stuffed after every 0xFF,
//     the last byte padded with 1-bits (jchuff.c).
// With optimised Huffman tables (cv2.IMWRITE_JPEG_OPTIMIZE = 1, libjpeg's optimize_coding) the stream is the same except
// for the two DHT segments: each frame gets the tables jchuff.c's jpeg_gen_optimal_table builds from its own DC category
// and AC symbol counts (see the optimised-table section below).
#pragma once
#include "dmc_jpeg_core.h"
#include <string.h>

namespace dmcjpeg {

constexpr int kEncHeaderBytes = 328;                       // SOI + APP0 + DQT + SOF0 + 2 x DHT + SOS
// Largest code + value of one block: DC category 11 (9-bit code + 11 bits) and 63 AC coefficients of category 10 with
// 16-bit codes (+ 10 bits).  ZRL (11 bits for 16 zeros) and EOB (4 bits for at least one zero) cost less than the
// non-zero coefficients they replace, so a block never needs more.
constexpr uint32_t kEncMaxBlockBits = (9 + 11) + 63 * (16 + 10);
constexpr uint64_t kEncMaxStreamBytes = 1ull << 28;       // the decoder's scan limit
// With optimised tables: a Huffman code over at most 12 DC categories + the reserved symbol 256 (13 leaves) is at most
// 12 bits long, and AC codes (ZRL, EOB included) are limited to 16 bits as before, so a block takes at most
// (12 + 11) + 63 * (16 + 10) bits; ZRL and EOB, at most 16 bits each, still cost less than the non-zero coefficients they
// replace.  The header is at most as long as the standard one (12 DC + 162 AC symbols).
constexpr uint32_t kEncMaxBlockBitsOpt = (12 + 11) + 63 * (16 + 10);

struct EncTables {
    uint32_t dc[16];          // (code length << 16) | code of DC category s; s <= 11
    uint32_t ac[256];         // (code length << 16) | code of AC symbol (run << 4) | size; 0 = not in the table
    uint32_t qmul[64];        // natural order: floor(2^32 / (8 Q)) + 1 (quant_div)
    uint32_t qhalf[64];       // natural order: 4 Q
    uint8_t header[kEncHeaderBytes];
};

// A frame's own Huffman coding in optimised mode (written by the table kernel): code tables as in EncTables, and the
// frame's header of header_bytes = 154 + (DC symbols) + (AC symbols) bytes.
struct EncFrameCode {
    uint32_t dc[16];
    uint32_t ac[256];
    uint32_t header_bytes;
    uint8_t header[kEncHeaderBytes];
};
constexpr int kEncHeaderDhtAt = 20 + 69 + 13;             // the DHT segments follow SOI + APP0, DQT and SOF0
constexpr int kEncSosBytes = 10;

// One block after the transform.  nz: bit k set iff zigzag coefficient k (1..63) is non-zero.
struct EncBlock { uint64_t nz; uint32_t ac_bits; int32_t dc; };

// Worst-case stream size of a rows x cols frame: header, EOI, and every scan byte followed by a stuffed zero.
inline uint64_t jpeg_encode_bound(int rows, int cols, bool optimize = false) {
    const uint64_t blocks = (uint64_t)((rows + 7) / 8) * (uint64_t)((cols + 7) / 8);
    return (uint64_t)kEncHeaderBytes + 2 + 2 * ((blocks * (optimize ? kEncMaxBlockBitsOpt : kEncMaxBlockBits) + 7) / 8);
}

// ---- tables and header (host) -----------------------------------------------------------------------------------------
inline const uint8_t* std_luminance_quant() {          // ITU T.81 K.1, natural order
    static const uint8_t t[64] = {16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
                                  14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
                                  49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
    return t;
}
static const uint8_t kStdDcBits[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};                  // K.3
static const uint8_t kStdDcVals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
static const uint8_t kStdAcBits[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};               // K.5
static const uint8_t kStdAcVals[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81, 0x91, 0xa1,
    0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26,
    0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56,
    0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85,
    0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa,
    0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6,
    0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

// cv2 clamps the quality to [0, 100]; libjpeg treats 0 as 1.  std[] and quant[] in natural order.
inline void scale_quant_table(const uint8_t* std, int quality, uint8_t quant[64]) {
    int q = quality < 1 ? 1 : (quality > 100 ? 100 : quality);
    const int scale = q < 50 ? 5000 / q : 200 - 2 * q;
    for (int i = 0; i < 64; i++) {
        const int v = ((int)std[i] * scale + 50) / 100;
        quant[i] = (uint8_t)(v < 1 ? 1 : (v > 255 ? 255 : v));
    }
}

inline void quality_table(int quality, uint8_t quant[64]) { scale_quant_table(std_luminance_quant(), quality, quant); }

// jcdctmgr's canonical code assignment (jpeg_make_c_derived_tbl): (length << 16) | code per symbol.
inline void make_code_table(const uint8_t bits[16], const uint8_t* vals, uint32_t* out, int nout) {
    memset(out, 0, sizeof(uint32_t) * nout);
    uint32_t code = 0; int p = 0;
    for (int l = 1; l <= 16; l++) {
        for (int i = 0; i < bits[l - 1]; i++, p++) out[vals[p]] = ((uint32_t)l << 16) | code++;
        code <<= 1;
    }
}

// SOI and the JFIF 1.1 APP0 segment cv2 writes (no thumbnail, 1:1 aspect)
static const uint8_t kSoiApp0[20] = {0xFF, 0xD8, 0xFF, 0xE0, 0x00, 0x10, 'J', 'F', 'I', 'F', 0x00, 0x01, 0x01, 0x00, 0x00, 0x01, 0x00, 0x01, 0x00, 0x00};

// The 328 header bytes cv2.imencode writes for an 8UC1 image.
inline void build_header(const uint8_t quant[64], int rows, int cols, uint8_t* h) {
    uint8_t* p = h;
    memcpy(p, kSoiApp0, 20); p += 20;
    *p++ = 0xFF; *p++ = 0xDB; *p++ = 0x00; *p++ = 0x43; *p++ = 0x00;
    for (int k = 0; k < 64; k++) *p++ = quant[zigzag_to_natural(k)];
    const uint8_t sof[13] = {0xFF, 0xC0, 0x00, 0x0B, 0x08, (uint8_t)(rows >> 8), (uint8_t)rows, (uint8_t)(cols >> 8), (uint8_t)cols, 0x01, 0x01, 0x11, 0x00};
    memcpy(p, sof, 13); p += 13;
    *p++ = 0xFF; *p++ = 0xC4; *p++ = 0x00; *p++ = 0x1F; *p++ = 0x00;
    memcpy(p, kStdDcBits, 16); p += 16; memcpy(p, kStdDcVals, 12); p += 12;
    *p++ = 0xFF; *p++ = 0xC4; *p++ = 0x00; *p++ = 0xB5; *p++ = 0x10;
    memcpy(p, kStdAcBits, 16); p += 16; memcpy(p, kStdAcVals, 162); p += 162;
    const uint8_t sos[10] = {0xFF, 0xDA, 0x00, 0x08, 0x01, 0x01, 0x00, 0x00, 0x3F, 0x00};
    memcpy(p, sos, 10);
}

// quant_div's constants for the table entry Q (divisor 8 Q).
inline void quant_recip(uint32_t q, uint32_t* qmul, uint32_t* qhalf) {
    const uint32_t d = 8u * q;
    *qmul = (uint32_t)((1ull << 32) / d) + 1u;
    *qhalf = d / 2u;
}

inline void make_enc_tables(int quality, int rows, int cols, EncTables* t) {
    uint8_t quant[64];
    quality_table(quality, quant);
    make_code_table(kStdDcBits, kStdDcVals, t->dc, 16);
    make_code_table(kStdAcBits, kStdAcVals, t->ac, 256);
    for (int i = 0; i < 64; i++) quant_recip(quant[i], &t->qmul[i], &t->qhalf[i]);
    build_header(quant, rows, cols, t->header);
}

// ---- transform --------------------------------------------------------------------------------------------------------
// IJG jfdctint.c "islow", in place on 64 centred samples (row-major): rows first, then columns.
DMC_HD void fdct_1d(int* d, int stride, int pass) {
    const int F_0_298 = 2446, F_0_390 = 3196, F_0_541 = 4433, F_0_765 = 6270, F_0_899 = 7373, F_1_175 = 9633,
              F_1_501 = 12299, F_1_847 = 15137, F_1_961 = 16069, F_2_053 = 16819, F_2_562 = 20995, F_3_072 = 25172;
    const int odd_shift = pass == 0 ? DMCJ_CONST_BITS - DMCJ_PASS1_BITS : DMCJ_CONST_BITS + DMCJ_PASS1_BITS;
    int tmp0 = d[0] + d[7 * stride], tmp7 = d[0] - d[7 * stride];
    int tmp1 = d[stride] + d[6 * stride], tmp6 = d[stride] - d[6 * stride];
    int tmp2 = d[2 * stride] + d[5 * stride], tmp5 = d[2 * stride] - d[5 * stride];
    int tmp3 = d[3 * stride] + d[4 * stride], tmp4 = d[3 * stride] - d[4 * stride];
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    if (pass == 0) {
        d[0] = (tmp10 + tmp11) * (1 << DMCJ_PASS1_BITS);
        d[4 * stride] = (tmp10 - tmp11) * (1 << DMCJ_PASS1_BITS);
    } else {
        d[0] = DMCJ_DESCALE(tmp10 + tmp11, DMCJ_PASS1_BITS);
        d[4 * stride] = DMCJ_DESCALE(tmp10 - tmp11, DMCJ_PASS1_BITS);
    }
    int z1 = (tmp12 + tmp13) * F_0_541;
    d[2 * stride] = DMCJ_DESCALE(z1 + tmp13 * F_0_765, odd_shift);
    d[6 * stride] = DMCJ_DESCALE(z1 + tmp12 * (-F_1_847), odd_shift);
    z1 = tmp4 + tmp7;
    int z2 = tmp5 + tmp6, z3 = tmp4 + tmp6, z4 = tmp5 + tmp7;
    const int z5 = (z3 + z4) * F_1_175;
    tmp4 *= F_0_298; tmp5 *= F_2_053; tmp6 *= F_3_072; tmp7 *= F_1_501;
    z1 *= -F_0_899; z2 *= -F_2_562; z3 *= -F_1_961; z4 *= -F_0_390;
    z3 += z5; z4 += z5;
    d[7 * stride] = DMCJ_DESCALE(tmp4 + z1 + z3, odd_shift);
    d[5 * stride] = DMCJ_DESCALE(tmp5 + z2 + z4, odd_shift);
    d[3 * stride] = DMCJ_DESCALE(tmp6 + z2 + z3, odd_shift);
    d[1 * stride] = DMCJ_DESCALE(tmp7 + z1 + z4, odd_shift);
}

DMC_HD void fdct_islow(int* d) {
#pragma unroll
    for (int r = 0; r < 8; r++) fdct_1d(d + 8 * r, 1, 0);
#pragma unroll
    for (int c = 0; c < 8; c++) fdct_1d(d + c, 8, 1);
}

DMC_HD uint32_t mulhi_u32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

// sign(x) * ((|x| + 4Q) / (8Q)) as a multiply-high: with m = floor(2^32 / d) + 1 = (2^32 + e) / d, 0 < e <= d, the
// product n * m / 2^32 exceeds n / d by n * e / (d * 2^32) < 1 / d whenever n * e < 2^32, i.e. for every n < 2^21 when
// d <= 2040; the fractional part of n / d is at most (d - 1) / d, so the floor is unchanged.  n = |x| + 4Q < 2^16 here.
// tests/test_jpeg_enc_emul.py checks it against the division for every |x| < 2^15 and every Q in 1..255.
DMC_HD int quant_div(int x, uint32_t qmul, uint32_t qhalf) {
    const uint32_t n = (uint32_t)(x < 0 ? -x : x) + qhalf;
    const int r = (int)mulhi_u32(n, qmul);
    return x < 0 ? -r : r;
}

// Quantises the transformed block d (natural order) into zz[64] (zigzag order) and returns the non-zero mask of the AC
// coefficients (bit k = zigzag index k).
DMC_HD uint64_t quantize_zigzag(const int* d, const uint32_t* qmul, const uint32_t* qhalf, int16_t* zz) {
    uint64_t nz = 0;
#pragma unroll
    for (int k = 0; k < 64; k++) {
        const int n = zigzag_to_natural(k);
        const int v = quant_div(d[n], qmul[n], qhalf[n]);
        zz[k] = (int16_t)v;
        if (k > 0 && v != 0) nz |= 1ull << k;
    }
    return nz;
}

DMC_HD int bit_length(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return 32 - __clz(v);
#else
    return v ? 32 - __builtin_clz(v) : 0;
#endif
}

DMC_HD uint32_t code_len(uint32_t e) { return e >> 16; }

// Bits of the AC part of one block (codes + value bits, ZRL and EOB included).
DMC_HD uint32_t block_ac_bits(const int16_t* zz, const uint32_t* ac) {
    uint32_t bits = 0; int last = 0;
#pragma unroll
    for (int k = 1; k < 64; k++) {
        const int v = zz[k];
        if (v != 0) {
            const int r = k - last - 1, s = bit_length((uint32_t)(v < 0 ? -v : v));
            bits += (uint32_t)(r >> 4) * code_len(ac[0xF0]) + code_len(ac[((r & 15) << 4) | s]) + (uint32_t)s;
            last = k;
        }
    }
    if (last < 63) bits += code_len(ac[0x00]);
    return bits;
}

// The Huffman symbols of the AC part of one block as emit_block emits them: add(symbol, count) for every run/size
// symbol, ZRL (0xF0) and EOB (0x00).  zz is indexed with constants only, so a register array stays in registers.
template <class Add>
DMC_HD void block_ac_symbols(const int16_t* zz, Add add) {
    int last = 0;
#pragma unroll
    for (int k = 1; k < 64; k++) {
        const int v = zz[k];
        if (v != 0) {
            const int r = k - last - 1, s = bit_length((uint32_t)(v < 0 ? -v : v));
            if (r >= 16) add(0xF0, r >> 4);
            add(((r & 15) << 4) | s, 1);
            last = k;
        }
    }
    if (last < 63) add(0x00, 1);
}

// block_ac_bits from the non-zero mask, reading only the non-zero coefficients zz(k).
template <class Coef>
DMC_HD uint32_t block_ac_bits_sparse(uint64_t nz, Coef zz, const uint32_t* ac) {
    uint32_t bits = 0; int last = 0;
    while (nz) {
#if defined(__CUDA_ARCH__)
        const int k = __ffsll((long long)nz) - 1;
#else
        const int k = __builtin_ctzll(nz);
#endif
        nz &= nz - 1;
        const int r = k - last - 1, v = zz(k), s = bit_length((uint32_t)(v < 0 ? -v : v));
        bits += (uint32_t)(r >> 4) * code_len(ac[0xF0]) + code_len(ac[((r & 15) << 4) | s]) + (uint32_t)s;
        last = k;
    }
    if (last < 63) bits += code_len(ac[0x00]);
    return bits;
}

// Bits of the DC part: code of the category of `diff` + the category's value bits.
DMC_HD uint32_t block_dc_bits(int diff, const uint32_t* dc) {
    const int s = bit_length((uint32_t)(diff < 0 ? -diff : diff));
    return code_len(dc[s]) + (uint32_t)s;
}

// ---- optimised Huffman tables ----------------------------------------------------------------------------------------
// jchuff.c's jpeg_gen_optimal_table, restated for one warp.  The serial original, with freq[256] = 1 reserving the
// all-ones code:
//   repeat: c1 = the symbol of the smallest non-zero freq, c2 = that of the next smallest (c2 != c1), both searches
//           taking the LARGER symbol on ties; stop when there is no c2; freq[c1] += freq[c2], freq[c2] = 0; codesize++
//           for every symbol of c1's tree and of c2's tree (walked through the `others` chains), c2's tree joins c1's.
//   bits[l] = number of symbols with codesize l; lengths over 16 are folded back (opt_fold); the reserved symbol is
//   taken from the longest length; HUFFVAL lists the symbols 0..255 by codesize, then by value.
// Here lane i owns the symbols i + 32 k (k < 9; symbol 256 is lane 0's k = 8).  The non-zero frequencies are exactly
// the roots of the trees, so a symbol's tree is named by its root: set[] starts as the symbol itself, and a merge
// increments codesize for the symbols of sets c1 and c2 and renames set c2 to c1 -- the increments of the chain walks.
// The searches combine the lanes' opt_lane_min with a warp min of the frequency, then a warp max of the symbol among
// the lanes holding that minimum.  Total counts stay below 2^26 (at most 64 symbols per block and 2^28 / 1661 * 8
// blocks), far from jchuff.c's 10^9 search sentinel, and a code length needs a total of at least Fibonacci(length + 2),
// so lengths stay below 40 < kOptMaxLen.
constexpr int kOptPer = 9, kOptMaxLen = 64;
struct OptLane { uint32_t fr[kOptPer]; uint16_t set[kOptPer], cs[kOptPer]; };

// hist: counts of symbols 0 .. nsym-1 (nsym <= 256)
DMC_HD void opt_lane_init(OptLane& L, const uint32_t* hist, int nsym, int lane) {
#pragma unroll
    for (int k = 0; k < kOptPer; k++) {
        const int s = lane + 32 * k;
        L.fr[k] = s < nsym ? hist[s] : (s == 256 ? 1u : 0u);
        L.set[k] = (uint16_t)s; L.cs[k] = 0;
    }
}

// The lane's smallest non-zero frequency among its symbols other than excl, the larger symbol on ties (ascending k):
// *f = 0xFFFFFFFF and *s = -1 when there is none.
DMC_HD void opt_lane_min(const OptLane& L, int lane, int excl, uint32_t* f, int* s) {
    uint32_t bf = 0xFFFFFFFFu; int bs = -1;
#pragma unroll
    for (int k = 0; k < kOptPer; k++) {
        const int sym = lane + 32 * k;
        if (L.fr[k] != 0u && sym != excl && L.fr[k] <= bf) { bf = L.fr[k]; bs = sym; }
    }
    *f = bf; *s = bs;
}

// Merges tree c2 (frequency f2) into tree c1.
DMC_HD void opt_lane_merge(OptLane& L, int lane, int c1, int c2, uint32_t f2) {
#pragma unroll
    for (int k = 0; k < kOptPer; k++) {
        const int sym = lane + 32 * k;
        if (sym == c1) L.fr[k] += f2;
        if (sym == c2) L.fr[k] = 0u;
        if (L.set[k] == c1 || L.set[k] == c2) { L.cs[k]++; L.set[k] = (uint16_t)c1; }
    }
}

// cnt[l] (l <= kOptMaxLen): symbols with codesize l, the reserved one included.  Folds lengths over 16 back exactly as
// jchuff.c, removes the reserved symbol from the longest length and returns BITS (bits[l - 1] = codes of length l) and
// the number of symbols.  cnt is clobbered.
DMC_HD int opt_fold(uint32_t* cnt, uint8_t bits[16]) {
    int i;
    for (i = kOptMaxLen; i > 16; i--)
        while (cnt[i] > 0) {
            int j = i - 2;
            while (cnt[j] == 0) j--;
            cnt[i] -= 2; cnt[i - 1]++; cnt[j + 1] += 2; cnt[j]--;
        }
    while (cnt[i] == 0) i--;
    cnt[i]--;
    int n = 0;
    for (int l = 1; l <= 16; l++) { bits[l - 1] = (uint8_t)cnt[l]; n += (int)cnt[l]; }
    return n;
}

// (length << 16) | code of the symbol at HUFFVAL position p: make_code_table's canonical assignment.
DMC_HD uint32_t opt_code(const uint8_t bits[16], int p) {
    uint32_t code = 0; int pos = 0;
    for (int l = 1; l <= 16; l++) {
        if (p < pos + bits[l - 1]) return ((uint32_t)l << 16) | (code + (uint32_t)(p - pos));
        code = (code + bits[l - 1]) << 1; pos += bits[l - 1];
    }
    return 0;
}

// One DHT segment (table class tc: 0 DC, 1 AC; table 0) at h; returns its length, 21 + n.
DMC_HD int opt_write_dht(uint8_t* h, int tc, const uint8_t bits[16], const uint8_t* vals, int n) {
    const int len = 19 + n;
    h[0] = 0xFF; h[1] = 0xC4; h[2] = (uint8_t)(len >> 8); h[3] = (uint8_t)len; h[4] = (uint8_t)(tc << 4);
    for (int l = 0; l < 16; l++) h[5 + l] = bits[l];
    for (int i = 0; i < n; i++) h[21 + i] = vals[i];
    return 21 + n;
}

// ---- bit packing ------------------------------------------------------------------------------------------------------
// The scan is packed into 32-bit words, bit 31 of word i being scan bit 32 i.  A writer starting at an arbitrary bit
// position hands every completed word to sink(word index, value, partial): partial is true for the first word when the
// writer started inside it and for the last, incomplete word -- those words are shared with the neighbouring writers
// and must be OR-ed into a zeroed word; every other word belongs to this writer alone.
template <class Sink>
struct BitWriter {
    uint64_t acc;     // pending bits, left-aligned
    int fill;         // pending bits in acc (the first (start & 31) of them are the neighbour's zeros)
    uint32_t wi;      // word index of acc's top 32 bits
    bool partial;
    Sink sink;
};

template <class Sink>
DMC_HD BitWriter<Sink> bw_start(uint32_t bitpos, Sink sink) {
    return BitWriter<Sink>{0ull, (int)(bitpos & 31u), bitpos >> 5, (bitpos & 31u) != 0u, sink};
}

// n in 1..32, v < 2^n
template <class Sink>
DMC_HD void bw_put(BitWriter<Sink>& w, uint32_t v, int n) {
    w.acc |= (uint64_t)v << (64 - w.fill - n);
    w.fill += n;
    if (w.fill >= 32) {
        w.sink(w.wi, (uint32_t)(w.acc >> 32), w.partial);
        w.partial = false; w.wi++; w.acc <<= 32; w.fill -= 32;
    }
}

template <class Sink>
DMC_HD void bw_finish(BitWriter<Sink>& w) {
    if (w.fill > 0) w.sink(w.wi, (uint32_t)(w.acc >> 32), true);
}

// Code + value bits of one coefficient of category s (value bits: v, or v - 1 when v < 0, low s bits).
template <class Sink>
DMC_HD void bw_put_coef(BitWriter<Sink>& w, uint32_t e, int v, int s) {
    const uint32_t val = (uint32_t)(v < 0 ? v - 1 : v) & ((1u << s) - 1u);
    bw_put(w, ((e & 0xFFFFu) << s) | val, (int)code_len(e) + s);
}

// Emits one block: the DC difference, then the AC coefficients zz[k] (zigzag order) at the set bits of nz.
template <class Sink, class Coef>
DMC_HD void emit_block(BitWriter<Sink>& w, int diff, uint64_t nz, Coef zz, const uint32_t* dc, const uint32_t* ac) {
    const int sd = bit_length((uint32_t)(diff < 0 ? -diff : diff));
    bw_put_coef(w, dc[sd], diff, sd);
    int last = 0;
    while (nz) {
#if defined(__CUDA_ARCH__)
        const int k = __ffsll((long long)nz) - 1;
#else
        const int k = __builtin_ctzll(nz);
#endif
        nz &= nz - 1;
        int r = k - last - 1;
        for (; r >= 16; r -= 16) bw_put(w, ac[0xF0] & 0xFFFFu, (int)code_len(ac[0xF0]));
        const int v = zz(k), s = bit_length((uint32_t)(v < 0 ? -v : v));
        bw_put_coef(w, ac[(r << 4) | s], v, s);
        last = k;
    }
    if (last < 63) bw_put(w, ac[0x00] & 0xFFFFu, (int)code_len(ac[0x00]));
}

// Pads the scan of `total_bits` bits with 1-bits to a whole byte.
DMC_HD void pad_scan(uint32_t* words, uint32_t total_bits) {
    const uint32_t b = total_bits & 7u;
    if (b) words[total_bits >> 5] |= (0xFFu >> b) << (24 - 8 * ((total_bits >> 3) & 3u));
}

// ---- byte stuffing ----------------------------------------------------------------------------------------------------
// A stuffing lane handles the 16 scan bytes [i0, i0 + 16) (i0 a multiple of 16) of a scan of L bytes.
DMC_HD void stuff_load(const uint32_t* words, uint32_t L, uint32_t i0, uint32_t w[4]) {
#pragma unroll
    for (int j = 0; j < 4; j++) w[j] = i0 + 4u * j < L ? words[(i0 >> 2) + j] : 0u;
}

DMC_HD uint8_t stuff_byte(const uint32_t w[4], int i) { return (uint8_t)(w[i >> 2] >> (24 - 8 * (i & 3))); }

// Number of 0xFF bytes among the lane's bytes.
DMC_HD uint32_t stuff_count(const uint32_t w[4], uint32_t L, uint32_t i0) {
    uint32_t n = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) n += (i0 + i < L && stuff_byte(w, i) == 0xFF) ? 1u : 0u;
    return n;
}

// Writes the lane's bytes to out[0..], a 0x00 after every 0xFF.
DMC_HD void stuff_write(const uint32_t w[4], uint32_t L, uint32_t i0, uint8_t* out) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        if (i0 + i >= L) break;
        const uint8_t b = stuff_byte(w, i);
        out[o++] = b;
        if (b == 0xFF) out[o++] = 0;
    }
}

}  // namespace dmcjpeg
