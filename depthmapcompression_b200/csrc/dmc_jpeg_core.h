// dmc_jpeg_core.h -- baseline-JPEG (SOF0, 8-bit, single component) decoding primitives shared by the CUDA kernels of
// dmc_jpeg.cu and by the host-side parser: marker parsing, Huffman table derivation, the entropy decoder of one
// 8x8 block and the integer inverse DCT.
//
// This is row (f)-1 of SURVEY.md section 8 ("on-GPU decode feeding the chain"): the reference obtains its decoded
// disparity maps from libjpeg(-turbo) -- cv::imdecode(buf, 0) at main.cpp:284,521 and jpeg_decode() with JDCT_ISLOW at
// jpegTurboDemo.cpp:217-271 / main.cpp:276.  To keep chain parity the decoded pixels must equal libjpeg's bit for bit,
// so the inverse DCT below is a restatement of the IJG "islow" algorithm (jidctint.c: 13-bit constants, PASS1_BITS 2,
// DESCALE rounding, range-limit table semantics); nvJPEG cannot be used for that (measured: 1.2 % of the pixels differ
// by one from libjpeg-turbo, tools/nvjpeg_probe.py).
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define DMC_HD __host__ __device__ __forceinline__
#else
#define DMC_HD inline
#endif

namespace dmcjpeg {

// Derived Huffman table: 9-bit look-ahead + canonical slow path (codes of 10..16 bits).
struct HuffTable {
    uint16_t look[512];      // (length << 8) | symbol for codes of <= 9 bits, 0 = longer code
    int32_t maxcode[18];     // largest code of each length (left-aligned compare as in jdhuff.c), -1 if none
    int32_t valoffset[18];   // huffval index of the first code of each length minus that code
    uint8_t huffval[256];
};

struct FrameDesc {
    uint64_t scan_offset;    // offset of the entropy-coded segment inside the blob
    uint64_t scan_end;       // one past the last byte of this frame's stream
    int32_t restart_interval;
    int32_t qt, dc, ac;      // indices into the de-duplicated table arrays
    uint64_t ds_offset;      // byte offset of this frame's de-stuffed copy of the scan inside the scratch buffer (16-aligned)
};

struct QuantTable { uint16_t q[64]; };   // natural (row-major) order

// zigzag index -> natural order (jpeg_natural_order)
DMC_HD int zigzag_to_natural(int k) {
    const unsigned char t[64] = {0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
                                 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return t[k];
}

// ---- bit reader over the entropy-coded segment (byte stuffing 0xFF00, stops feeding at any marker) -----------------
struct BitReader {
    const uint8_t* p;
    uint64_t pos, end;
    uint64_t acc;     // bits are consumed from the top
    int nbits;
    int marker;       // 0 = none seen, else the marker byte that stopped the feeder
};

DMC_HD void br_init(BitReader& br, const uint8_t* p, uint64_t pos, uint64_t end) { br.p = p; br.pos = pos; br.end = end; br.acc = 0; br.nbits = 0; br.marker = 0; }

// Keeps at least 33 valid bits in the accumulator (a code of <= 16 bits or a value of <= 16 bits is consumed between two
// calls).  Fast path: four stream bytes at once when none of them is 0xFF (their loads are independent, so the chain waits
// for one memory latency per four bytes instead of one per byte); otherwise byte by byte with stuffing / marker handling.
DMC_HD void br_fill(BitReader& br) {
    if (br.nbits > 32) return;
    if (!br.marker && br.pos + 4 <= br.end) {
        const uint8_t* q = br.p + br.pos;
        const uint32_t w = ((uint32_t)q[0] << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | (uint32_t)q[3];
        const uint32_t nw = ~w;                                        // a 0xFF byte of w is a zero byte of nw
        if (((nw - 0x01010101u) & ~nw & 0x80808080u) == 0u) {
            br.acc |= (uint64_t)w << (32 - br.nbits);
            br.nbits += 32; br.pos += 4;
            return;
        }
    }
    while (br.nbits <= 32) {
        uint64_t b = 0;
        if (!br.marker && br.pos < br.end) {
            b = br.p[br.pos];
            if (b == 0xFF) {
                uint8_t n = br.pos + 1 < br.end ? br.p[br.pos + 1] : 0xD9;
                if (n == 0) br.pos += 2;                 // stuffed zero
                else { br.marker = n; b = 0; }           // a marker: leave pos at the 0xFF, feed zeros from now on
            } else br.pos += 1;
        }
        br.acc |= b << (56 - br.nbits);
        br.nbits += 8;
    }
}
DMC_HD uint32_t br_peek(BitReader& br, int n) { return (uint32_t)(br.acc >> (64 - n)); }     // n in 1..32, after br_fill
DMC_HD void br_skip(BitReader& br, int n) { br.acc <<= n; br.nbits -= n; }

// Derives the decoding tables of one DHT entry (bits[1..16], vals[nvals]); used by the host parser and by the encoder's
// table kernel, which derives the decoder tables of the optimised tables it builds.  Returns false for tables libjpeg's
// jpeg_make_d_derived_tbl rejects with JERR_BAD_HUFF_TABLE: more than 256 symbols, or code lengths that do not form a
// prefix code (a code of length l must be < 2^l; an over-subscribed BITS array would otherwise index past look[]).
DMC_HD bool derive_table(const uint8_t bits[17], const uint8_t* vals, int nvals, HuffTable* t) {
    memset(t, 0, sizeof *t);
    int huffsize[257], huffcode[257], p = 0;
    for (int l = 1; l <= 16; l++) {
        if (p + bits[l] > 256) return false;
        for (int i = 0; i < bits[l]; i++) huffsize[p++] = l;
    }
    if (p != nvals) return false;
    huffsize[p] = 0;
    int code = 0, si = huffsize[0]; p = 0;
    while (huffsize[p]) {
        while (huffsize[p] == si) huffcode[p++] = code++;
        if (code > (1 << si)) return false;                   // jdhuff.c: "code is now 1 more than the last code used for codelength si"
        code <<= 1; si++;
    }
    p = 0;
    for (int l = 1; l <= 16; l++) {
        if (bits[l]) { t->valoffset[l] = p - huffcode[p]; p += bits[l]; t->maxcode[l] = huffcode[p - 1]; }
        else t->maxcode[l] = -1;
    }
    t->maxcode[17] = 0xFFFFF;
    for (int i = 0; i < nvals; i++) t->huffval[i] = vals[i];
    p = 0;
    for (int l = 1; l <= 9; l++)
        for (int i = 0; i < bits[l]; i++, p++) {
            const int lookbits = huffcode[p] << (9 - l), span = 1 << (9 - l);
            if (lookbits + span > 512) return false;          // (cannot happen once the prefix-code check passed; belt and braces)
            for (int c = 0; c < span; c++) t->look[lookbits + c] = (uint16_t)((l << 8) | vals[p]);
        }
    return true;
}

DMC_HD int huff_decode(BitReader& br, const HuffTable& t) {
    br_fill(br);
    uint32_t look = t.look[br_peek(br, 9)];
    if (look) { br_skip(br, (int)(look >> 8)); return (int)(look & 0xFF); }
    int32_t code = (int32_t)br_peek(br, 16);
    for (int l = 10; l <= 16; l++) {
        int32_t c = code >> (16 - l);
        if (t.maxcode[l] >= 0 && c <= t.maxcode[l]) { br_skip(br, l); return t.huffval[(c + t.valoffset[l]) & 0xFF]; }
    }
    br_skip(br, 16);
    return 0;     // corrupt stream: libjpeg warns and returns 0 as well
}

DMC_HD int huff_extend(int v, int s) { return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v; }     // HUFF_EXTEND

// Decodes one 8x8 block into coef[64] (natural order, NOT dequantised); coef must be zero on entry.
DMC_HD void decode_block(BitReader& br, const HuffTable& dc, const HuffTable& ac, int& pred, int16_t* coef) {
    int s = huff_decode(br, dc);
    if (s) { br_fill(br); int r = (int)br_peek(br, s); br_skip(br, s); pred += huff_extend(r, s); }
    coef[0] = (int16_t)pred;
    for (int k = 1; k < 64;) {
        int rs = huff_decode(br, ac), r = rs >> 4; s = rs & 15;
        if (s) {
            k += r;
            br_fill(br); int v = (int)br_peek(br, s); br_skip(br, s);
            if (k < 64) coef[zigzag_to_natural(k)] = (int16_t)huff_extend(v, s);
            k++;
        } else { if (r == 15) k += 16; else break; }
    }
}

// ---- IJG jidctint.c "islow" inverse DCT -----------------------------------------------------------------------
#define DMCJ_CONST_BITS 13
#define DMCJ_PASS1_BITS 2
#define DMCJ_DESCALE(x, n) (((x) + (1 << ((n) - 1))) >> (n))

// range_limit[(x) & RANGE_MASK] of jdmaster.c's prepare_range_limit_table: clamp(x + 128) for x in [-512, 511],
// with the 10-bit wrap-around of the table index for values outside.
DMC_HD uint8_t idct_range_limit(int x) {
    x &= 1023; if (x >= 512) x -= 1024;
    x += 128;
    return (uint8_t)(x < 0 ? 0 : (x > 255 ? 255 : x));
}

// One 1-D pass.  in[] are the 8 (dequantised for pass 1) inputs, out[] the 8 results before descaling.
// Valid streams stay far inside 32 bits; a corrupt stream can overflow the intermediates exactly as it does in libjpeg
// (two's-complement wrap-around on the device; the CPU emulation of the tests is compiled with -fwrapv; an ASAN/UBSAN
// mutation campaign over parser + decoder -- 150 k mutated streams -- found no memory error).
DMC_HD void idct_1d(const int* in, int* out) {
    const int F_0_298 = 2446, F_0_390 = 3196, F_0_541 = 4433, F_0_765 = 6270, F_0_899 = 7373, F_1_175 = 9633,
              F_1_501 = 12299, F_1_847 = 15137, F_1_961 = 16069, F_2_053 = 16819, F_2_562 = 20995, F_3_072 = 25172;
    int z2 = in[2], z3 = in[6];
    int z1 = (z2 + z3) * F_0_541;
    int tmp2 = z1 + z3 * (-F_1_847);
    int tmp3 = z1 + z2 * F_0_765;
    z2 = in[0]; z3 = in[4];
    int tmp0 = (z2 + z3) * (1 << DMCJ_CONST_BITS);
    int tmp1 = (z2 - z3) * (1 << DMCJ_CONST_BITS);
    int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    tmp0 = in[7]; tmp1 = in[5]; tmp2 = in[3]; tmp3 = in[1];
    z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2; int z4 = tmp1 + tmp3;
    int z5 = (z3 + z4) * F_1_175;
    tmp0 *= F_0_298; tmp1 *= F_2_053; tmp2 *= F_3_072; tmp3 *= F_1_501;
    z1 *= -F_0_899; z2 *= -F_2_562; z3 *= -F_1_961; z4 *= -F_0_390;
    z3 += z5; z4 += z5;
    tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
    out[0] = tmp10 + tmp3; out[7] = tmp10 - tmp3; out[1] = tmp11 + tmp2; out[6] = tmp11 - tmp2;
    out[2] = tmp12 + tmp1; out[5] = tmp12 - tmp1; out[3] = tmp13 + tmp0; out[4] = tmp13 - tmp0;
}

// Full 8x8 block: coef (natural order, raw) x quant -> 64 samples (row-major).  Mirrors jpeg_idct_islow including the
// zero-AC shortcuts (which produce the same values as the full computation would not -- they are part of the
// definition: a column with only a DC term is NOT run through the multiplications).
DMC_HD void idct_islow_block(const int16_t* coef, const uint16_t* quant, uint8_t* out /*64*/) {
    int ws[64];
    for (int c = 0; c < 8; c++) {
        if (coef[8 + c] == 0 && coef[16 + c] == 0 && coef[24 + c] == 0 && coef[32 + c] == 0 && coef[40 + c] == 0 && coef[48 + c] == 0 && coef[56 + c] == 0) {
            int dcval = ((int)coef[c] * (int)quant[c]) * (1 << DMCJ_PASS1_BITS);
            for (int r = 0; r < 8; r++) ws[r * 8 + c] = dcval;
            continue;
        }
        int in[8], o[8];
        for (int r = 0; r < 8; r++) in[r] = (int)coef[r * 8 + c] * (int)quant[r * 8 + c];
        idct_1d(in, o);
        for (int r = 0; r < 8; r++) ws[r * 8 + c] = DMCJ_DESCALE(o[r], DMCJ_CONST_BITS - DMCJ_PASS1_BITS);
    }
    for (int r = 0; r < 8; r++) {
        const int* w = ws + r * 8;
        if (w[1] == 0 && w[2] == 0 && w[3] == 0 && w[4] == 0 && w[5] == 0 && w[6] == 0 && w[7] == 0) {
            uint8_t v = idct_range_limit(DMCJ_DESCALE(w[0], DMCJ_PASS1_BITS + 3));
            for (int c = 0; c < 8; c++) out[r * 8 + c] = v;
            continue;
        }
        int o[8];
        idct_1d(w, o);
        for (int c = 0; c < 8; c++) out[r * 8 + c] = idct_range_limit(DMCJ_DESCALE(o[c], DMCJ_CONST_BITS + DMCJ_PASS1_BITS + 3));
    }
}

// =====================================================================================================================
// Parallel entropy decoding inside one frame (self-synchronising sub-sequences).
//
// A Huffman-coded scan has no entry points, but a decoder started at an arbitrary bit resynchronises with the true symbol
// boundaries after a few dozen symbols with overwhelming probability.  The scan (byte stuffing removed, big-endian 32-bit
// words) is cut into sub-sequences of S bits; decoder j starts at bit j*S in state "expecting a DC code", decodes to the end
// of its sub-sequence and records where it ended: (bit position of the first symbol that starts in the next sub-sequence,
// zigzag index expected there).  In round r = 1, 2, ... every still-active decoder j carries on through sub-sequence j+r
// from its own running state, overwrites the record of that sub-sequence with what IT found (end state, number of blocks
// that start inside, sum of their DC differences) and retires as soon as its end state equals the one that was recorded
// before.  Decoder 0 starts from the true state, so by induction the LAST writer of every record started that sub-sequence
// from the true state (proof sketch in DESIGN.md); when nobody is active any more all records are exact.  Prefix sums over
// (blocks, DC differences) then tell every decoder the index of its first block and the DC predictor, and a final pass
// decodes each sub-sequence once more, this time producing coefficients.  Work: about three passes over the scan instead
// of one, on several hundred lanes instead of one.
// =====================================================================================================================

// 32 bits of the de-stuffed scan starting at bit position p (p / 32 + 1 < nwords: the caller pads with zero words, which
// is what libjpeg feeds once the data has run out).
DMC_HD uint32_t scan_window(const uint32_t* words, uint32_t last_word, uint32_t p) {
    uint32_t i = p >> 5, sh = p & 31;
    if (i > last_word) i = last_word;                    // runaway decoders of corrupt streams read the zero padding
    const uint32_t hi = words[i], lo = words[i + 1];
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(lo, hi, sh);
#else
    return sh ? (hi << sh) | (lo >> (32 - sh)) : hi;
#endif
}

// One Huffman code from the top of `win`; *len = its length.
DMC_HD int huff_decode_window(uint32_t win, const HuffTable& t, int* len) {
    const uint32_t look = t.look[win >> 23];
    if (look) { *len = (int)(look >> 8); return (int)(look & 0xFF); }
    const int32_t code = (int32_t)(win >> 16);
    for (int l = 10; l <= 16; l++) {
        const int32_t c = code >> (16 - l);
        if (t.maxcode[l] >= 0 && c <= t.maxcode[l]) { *len = l; return t.huffval[(c + t.valoffset[l]) & 0xFF]; }
    }
    *len = 16;
    return 0;     // corrupt stream: libjpeg warns and returns 0 as well
}

// Decoder state between two symbols: bit position and the zigzag index the next symbol addresses (0 = a DC code follows).
struct ScanState { uint32_t p; int k; };

// One symbol.  Returns the coefficient value (valid when *kz >= 0: zigzag index it belongs to; -1 = nothing to store).
DMC_HD int scan_symbol(const uint32_t* words, uint32_t last_word, const HuffTable& dc, const HuffTable& ac, ScanState& st, int* kz) {
    const uint32_t win = scan_window(words, last_word, st.p);
    int len, val = 0;
    if (st.k == 0) {
        const int s = huff_decode_window(win, dc, &len) & 15;
        if (s) { const int v = (int)((win << len) >> (32 - s)); val = huff_extend(v, s); }
        st.p += (uint32_t)(len + s); st.k = 1; *kz = 0;
        return val;                                       // the DC DIFFERENCE
    }
    const int rs = huff_decode_window(win, ac, &len), r = rs >> 4, s = rs & 15;
    *kz = -1;
    if (s) {
        const int k = st.k + r;
        const int v = (int)((win << len) >> (32 - s)); val = huff_extend(v, s);
        if (k < 64) *kz = k;
        st.k = k + 1;
    } else if (r == 15) st.k += 16;
    else st.k = 64;                                       // EOB
    st.p += (uint32_t)(len + s);
    if (st.k >= 64) st.k = 0;                             // block complete
    return val;
}

// Counting pass over one sub-sequence: symbols that START in [st.p, hi).  nb = blocks whose DC code starts here,
// dcsum = sum of their DC differences.
DMC_HD void scan_count(const uint32_t* words, uint32_t last_word, const HuffTable& dc, const HuffTable& ac, ScanState& st, uint32_t hi,
                       uint32_t* nb, int32_t* dcsum) {
    uint32_t n = 0; int32_t sum = 0;
    while (st.p < hi) {
        int kz; const int v = scan_symbol(words, last_word, dc, ac, st, &kz);
        if (kz == 0) { n++; sum += v; }
    }
    *nb = n; *dcsum = sum;
}

// In-place islow IDCT on 64 ints reached through an accessor (A(i) = reference to natural-order coefficient i, raw,
// NOT dequantised); `mask` has bit i set iff coefficient i may be non-zero.  Produces the 64 samples through
// emit(row, eight bytes).  Same arithmetic and the same zero shortcuts as idct_islow_block.
template <class Acc, class Emit>
DMC_HD void idct_islow_inplace(Acc A, const int* quant, uint64_t mask, Emit emit) {
    if ((mask & ~1ull) == 0) {                            // DC only: every column and row takes libjpeg's shortcut
        const int dcval = (A(0) * quant[0]) * (1 << DMCJ_PASS1_BITS);
        const uint8_t v = idct_range_limit(DMCJ_DESCALE(dcval, DMCJ_PASS1_BITS + 3));
        uint8_t row[8];
        for (int c = 0; c < 8; c++) row[c] = v;
        for (int r = 0; r < 8; r++) emit(r, row);
        return;
    }
    for (int c = 0; c < 8; c++) {
        if (((mask >> c) & 0x0101010101010100ull) == 0) {       // rows 1..7 of this column are zero
            const int dcval = (A(c) * quant[c]) * (1 << DMCJ_PASS1_BITS);
            for (int r = 0; r < 8; r++) A(r * 8 + c) = dcval;
            continue;
        }
        int in[8], o[8];
        for (int r = 0; r < 8; r++) in[r] = A(r * 8 + c) * quant[r * 8 + c];
        idct_1d(in, o);
        for (int r = 0; r < 8; r++) A(r * 8 + c) = DMCJ_DESCALE(o[r], DMCJ_CONST_BITS - DMCJ_PASS1_BITS);
    }
    for (int r = 0; r < 8; r++) {
        int w[8];
        for (int c = 0; c < 8; c++) w[c] = A(r * 8 + c);
        uint8_t row[8];
        if (w[1] == 0 && w[2] == 0 && w[3] == 0 && w[4] == 0 && w[5] == 0 && w[6] == 0 && w[7] == 0) {
            const uint8_t v = idct_range_limit(DMCJ_DESCALE(w[0], DMCJ_PASS1_BITS + 3));
            for (int c = 0; c < 8; c++) row[c] = v;
        } else {
            int o[8];
            idct_1d(w, o);
            for (int c = 0; c < 8; c++) row[c] = idct_range_limit(DMCJ_DESCALE(o[c], DMCJ_CONST_BITS + DMCJ_PASS1_BITS + 3));
        }
        emit(r, row);
    }
}

// Sub-sequence size (bits, a multiple of 32) for a scan of `total_bits` decoded by `lanes` decoders.
DMC_HD uint32_t scan_subseq_bits(uint32_t total_bits, uint32_t lanes) {
    uint32_t s = (total_bits + lanes - 1) / lanes;
    s = (s + 31u) & ~31u;
    return s < 128u ? 128u : s;
}

}  // namespace dmcjpeg
