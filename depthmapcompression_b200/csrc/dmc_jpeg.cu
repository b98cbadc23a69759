// dmc_jpeg.cu -- frame-parallel baseline-JPEG decoder on sm_100a (row (f)-1 of SURVEY.md section 8: the decode that
// feeds the post filter set, done by libjpeg in the reference: main.cpp:284,521, jpegTurboDemo.cpp:217-271).
//
//   host   : parse the markers of every frame (DQT / SOF0 / DHT / DRI / SOS), derive and de-duplicate the tables
//   jpeg_frame_kernel (the path of streams WITHOUT restart markers, i.e. everything cv2 / libjpeg write by default):
//             ONE CTA per frame does the whole decode -- removes the byte stuffing, decodes the Huffman scan on all of its
//             lanes at once (self-synchronising sub-sequences, dmc_jpeg_core.h), prefix-sums block counts and DC
//             differences, and in the final pass every lane dequantises and inverse-transforms the blocks it decodes out of
//             shared memory and writes pixels: coefficients never travel through HBM.
//   legacy pair (streams WITH restart intervals): one lane per frame walks the scan and writes int16 coefficients,
//             a second kernel dequantises + IDCTs one block per thread.
//
// Output is bit-identical to libjpeg / libjpeg-turbo's default decoder (JDCT_ISLOW), checked against cv2.imdecode.
#include "dmc_common.cuh"
#include "dmc_jpeg_core.h"
#include "dmc_jpeg_parse.h"
#include "dmc_kernels.cuh"
#include <string.h>
#include <string>
#include <vector>

namespace dmc {

using namespace dmcjpeg;

// ---- kernel 1: entropy decoding, one warp (lane 0) per frame ----------------------------------------------------------
__global__ void __launch_bounds__(128) jpeg_huff_kernel(const uint8_t* __restrict__ blob, const FrameDesc* __restrict__ desc,
                                                        const HuffTable* __restrict__ ht, int16_t* __restrict__ coefs, int n, int blocks_per_frame) {
    // The decode loop is one dependent chain per frame (peek -> table look-up -> shift): ncu shows ~60 instructions per
    // symbol at ~5 cycles each, i.e. latency of dependent instructions, not memory.  The warp's 32 lanes first copy the
    // frame's two tables into shared memory (shorter look-up latency), then lane 0 decodes.
    __shared__ HuffTable s_tab[4][2];
    const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (f >= n) return;                              // uniform per warp
    const FrameDesc d = desc[f];
    if (d.restart_interval == 0) return;             // decoded by jpeg_frame_kernel
    {
        const uint32_t* g0 = reinterpret_cast<const uint32_t*>(&ht[d.dc]); const uint32_t* g1 = reinterpret_cast<const uint32_t*>(&ht[d.ac]);
        uint32_t* s0 = reinterpret_cast<uint32_t*>(&s_tab[w][0]); uint32_t* s1 = reinterpret_cast<uint32_t*>(&s_tab[w][1]);
        for (int i = lane; i < (int)(sizeof(HuffTable) / 4); i += 32) { s0[i] = g0[i]; s1[i] = g1[i]; }
    }
    __syncwarp();
    if (lane != 0) return;
    const HuffTable& dc = s_tab[w][0]; const HuffTable& ac = s_tab[w][1];
    BitReader br; br_init(br, blob, d.scan_offset, d.scan_end);
    int pred = 0, until_restart = d.restart_interval;
    int16_t* c = coefs + (size_t)f * blocks_per_frame * 64;
    for (int b = 0; b < blocks_per_frame; b++, c += 64) {
        if (d.restart_interval) {
            if (until_restart == 0) {       // byte-align, consume RSTn, reset the predictor (jdhuff.c process_restart)
                if (!br.marker) { br.nbits = 0; br_fill(br); }       // (all data bits are consumed; make the feeder meet the marker)
                if (br.marker >= 0xD0 && br.marker <= 0xD7) br.pos += 2;
                br.acc = 0; br.nbits = 0; br.marker = 0; pred = 0; until_restart = d.restart_interval;
            }
            until_restart--;
        }
        decode_block(br, dc, ac, pred, c);
    }
}

// ---- kernel 2: dequantise + islow IDCT + range limit, one thread per 8x8 block ---------------------------------------
__global__ void __launch_bounds__(128) jpeg_idct_kernel(const int16_t* __restrict__ coefs, const FrameDesc* __restrict__ desc, const QuantTable* __restrict__ qts,
                                                        uint8_t* __restrict__ dst, int n, int H, int W, int bw, int bh) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;
    if (desc[f].restart_interval == 0) return;       // decoded by jpeg_frame_kernel (uniform per CTA)
    __shared__ uint16_t sq[64];
    // (every thread of the CTA works on frame f: stage its quantisation table once)
    if (threadIdx.x < 64) sq[threadIdx.x] = qts[desc[f].qt].q[threadIdx.x];
    __syncthreads();
    if (b >= bw * bh) return;
    int16_t cf[64];
    const uint4* cp = (const uint4*)(coefs + ((size_t)f * bw * bh + b) * 64);
#pragma unroll
    for (int i = 0; i < 8; i++) { uint4 v = cp[i]; *(uint4*)&cf[i * 8] = v; }
    uint8_t px[64];
    idct_islow_block(cf, sq, px);
    const int bx = b % bw, by = b / bw, x0 = bx * 8, y0 = by * 8;
    uint8_t* o = dst + (size_t)f * H * W;
    const bool wide = x0 + 8 <= W && (W & 7) == 0 && (reinterpret_cast<size_t>(dst) & 7) == 0 && ((size_t)H * W & 7) == 0;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        if (y0 + r >= H) break;
        uint8_t* row = o + (size_t)(y0 + r) * W + x0;
        if (wide) *(uint2*)row = *(uint2*)&px[r * 8];
        else for (int c = 0; c < 8 && x0 + c < W; c++) row[c] = px[r * 8 + c];
    }
}

// ---- the whole decode of one frame in one CTA ------------------------------------------------------------------------
constexpr int kJT = 768;                    // lanes per frame; 64 ints of coefficient workspace per lane live in shared memory

struct JpegShared {
    int coef[64 * kJT];                     // [coefficient][lane]: conflict-free, one column per lane
    uint32_t rec_p[kJT];                    // per sub-sequence: where its successor starts (bit position) ...
    uint32_t rec_kn[kJT];                   // ... the zigzag index expected there (low 8 bits) | blocks that start inside << 8
    int32_t rec_dc[kJT];                    // ... and the sum of their DC differences
    HuffTable tab[2];
    int quant[64];
    uint32_t warp_tot[32];
    uint32_t marker, total, tile_total;
};

__global__ void __launch_bounds__(kJT, 1) jpeg_frame_kernel(const uint8_t* __restrict__ blob, const FrameDesc* __restrict__ desc, const HuffTable* __restrict__ ht,
                                                           const QuantTable* __restrict__ qts, uint8_t* scratch, uint8_t* __restrict__ dst, int H, int W) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    JpegShared& sm = *reinterpret_cast<JpegShared*>(smem_raw);
    const int f = blockIdx.x, tid = threadIdx.x;
    const FrameDesc d = desc[f];
    if (d.restart_interval != 0) return;             // legacy pair (uniform per CTA)
    {
        const uint32_t* g0 = reinterpret_cast<const uint32_t*>(&ht[d.dc]); const uint32_t* g1 = reinterpret_cast<const uint32_t*>(&ht[d.ac]);
        uint32_t* s0 = reinterpret_cast<uint32_t*>(&sm.tab[0]); uint32_t* s1 = reinterpret_cast<uint32_t*>(&sm.tab[1]);
        for (int i = tid; i < (int)(sizeof(HuffTable) / 4); i += kJT) { s0[i] = g0[i]; s1[i] = g1[i]; }
        if (tid < 64) sm.quant[tid] = qts[d.qt].q[tid];
        if (tid == 0) sm.marker = 0xFFFFFFFFu;
#pragma unroll 8
        for (int i = 0; i < 64; i++) sm.coef[i * kJT + tid] = 0;
    }
    __syncthreads();

    // ---- phase 0: copy the scan without its stuffed zero bytes, up to the first marker ------------------------------
    const uint8_t* raw = blob + d.scan_offset;
    const uint32_t raw_len = (uint32_t)(d.scan_end - d.scan_offset);
    uint8_t* ds = scratch + d.ds_offset;
    uint32_t out_base = 0;
    for (uint32_t t0 = 0; t0 < raw_len; t0 += 16u * kJT) {
        const uint32_t i0 = t0 + 16u * tid;
        uint8_t b[16]; uint32_t keep = 0;
        uint32_t prev = (i0 > 0 && i0 <= raw_len) ? raw[i0 - 1] : 0;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const uint32_t idx = i0 + i;
            const uint32_t cur = idx < raw_len ? raw[idx] : 0xD9u;      // past the end: behaves like an EOI after a trailing 0xFF
            b[i] = (uint8_t)cur;
            if (idx <= raw_len && prev == 0xFFu && cur != 0u && idx > 0) atomicMin(&sm.marker, idx - 1);
            if (idx < raw_len && !(prev == 0xFFu && cur == 0u)) keep |= 1u << i;
            prev = cur;
        }
        __syncthreads();
        const uint32_t m = sm.marker;
        if (m < i0 + 16u) keep &= (m <= i0) ? 0u : ((1u << (m - i0)) - 1u);       // nothing at or after the marker's 0xFF
        uint32_t tile_total;
        uint32_t o = out_base + cta_scan_excl<kJT>(__popc(keep), sm.warp_tot, &tile_total);
#pragma unroll
        for (int i = 0; i < 16; i++) if (keep & (1u << i)) ds[o++] = b[i];
        out_base += tile_total;
        if (m != 0xFFFFFFFFu) break;                  // uniform
    }
    const uint32_t L = out_base;                     // de-stuffed bytes
    const uint32_t last_word = (L + 3u) / 4u;        // index of the first all-padding word
    if (tid < 12) { const uint32_t z = L + tid; if (z < 4u * (last_word + 2u)) ds[z] = 0; }
    __syncthreads();
    uint32_t* words = reinterpret_cast<uint32_t*>(ds);
    for (uint32_t i = tid; i < last_word + 2u; i += kJT) words[i] = __byte_perm(words[i], 0, 0x0123);      // big-endian bit order
    __syncthreads();

    // ---- phases 1 and 2: every lane decodes its own sub-sequence, then keeps going until it meets a recorded state --------
    const uint32_t total_bits = L * 8u;
    const uint32_t S = scan_subseq_bits(total_bits, kJT);
    const uint32_t nsub = total_bits ? (total_bits + S - 1u) / S : 1u;       // an empty scan is still decoded (zero bits) by lane 0
    const HuffTable& dc = sm.tab[0]; const HuffTable& ac = sm.tab[1];
    ScanState st; st.p = (uint32_t)tid * S; st.k = 0;
    bool active = false;
    if ((uint32_t)tid < nsub) {
        uint32_t nb; int32_t dcs;
        const uint32_t hi = min((uint32_t)(tid + 1) * S, total_bits);
        scan_count(words, last_word, dc, ac, st, hi, &nb, &dcs);
        sm.rec_p[tid] = st.p; sm.rec_kn[tid] = (uint32_t)st.k | (nb << 8); sm.rec_dc[tid] = dcs;
        active = (uint32_t)tid + 1u < nsub;
    }
    for (uint32_t r = 1; __syncthreads_or(active); r++) {
        if (active) {
            const uint32_t tgt = (uint32_t)tid + r;
            const uint32_t hi = min((tgt + 1u) * S, total_bits);
            uint32_t nb; int32_t dcs;
            scan_count(words, last_word, dc, ac, st, hi, &nb, &dcs);
            const bool met = sm.rec_p[tgt] == st.p && (sm.rec_kn[tgt] & 0xFFu) == (uint32_t)st.k;
            sm.rec_p[tgt] = st.p; sm.rec_kn[tgt] = (uint32_t)st.k | (nb << 8); sm.rec_dc[tgt] = dcs;      // the last writer started from the true state
            if (met || tgt + 1u >= nsub) active = false;
        }
    }

    // ---- phase 3: first block and DC predictor of every sub-sequence ------------------------------------------------------
    uint32_t dummy;
    const uint32_t my_nb = (uint32_t)tid < nsub ? sm.rec_kn[tid] >> 8 : 0u;
    const uint32_t my_dc = (uint32_t)tid < nsub ? (uint32_t)sm.rec_dc[tid] : 0u;
    uint32_t blk = cta_scan_excl<kJT>(my_nb, sm.warp_tot, &dummy);
    int pred = (int)cta_scan_excl<kJT>(my_dc, sm.warp_tot, &dummy);

    // ---- phase 4: decode again, this time for real: coefficients -> shared memory -> IDCT -> pixels ---------------------
    if ((uint32_t)tid >= nsub) return;
    if (tid == 0) { st.p = 0; st.k = 0; } else { st.p = sm.rec_p[tid - 1]; st.k = (int)(sm.rec_kn[tid - 1] & 0xFFu); }
    const uint32_t hi = (uint32_t)tid + 1u == nsub ? 0xFFFFFFFFu : (uint32_t)(tid + 1) * S;      // the last lane also decodes what a truncated stream leaves over (zero bits, like libjpeg)
    const int bw = (W + 7) >> 3, nblocks = bw * ((H + 7) >> 3);
    uint8_t* frame = dst + (size_t)f * H * W;
    const bool wide = (W & 7) == 0 && (reinterpret_cast<size_t>(dst) & 7) == 0 && (((size_t)H * W) & 7) == 0;
    int* cf = sm.coef + tid;
    int kz;
    while (st.k != 0 && st.p < hi) scan_symbol(words, last_word, dc, ac, st, &kz);      // tail of a block that belongs to an earlier lane
    while (st.k == 0 && st.p < hi && blk < (uint32_t)nblocks) {
        pred += scan_symbol(words, last_word, dc, ac, st, &kz);
        cf[0] = (int)(int16_t)pred;
        uint64_t mask = 0;
        while (st.k != 0) {
            const int v = scan_symbol(words, last_word, dc, ac, st, &kz);
            if (kz > 0) { const int nat = zigzag_to_natural(kz); cf[nat * kJT] = v; mask |= 1ull << nat; }
        }
        const int x0 = (int)(blk % (uint32_t)bw) * 8, y0 = (int)(blk / (uint32_t)bw) * 8;
        idct_islow_inplace([cf](int i) -> int& { return cf[i * kJT]; }, sm.quant, mask,
                           [&](int r, const uint8_t* row) {
                               if (y0 + r >= H) return;
                               uint8_t* o = frame + (size_t)(y0 + r) * W + x0;
                               if (wide) {
                                   uint2 v;
                                   v.x = (uint32_t)row[0] | ((uint32_t)row[1] << 8) | ((uint32_t)row[2] << 16) | ((uint32_t)row[3] << 24);
                                   v.y = (uint32_t)row[4] | ((uint32_t)row[5] << 8) | ((uint32_t)row[6] << 16) | ((uint32_t)row[7] << 24);
                                   *reinterpret_cast<uint2*>(o) = v;
                               } else for (int c = 0; c < 8 && x0 + c < W; c++) o[c] = row[c];
                           });
        if (mask & ~1ull) {
#pragma unroll 8
            for (int i = 1; i < 64; i++) cf[i * kJT] = 0;
        }
        blk++;
    }
}

// Bytes of de-stuffing scratch a frame with `scan_bytes` of entropy-coded data needs (multiple of 16).
size_t jpeg_scratch_bytes(uint64_t scan_bytes) { return (size_t)((scan_bytes + 16 + 15) & ~(uint64_t)15); }

int launch_jpeg_decode(const uint8_t* blob, const void* desc, const void* hts, const void* qts, uint8_t* scratch, int16_t* coefs, uint8_t* dst,
                       int n, int n_restart, int H, int W, cudaStream_t s) {
    const int bw = (W + 7) / 8, bh = (H + 7) / 8;
    int nk = 0;
    if (n_restart < n) {
        // (the attribute is per function and per device: set on every call, setting it again is harmless)
        cudaFuncSetAttribute(jpeg_frame_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(JpegShared));
        jpeg_frame_kernel<<<n, kJT, sizeof(JpegShared), s>>>(blob, (const FrameDesc*)desc, (const HuffTable*)hts, (const QuantTable*)qts, scratch, dst, H, W);
        nk += 1;
    }
    if (n_restart > 0) {                       // streams with restart intervals: the one-lane-per-frame pair (coefs: n frames of int16 coefficients)
        cudaMemsetAsync(coefs, 0, (size_t)n * bw * bh * 64 * sizeof(int16_t), s);
        jpeg_huff_kernel<<<(n * 32 + 127) / 128, 128, 0, s>>>(blob, (const FrameDesc*)desc, (const HuffTable*)hts, coefs, n, bw * bh);
        dim3 grid((bw * bh + 127) / 128, n);
        jpeg_idct_kernel<<<grid, 128, 0, s>>>(coefs, (const FrameDesc*)desc, (const QuantTable*)qts, dst, n, H, W, bw, bh);
        nk += 2;
    }
    return nk;
}

}  // namespace dmc
