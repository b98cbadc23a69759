// dmc_jpeg_color.cu -- frame-parallel baseline colour JPEG decoder on sm_100a, bit-identical to cv2.imdecode(buf,
// IMREAD_COLOR) with libjpeg-turbo (islow IDCT, fancy upsampling, jdcolor.c YCbCr -> BGR).  The colour counterpart of
// dmc_jpeg.cu; the primitives are in dmc_jpeg_color_core.h.
//
//   jpeg_color_frame_kernel (streams without restart markers): ONE CTA per frame de-stuffs the scan, decodes it on all
//             lanes at once (self-synchronising sub-sequences whose state includes the block's position in the MCU),
//             prefix-sums block counts and the three components' DC differences, and in the final pass every lane
//             dequantises and inverse-transforms its blocks into the frame's component planes in device scratch.
//   legacy pair (streams with restart intervals): one lane per frame walks the scan into int16 coefficients, a second
//             kernel transforms one block per thread into the planes.
//   jpeg_color_convert_kernel: one output tile per CTA, upsampling and colour conversion of the planes to dense BGR.
#include "dmc_common.cuh"
#include "dmc_jpeg_color_core.h"
#include "dmc_kernels.cuh"

namespace dmc {

using namespace dmcjpeg;

// ---- restart-interval streams: entropy decoding, one warp (lane 0) per frame -----------------------------------------
__global__ void __launch_bounds__(128) jpeg_color_huff_kernel(const uint8_t* __restrict__ blob, const ColorFrameDesc* __restrict__ desc,
                                                              const HuffTable* __restrict__ ht, int16_t* __restrict__ coefs, int n) {
    __shared__ HuffTable s_tab[4][6];
    const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (f >= n) return;                              // uniform per warp
    const ColorFrameDesc d = desc[f];
    if (d.restart_interval == 0) return;             // decoded by jpeg_color_frame_kernel
    for (int t = 0; t < 6; t++) {
        const uint32_t* g = reinterpret_cast<const uint32_t*>(&ht[(t & 1) ? d.ac[t >> 1] : d.dc[t >> 1]]);
        uint32_t* s = reinterpret_cast<uint32_t*>(&s_tab[w][t]);
        for (int i = lane; i < (int)(sizeof(HuffTable) / 4); i += 32) s[i] = g[i];
    }
    __syncwarp();
    if (lane != 0) return;
    color_decode_serial(blob, d, s_tab[w], coefs + d.coef_offset * 64);
}

// ---- restart-interval streams: dequantise + islow IDCT into the planes, one thread per block -----------------------
__global__ void __launch_bounds__(128) jpeg_color_idct_kernel(const int16_t* __restrict__ coefs, const ColorFrameDesc* __restrict__ desc,
                                                              const QuantTable* __restrict__ qts, uint8_t* __restrict__ planes) {
    const int f = blockIdx.y;
    const ColorFrameDesc d = desc[f];
    if (d.restart_interval == 0) return;             // uniform per CTA
    __shared__ uint16_t sq[3][64];
    if (threadIdx.x < 64) for (int c = 0; c < 3; c++) sq[c][threadIdx.x] = qts[d.qt[c]].q[threadIdx.x];
    __syncthreads();
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= color_blocks(d)) return;
    int16_t cf[64];
    const uint4* cp = reinterpret_cast<const uint4*>(coefs + (d.coef_offset + b) * 64);
#pragma unroll
    for (int i = 0; i < 8; i++) *reinterpret_cast<uint4*>(&cf[i * 8]) = cp[i];
    int comp, stride;
    uint8_t* o = planes + d.plane_offset + color_block_origin(d, b, &comp, &stride);
    uint8_t px[64];
    idct_islow_block(cf, sq[comp], px);
#pragma unroll
    for (int r = 0; r < 8; r++) *reinterpret_cast<uint2*>(o + (size_t)r * stride) = *reinterpret_cast<const uint2*>(&px[r * 8]);
}

// ---- the entropy decode and IDCT of one frame in one CTA -------------------------------------------------------------
constexpr int kJCT = 768;                   // lanes per frame; 64 ints of coefficient workspace per lane live in shared memory

struct JpegColorShared {
    int coef[64 * kJCT];                    // [coefficient][lane]: conflict-free, one column per lane
    uint32_t rec_p[kJCT];                   // per sub-sequence: where its successor starts (bit position) ...
    uint32_t rec_km[kJCT];                  // ... the zigzag index (low 8 bits) and MCU position (<< 8) expected there ...
    uint32_t rec_nb[kJCT];                  // ... the blocks that start inside ...
    int32_t rec_dc[3][kJCT];                // ... and the sums of their DC differences, per component
    HuffTable tab[6];                       // DC, AC of Y, Cb, Cr
    int quant[3][64];
    uint32_t warp_tot[32];
    uint32_t marker;
};
static_assert(sizeof(JpegColorShared) <= 227 * 1024, "jpeg_color_frame_kernel exceeds the shared memory of a CTA");

__global__ void __launch_bounds__(kJCT, 1) jpeg_color_frame_kernel(const uint8_t* __restrict__ blob, const ColorFrameDesc* __restrict__ desc,
                                                                  const HuffTable* __restrict__ ht, const QuantTable* __restrict__ qts,
                                                                  uint8_t* scratch, uint8_t* __restrict__ planes) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    JpegColorShared& sm = *reinterpret_cast<JpegColorShared*>(smem_raw);
    const int f = blockIdx.x, tid = threadIdx.x;
    const ColorFrameDesc d = desc[f];
    if (d.restart_interval != 0) return;             // legacy pair (uniform per CTA)
    for (int t = 0; t < 6; t++) {
        const uint32_t* g = reinterpret_cast<const uint32_t*>(&ht[(t & 1) ? d.ac[t >> 1] : d.dc[t >> 1]]);
        uint32_t* s = reinterpret_cast<uint32_t*>(&sm.tab[t]);
        for (int i = tid; i < (int)(sizeof(HuffTable) / 4); i += kJCT) s[i] = g[i];
    }
    if (tid < 3 * 64) sm.quant[tid >> 6][tid & 63] = qts[d.qt[tid >> 6]].q[tid & 63];
    if (tid == 0) sm.marker = 0xFFFFFFFFu;
#pragma unroll 8
    for (int i = 0; i < 64; i++) sm.coef[i * kJCT + tid] = 0;
    __syncthreads();

    // ---- phase 0: copy the scan without its stuffed zero bytes, up to the first marker ----------------------------------
    const uint8_t* raw = blob + d.scan_offset;
    const uint32_t raw_len = (uint32_t)(d.scan_end - d.scan_offset);
    uint8_t* ds = scratch + d.ds_offset;
    uint32_t out_base = 0;
    for (uint32_t t0 = 0; t0 < raw_len; t0 += 16u * kJCT) {
        const uint32_t i0 = t0 + 16u * tid;
        uint8_t b[16]; uint32_t keep = 0;
        uint32_t prev = (i0 > 0 && i0 <= raw_len) ? raw[i0 - 1] : 0;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const uint32_t idx = i0 + i;
            const uint32_t cur = idx < raw_len ? raw[idx] : 0xD9u;
            b[i] = (uint8_t)cur;
            if (idx <= raw_len && prev == 0xFFu && cur != 0u && idx > 0) atomicMin(&sm.marker, idx - 1);
            if (idx < raw_len && !(prev == 0xFFu && cur == 0u)) keep |= 1u << i;
            prev = cur;
        }
        __syncthreads();
        const uint32_t m = sm.marker;
        if (m < i0 + 16u) keep &= (m <= i0) ? 0u : ((1u << (m - i0)) - 1u);
        uint32_t tile_total;
        uint32_t o = out_base + cta_scan_excl<kJCT>(__popc(keep), sm.warp_tot, &tile_total);
#pragma unroll
        for (int i = 0; i < 16; i++) if (keep & (1u << i)) ds[o++] = b[i];
        out_base += tile_total;
        if (m != 0xFFFFFFFFu) break;                  // uniform
    }
    const uint32_t L = out_base;
    const uint32_t last_word = (L + 3u) / 4u;
    if (tid < 12) { const uint32_t z = L + tid; if (z < 4u * (last_word + 2u)) ds[z] = 0; }
    __syncthreads();
    uint32_t* words = reinterpret_cast<uint32_t*>(ds);
    for (uint32_t i = tid; i < last_word + 2u; i += kJCT) words[i] = __byte_perm(words[i], 0, 0x0123);
    __syncthreads();

    // ---- phases 1 and 2: every lane decodes its own sub-sequence, then keeps going until it meets a recorded state ------
    const int bpm = color_blocks_per_mcu(d), ny = color_luma_blocks(d);
    const uint32_t total_bits = L * 8u;
    const uint32_t S = scan_subseq_bits(total_bits, kJCT);
    const uint32_t nsub = total_bits ? (total_bits + S - 1u) / S : 1u;
    ColorScanState st; st.p = (uint32_t)tid * S; st.k = 0; st.m = 0;
    bool active = false;
    if ((uint32_t)tid < nsub) {
        uint32_t nb; int32_t dcs[3];
        color_scan_count(words, last_word, sm.tab, ny, bpm, st, min((uint32_t)(tid + 1) * S, total_bits), &nb, dcs);
        sm.rec_p[tid] = st.p; sm.rec_km[tid] = (uint32_t)st.k | ((uint32_t)st.m << 8); sm.rec_nb[tid] = nb;
        sm.rec_dc[0][tid] = dcs[0]; sm.rec_dc[1][tid] = dcs[1]; sm.rec_dc[2][tid] = dcs[2];
        active = (uint32_t)tid + 1u < nsub;
    }
    for (uint32_t r = 1; __syncthreads_or(active); r++) {
        if (active) {
            const uint32_t tgt = (uint32_t)tid + r;
            uint32_t nb; int32_t dcs[3];
            color_scan_count(words, last_word, sm.tab, ny, bpm, st, min((tgt + 1u) * S, total_bits), &nb, dcs);
            const uint32_t km = (uint32_t)st.k | ((uint32_t)st.m << 8);
            const bool met = sm.rec_p[tgt] == st.p && sm.rec_km[tgt] == km;
            sm.rec_p[tgt] = st.p; sm.rec_km[tgt] = km; sm.rec_nb[tgt] = nb;      // the last writer started from the true state
            sm.rec_dc[0][tgt] = dcs[0]; sm.rec_dc[1][tgt] = dcs[1]; sm.rec_dc[2][tgt] = dcs[2];
            if (met || tgt + 1u >= nsub) active = false;
        }
    }

    // ---- phase 3: first block and the three DC predictors of every sub-sequence -----------------------------------------
    uint32_t dummy;
    const bool mine = (uint32_t)tid < nsub;
    uint32_t blk = cta_scan_excl<kJCT>(mine ? sm.rec_nb[tid] : 0u, sm.warp_tot, &dummy);
    int pred[3];
    for (int c = 0; c < 3; c++) pred[c] = (int)cta_scan_excl<kJCT>(mine ? (uint32_t)sm.rec_dc[c][tid] : 0u, sm.warp_tot, &dummy);

    // ---- phase 4: decode again, this time for real: coefficients -> shared memory -> IDCT -> planes ---------------------
    if (!mine) return;
    if (tid == 0) { st.p = 0; st.k = 0; st.m = 0; }
    else { st.p = sm.rec_p[tid - 1]; st.k = (int)(sm.rec_km[tid - 1] & 0xFFu); st.m = (int)(sm.rec_km[tid - 1] >> 8); }
    const uint32_t hi = (uint32_t)tid + 1u == nsub ? 0xFFFFFFFFu : (uint32_t)(tid + 1) * S;
    const uint32_t nblocks = color_blocks(d);
    uint8_t* frame = planes + d.plane_offset;
    int* cf = sm.coef + tid;
    int kz, comp;
    while (st.k != 0 && st.p < hi) color_scan_symbol(words, last_word, sm.tab, ny, bpm, st, &kz, &comp);      // tail of an earlier lane's block
    while (st.k == 0 && st.p < hi && blk < nblocks) {
        const int v = color_scan_symbol(words, last_word, sm.tab, ny, bpm, st, &kz, &comp);
        const int c = comp;
        pred[c] += v;
        cf[0] = (int)(int16_t)pred[c];
        uint64_t mask = 0;
        while (st.k != 0) {
            const int a = color_scan_symbol(words, last_word, sm.tab, ny, bpm, st, &kz, &comp);
            if (kz > 0) { const int nat = zigzag_to_natural(kz); cf[nat * kJCT] = a; mask |= 1ull << nat; }
        }
        int pc, stride;
        uint8_t* o = frame + color_block_origin(d, blk, &pc, &stride);
        idct_islow_inplace([cf](int i) -> int& { return cf[i * kJCT]; }, sm.quant[c], mask,
                           [&](int r, const uint8_t* row) {
                               uint2 w;
                               w.x = (uint32_t)row[0] | ((uint32_t)row[1] << 8) | ((uint32_t)row[2] << 16) | ((uint32_t)row[3] << 24);
                               w.y = (uint32_t)row[4] | ((uint32_t)row[5] << 8) | ((uint32_t)row[6] << 16) | ((uint32_t)row[7] << 24);
                               *reinterpret_cast<uint2*>(o + (size_t)r * stride) = w;
                           });
        if (mask & ~1ull) {
#pragma unroll 8
            for (int i = 1; i < 64; i++) cf[i * kJCT] = 0;
        }
        blk++;
    }
}

// ---- upsampling and colour conversion: one 64 x 4 output tile per CTA ------------------------------------------------
__global__ void __launch_bounds__(256) jpeg_color_convert_kernel(const ColorFrameDesc* __restrict__ desc, const YccTables* __restrict__ ycc,
                                                                 const uint8_t* __restrict__ planes, uint8_t* __restrict__ dst, int H, int W) {
    __shared__ YccTables t;
    for (int i = threadIdx.x; i < (int)(sizeof(YccTables) / 4); i += 256) reinterpret_cast<int32_t*>(&t)[i] = reinterpret_cast<const int32_t*>(ycc)[i];
    __syncthreads();
    const int f = blockIdx.z, x = blockIdx.x * 64 + (threadIdx.x & 63), y = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (x >= W || y >= H) return;
    const ColorFrameDesc d = desc[f];
    uint8_t bgr[3];
    color_pixel_bgr(d, planes + d.plane_offset, t, H, W, x, y, bgr);
    uint8_t* o = dst + ((size_t)f * H * W + (size_t)y * W + x) * 3;
    o[0] = bgr[0]; o[1] = bgr[1]; o[2] = bgr[2];
}

int launch_jpeg_color_decode(const uint8_t* blob, const void* desc, const void* hts, const void* qts, const void* ycc, uint8_t* scratch, uint8_t* planes,
                             int16_t* coefs, uint8_t* dst, int n, int n_restart, uint32_t max_blocks, int H, int W, cudaStream_t s) {
    const ColorFrameDesc* dd = (const ColorFrameDesc*)desc;
    int nk = 0;
    if (n_restart < n) {
        cudaFuncSetAttribute(jpeg_color_frame_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(JpegColorShared));
        jpeg_color_frame_kernel<<<n, kJCT, sizeof(JpegColorShared), s>>>(blob, dd, (const HuffTable*)hts, (const QuantTable*)qts, scratch, planes);
        nk += 1;
    }
    if (n_restart > 0) {                       // coefs: the restart frames' blocks at their coef_offset, zeroed here
        jpeg_color_huff_kernel<<<(n * 32 + 127) / 128, 128, 0, s>>>(blob, dd, (const HuffTable*)hts, coefs, n);
        jpeg_color_idct_kernel<<<dim3((max_blocks + 127) / 128, n), 128, 0, s>>>(coefs, dd, (const QuantTable*)qts, planes);
        nk += 2;
    }
    jpeg_color_convert_kernel<<<dim3((W + 63) / 64, (H + 3) / 4, n), 256, 0, s>>>(dd, (const YccTables*)ycc, planes, dst, H, W);
    return nk + 1;
}

}  // namespace dmc
