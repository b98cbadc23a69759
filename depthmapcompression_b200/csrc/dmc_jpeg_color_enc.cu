// dmc_jpeg_color_enc.cu -- frame-parallel baseline colour JPEG ENCODER on sm_100a, byte-identical to cv2.imencode
// (libjpeg-turbo) of an 8UC3 BGR image at a given quality and sampling (rules and primitives: dmc_jpeg_color_enc_core.h;
// transform, bit packing and stuffing: dmc_jpeg_enc_core.h).  The colour counterpart of dmc_jpeg_enc.cu.
//
//   jpeg_color_enc_transform_kernel: one thread per block of every frame of the group, the luma blocks of a frame first
//             and then its chroma blocks (Cb and Cr of one MCU side by side), so that a warp runs one path and the two
//             chroma threads of an MCU read the same pixels.  Each loads the BGR pixels its block needs at libjpeg's
//             edge coordinates, converts and downsamples them, and writes the int16 coefficients and the EncBlock at the
//             block's position in the scan.  A dummy block transforms its source block and keeps only the DC.
//   jpeg_color_enc_entropy_kernel: one CTA per frame -- every lane owns a contiguous run of MCUs, starting its three DC
//             predictors from the previous MCU's blocks; then the gray encoder's bit-offset scan, word packing and
//             stuffing behind the 623-byte header, and with `desc` the ColorFrameDesc that decodes the slot in place.
//   jpeg_enc_gather_kernel (dmc_jpeg_enc.cu) places the streams back to back.
#include "dmc_common.cuh"
#include "dmc_jpeg_color_enc_core.h"
#include "dmc_kernels.cuh"

namespace dmc {

using namespace dmcjpeg;

JpegEncLayout jpeg_color_enc_layout(int rows, int cols, int hy, int vy) {
    JpegEncLayout l;
    l.blocks = color_enc_blocks(color_enc_geom(rows, cols, hy, vy));
    l.coef_bytes = l.blocks * 64 * sizeof(int16_t);
    l.info_bytes = l.blocks * sizeof(EncBlock);
    // packed scan of at most blocks * kColorEncMaxBlockBits bits; the colour decoder reuses the region as its de-stuffing
    // scratch, which takes the de-stuffed scan (that many bytes at most) plus up to 12 bytes of padding words
    l.word_bytes = ((l.blocks * kColorEncMaxBlockBits + 7) / 8 + 16 + 15) & ~(size_t)15;
    l.slot_bytes = (jpeg_encode_color_bound(rows, cols, hy, vy) + 15) & ~(size_t)15;
    l.opt_bytes = 0;
    return l;
}

__global__ void __launch_bounds__(128) jpeg_color_enc_transform_kernel(const uint8_t* __restrict__ src, const EncColorTables* __restrict__ tabs,
                                                                       int16_t* __restrict__ coefs, EncBlock* __restrict__ info, ColorEncGeom g,
                                                                       uint32_t nb, uint32_t total) {
    __shared__ uint32_t s_qmul[2][64], s_qhalf[2][64], s_ac[2][256];
    for (int i = threadIdx.x; i < 512; i += blockDim.x) (&s_ac[0][0])[i] = (&tabs->ac[0][0])[i];
    (&s_qmul[0][0])[threadIdx.x] = (&tabs->qmul[0][0])[threadIdx.x];
    (&s_qhalf[0][0])[threadIdx.x] = (&tabs->qhalf[0][0])[threadIdx.x];
    __syncthreads();
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    // thread -> block of the scan: a frame's luma blocks MCU by MCU, then its chroma blocks
    const uint32_t f = t / nb, i = t - f * nb, nm = nb / (uint32_t)g.bpm, nl = nm * (uint32_t)g.ny;
    const uint32_t b = i < nl ? (i / (uint32_t)g.ny) * (uint32_t)g.bpm + i % (uint32_t)g.ny
                              : ((i - nl) >> 1) * (uint32_t)g.bpm + (uint32_t)g.ny + ((i - nl) & 1u);
    const uint8_t* frame = src + (size_t)f * g.rows * g.cols * 3;
    const int W = g.cols;
    auto px = [frame, W](int x, int y, int* B, int* G, int* R) {
        const uint8_t* p = frame + ((size_t)y * W + x) * 3;
        *B = __ldg(p); *G = __ldg(p + 1); *R = __ldg(p + 2);
    };
    int16_t zz[64];
    const EncBlock e = color_transform_block(g, px, b, s_qmul, s_qhalf, s_ac, zz);
    const size_t gb = (size_t)f * nb + b;
    uint4* cp = reinterpret_cast<uint4*>(coefs + gb * 64);
#pragma unroll
    for (int k = 0; k < 8; k++) {
        uint4 v;
        v.x = (uint32_t)(uint16_t)zz[8 * k + 0] | ((uint32_t)(uint16_t)zz[8 * k + 1] << 16);
        v.y = (uint32_t)(uint16_t)zz[8 * k + 2] | ((uint32_t)(uint16_t)zz[8 * k + 3] << 16);
        v.z = (uint32_t)(uint16_t)zz[8 * k + 4] | ((uint32_t)(uint16_t)zz[8 * k + 5] << 16);
        v.w = (uint32_t)(uint16_t)zz[8 * k + 6] | ((uint32_t)(uint16_t)zz[8 * k + 7] << 16);
        cp[k] = v;
    }
    info[gb] = e;
}

constexpr int kCET = 1024;                  // lanes of the per-frame entropy CTA

__global__ void __launch_bounds__(kCET, 1) jpeg_color_enc_entropy_kernel(const int16_t* __restrict__ coefs, const EncBlock* __restrict__ info,
                                                                         const EncColorTables* __restrict__ tabs, uint32_t* words_base, uint8_t* __restrict__ slots,
                                                                         uint32_t* __restrict__ lens, ColorFrameDesc* __restrict__ desc, ColorFrameDesc tmpl,
                                                                         uint64_t plane_bytes, int nb, int bpm, int ny, size_t word_bytes, size_t slot_bytes) {
    __shared__ uint32_t s_dc[2][16], s_ac[2][256], warp_tot[32];
    __shared__ uint8_t s_hdr[kColorEncHeaderBytes];
    const int f = blockIdx.x, tid = threadIdx.x;
    for (int i = tid; i < 512; i += kCET) (&s_ac[0][0])[i] = (&tabs->ac[0][0])[i];
    if (tid < 32) (&s_dc[0][0])[tid] = (&tabs->dc[0][0])[tid];
    for (int i = tid; i < kColorEncHeaderBytes; i += kCET) s_hdr[i] = tabs->header[i];
    __syncthreads();
    const EncBlock* inf = info + (size_t)f * nb;
    const int16_t* cf = coefs + (size_t)f * nb * 64;
    uint32_t* words = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(words_base) + (size_t)f * word_bytes);
    uint8_t* out = slots + (size_t)f * slot_bytes;

    // ---- bit offsets of the lanes: lane j owns MCUs [m0, m1) ---------------------------------------------------------------
    const int nm = nb / bpm, per = (nm + kCET - 1) / kCET, m0 = min(tid * per, nm), m1 = min(m0 + per, nm);
    const int p0 = m0 > 0 ? inf[m0 * bpm - 3].dc : 0, p1 = m0 > 0 ? inf[m0 * bpm - 2].dc : 0, p2 = m0 > 0 ? inf[m0 * bpm - 1].dc : 0;
    uint32_t bits = 0;
    {
        int q0 = p0, q1 = p1, q2 = p2;
        for (int b = m0 * bpm, pos = 0; b < m1 * bpm; b++, pos = pos + 1 == bpm ? 0 : pos + 1) {
            const int c = pos < ny ? 0 : pos - ny + 1, dc = inf[b].dc;
            bits += inf[b].ac_bits + block_dc_bits(dc - (c == 0 ? q0 : c == 1 ? q1 : q2), s_dc[c > 0]);
            if (c == 0) q0 = dc; else if (c == 1) q1 = dc; else q2 = dc;
        }
    }
    uint32_t T;
    const uint32_t B = cta_scan_excl<kCET>(bits, warp_tot, &T), E = B + bits;

    // ---- pack: words shared with a neighbouring lane are zeroed first and OR-ed into ------------------------------------
    if (B & 31u) words[B >> 5] = 0;
    if (E & 31u) words[E >> 5] = 0;
    __syncthreads();
    {
        auto w = bw_start(B, [words](uint32_t wi, uint32_t v, bool partial) { if (partial) atomicOr(words + wi, v); else words[wi] = v; });
        int q0 = p0, q1 = p1, q2 = p2;
        for (int b = m0 * bpm, pos = 0; b < m1 * bpm; b++, pos = pos + 1 == bpm ? 0 : pos + 1) {
            const int c = pos < ny ? 0 : pos - ny + 1, k = c > 0;
            const EncBlock e = inf[b];
            const int16_t* zz = cf + (size_t)b * 64;
            emit_block(w, e.dc - (c == 0 ? q0 : c == 1 ? q1 : q2), e.nz, [zz](int i) { return (int)zz[i]; }, s_dc[k], s_ac[k]);
            if (c == 0) q0 = e.dc; else if (c == 1) q1 = e.dc; else q2 = e.dc;
        }
        bw_finish(w);
    }
    __syncthreads();
    if (tid == 0) pad_scan(words, T);
    __syncthreads();

    // ---- byte stuffing behind the header ----------------------------------------------------------------------------------
    const uint32_t L = (T + 7u) / 8u;
    uint32_t stuffed = 0;
    for (uint32_t t0 = 0; t0 < L; t0 += 16u * kCET) {
        const uint32_t i0 = t0 + 16u * tid;
        uint32_t wv[4];
        stuff_load(words, L, i0, wv);
        uint32_t tile_ff;
        const uint32_t o = cta_scan_excl<kCET>(stuff_count(wv, L, i0), warp_tot, &tile_ff);
        if (i0 < L) stuff_write(wv, L, i0, out + kColorEncHeaderBytes + i0 + stuffed + o);
        stuffed += tile_ff;
    }
    const uint32_t len = (uint32_t)kColorEncHeaderBytes + L + stuffed + 2u;
    for (int i = tid; i < kColorEncHeaderBytes; i += kCET) out[i] = s_hdr[i];
    if (tid == 0) {
        out[len - 2] = 0xFF; out[len - 1] = 0xD9;
        lens[f] = len;
        if (desc) {
            ColorFrameDesc d = tmpl;
            d.scan_offset = (uint64_t)f * slot_bytes + kColorEncHeaderBytes;
            d.scan_end = (uint64_t)f * slot_bytes + len;
            d.ds_offset = (uint64_t)f * word_bytes;
            d.plane_offset = (uint64_t)f * plane_bytes;
            d.coef_offset = 0;
            desc[f] = d;
        }
    }
}

int launch_jpeg_color_encode(const uint8_t* src, const void* tabs, void* coefs, void* info, void* words, uint8_t* slots, uint32_t* lens,
                             void* desc, const ColorFrameDesc* tmpl, uint64_t plane_bytes, int n, int H, int W, int hy, int vy, cudaStream_t s) {
    const ColorEncGeom g = color_enc_geom(H, W, hy, vy);
    const JpegEncLayout l = jpeg_color_enc_layout(H, W, hy, vy);
    const uint32_t nb = (uint32_t)l.blocks, total = (uint32_t)((size_t)n * nb);
    jpeg_color_enc_transform_kernel<<<(total + 127) / 128, 128, 0, s>>>(src, (const EncColorTables*)tabs, (int16_t*)coefs, (EncBlock*)info, g, nb, total);
    ColorFrameDesc t{};
    if (tmpl) t = *tmpl;
    jpeg_color_enc_entropy_kernel<<<n, kCET, 0, s>>>((const int16_t*)coefs, (const EncBlock*)info, (const EncColorTables*)tabs, (uint32_t*)words, slots, lens,
                                                     (ColorFrameDesc*)desc, t, plane_bytes, (int)nb, g.bpm, g.ny, l.word_bytes, l.slot_bytes);
    return 2;
}

}  // namespace dmc
