// dmc_jpeg_enc.cu -- frame-parallel baseline-JPEG ENCODER on sm_100a, byte-identical to cv2.imencode (libjpeg-turbo) of an
// 8UC1 image at a given quality (rules and primitives: dmc_jpeg_enc_core.h).
//
//   jpeg_enc_transform_kernel: one thread per 8x8 block of every frame of the group -- load with edge replication,
//             islow FDCT, quantisation, zigzag; writes the 64 int16 coefficients and an EncBlock (non-zero mask, AC bit
//             count, quantised DC).
//   jpeg_enc_entropy_kernel: one CTA per frame -- every lane owns a contiguous run of blocks; the lanes' bit counts
//             (AC + DC difference) are prefix-summed into bit offsets, every lane packs its blocks' codes into 32-bit
//             words (words it shares with a neighbour are OR-ed atomically into zeroed words), the last byte is padded,
//             and the scan is byte-stuffed tile by tile (count the 0xFF bytes per lane, prefix-sum, scatter with the 0x00
//             insertion) behind the header into the frame's slot; the frame's stream length goes to lens[f], and with
//             `desc` the FrameDesc the decoder of dmc_jpeg.cu needs to decode the slot in place.
//   jpeg_enc_gather_kernel: copies the streams from their slots to their final offsets, back to back.
//
// No host synchronisation between the kernels; the host only reads the lengths back to place the streams.
#include "dmc_common.cuh"
#include "dmc_jpeg_enc_core.h"
#include "dmc_kernels.cuh"

namespace dmc {

using namespace dmcjpeg;

JpegEncLayout jpeg_enc_layout(int rows, int cols) {
    JpegEncLayout l;
    l.blocks = (size_t)((rows + 7) / 8) * (size_t)((cols + 7) / 8);
    l.coef_bytes = l.blocks * 64 * sizeof(int16_t);
    l.info_bytes = l.blocks * sizeof(EncBlock);
    // packed scan of at most blocks * kEncMaxBlockBits bits; the decoder reuses the region as its de-stuffing scratch, which
    // takes the de-stuffed scan plus up to 12 bytes of padding words
    l.word_bytes = ((l.blocks * kEncMaxBlockBits + 7) / 8 + 16 + 15) & ~(size_t)15;
    l.slot_bytes = (jpeg_encode_bound(rows, cols) + 15) & ~(size_t)15;
    return l;
}

__global__ void __launch_bounds__(128) jpeg_enc_transform_kernel(const uint8_t* __restrict__ src, const EncTables* __restrict__ tabs, int16_t* __restrict__ coefs,
                                                                 EncBlock* __restrict__ info, int H, int W, int bw, int nb, uint32_t total) {
    __shared__ uint32_t s_qmul[64], s_qhalf[64], s_ac[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_ac[i] = tabs->ac[i];
    if (threadIdx.x < 64) { s_qmul[threadIdx.x] = tabs->qmul[threadIdx.x]; s_qhalf[threadIdx.x] = tabs->qhalf[threadIdx.x]; }
    __syncthreads();
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    const uint32_t f = g / (uint32_t)nb, b = g - f * (uint32_t)nb, by = b / (uint32_t)bw, bx = b - by * (uint32_t)bw;
    const uint8_t* frame = src + (size_t)f * H * W;
    const int x0 = (int)bx * 8, y0 = (int)by * 8;
    int d[64];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const uint8_t* row = frame + (size_t)min(y0 + r, H - 1) * W;
        if (x0 + 8 <= W && (reinterpret_cast<size_t>(row + x0) & 7) == 0) {      // adjacent threads: adjacent 8-byte pieces
            const uint2 v = *reinterpret_cast<const uint2*>(row + x0);
#pragma unroll
            for (int c = 0; c < 4; c++) { d[r * 8 + c] = (int)((v.x >> (8 * c)) & 0xFF) - 128; d[r * 8 + 4 + c] = (int)((v.y >> (8 * c)) & 0xFF) - 128; }
        } else {
#pragma unroll
            for (int c = 0; c < 8; c++) d[r * 8 + c] = (int)row[min(x0 + c, W - 1)] - 128;
        }
    }
    fdct_islow(d);
    int16_t zz[64];
    EncBlock e;
    e.nz = quantize_zigzag(d, s_qmul, s_qhalf, zz);
    e.ac_bits = block_ac_bits(zz, s_ac);
    e.dc = zz[0];
    uint4* cp = reinterpret_cast<uint4*>(coefs + (size_t)g * 64);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint4 v;
        v.x = (uint32_t)(uint16_t)zz[8 * i + 0] | ((uint32_t)(uint16_t)zz[8 * i + 1] << 16);
        v.y = (uint32_t)(uint16_t)zz[8 * i + 2] | ((uint32_t)(uint16_t)zz[8 * i + 3] << 16);
        v.z = (uint32_t)(uint16_t)zz[8 * i + 4] | ((uint32_t)(uint16_t)zz[8 * i + 5] << 16);
        v.w = (uint32_t)(uint16_t)zz[8 * i + 6] | ((uint32_t)(uint16_t)zz[8 * i + 7] << 16);
        cp[i] = v;
    }
    info[g] = e;
}

constexpr int kET = 1024;                   // lanes of the per-frame entropy CTA

__global__ void __launch_bounds__(kET, 1) jpeg_enc_entropy_kernel(const int16_t* __restrict__ coefs, const EncBlock* __restrict__ info, const EncTables* __restrict__ tabs,
                                                                  uint32_t* words_base, uint8_t* __restrict__ slots, uint32_t* __restrict__ lens, FrameDesc* __restrict__ desc,
                                                                  int nb, size_t word_bytes, size_t slot_bytes) {
    __shared__ uint32_t s_dc[16], s_ac[256], warp_tot[32];
    __shared__ uint8_t s_hdr[kEncHeaderBytes];
    const int f = blockIdx.x, tid = threadIdx.x;
    for (int i = tid; i < 256; i += kET) s_ac[i] = tabs->ac[i];
    if (tid < 16) s_dc[tid] = tabs->dc[tid];
    for (int i = tid; i < kEncHeaderBytes; i += kET) s_hdr[i] = tabs->header[i];
    __syncthreads();
    const EncBlock* inf = info + (size_t)f * nb;
    const int16_t* cf = coefs + (size_t)f * nb * 64;
    uint32_t* words = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(words_base) + (size_t)f * word_bytes);
    uint8_t* out = slots + (size_t)f * slot_bytes;

    // ---- bit offsets of the lanes ---------------------------------------------------------------------------------------
    const int per = (nb + kET - 1) / kET, b0 = min(tid * per, nb), b1 = min(b0 + per, nb);
    uint32_t bits = 0;
    {
        int prev = b0 > 0 ? inf[b0 - 1].dc : 0;
        for (int b = b0; b < b1; b++) { const int dc = inf[b].dc; bits += inf[b].ac_bits + block_dc_bits(dc - prev, s_dc); prev = dc; }
    }
    uint32_t T;
    const uint32_t B = cta_scan_excl<kET>(bits, warp_tot, &T), E = B + bits;

    // ---- pack: words shared with a neighbouring lane are zeroed first and OR-ed into ------------------------------------
    if (B & 31u) words[B >> 5] = 0;
    if (E & 31u) words[E >> 5] = 0;
    __syncthreads();
    {
        auto w = bw_start(B, [words](uint32_t wi, uint32_t v, bool partial) { if (partial) atomicOr(words + wi, v); else words[wi] = v; });
        int prev = b0 > 0 ? inf[b0 - 1].dc : 0;
        for (int b = b0; b < b1; b++) {
            const EncBlock e = inf[b];
            const int16_t* zz = cf + (size_t)b * 64;
            emit_block(w, e.dc - prev, e.nz, [zz](int k) { return (int)zz[k]; }, s_dc, s_ac);
            prev = e.dc;
        }
        bw_finish(w);
    }
    __syncthreads();
    if (tid == 0) pad_scan(words, T);
    __syncthreads();

    // ---- byte stuffing behind the header ----------------------------------------------------------------------------------
    const uint32_t L = (T + 7u) / 8u;
    uint32_t stuffed = 0;
    for (uint32_t t0 = 0; t0 < L; t0 += 16u * kET) {
        const uint32_t i0 = t0 + 16u * tid;
        uint32_t wv[4];
        stuff_load(words, L, i0, wv);
        uint32_t tile_ff;
        const uint32_t o = cta_scan_excl<kET>(stuff_count(wv, L, i0), warp_tot, &tile_ff);
        if (i0 < L) stuff_write(wv, L, i0, out + kEncHeaderBytes + i0 + stuffed + o);
        stuffed += tile_ff;
    }
    const uint32_t len = (uint32_t)kEncHeaderBytes + L + stuffed + 2u;
    for (int i = tid; i < kEncHeaderBytes; i += kET) out[i] = s_hdr[i];
    if (tid == 0) {
        out[len - 2] = 0xFF; out[len - 1] = 0xD9;
        lens[f] = len;
        if (desc) {
            FrameDesc d;
            d.scan_offset = (uint64_t)f * slot_bytes + kEncHeaderBytes;
            d.scan_end = (uint64_t)f * slot_bytes + len;
            d.restart_interval = 0; d.qt = 0; d.dc = 0; d.ac = 1;
            d.ds_offset = (uint64_t)f * word_bytes;
            desc[f] = d;
        }
    }
}

__global__ void __launch_bounds__(256) jpeg_enc_gather_kernel(const uint8_t* __restrict__ slots, size_t slot_bytes, const uint32_t* __restrict__ lens,
                                                              const uint64_t* __restrict__ offs, uint8_t* __restrict__ dst) {
    const int f = blockIdx.y;
    const uint8_t* s = slots + (size_t)f * slot_bytes;
    uint8_t* d = dst + offs[f];
    const uint32_t n = lens[f];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) d[i] = s[i];
}

int launch_jpeg_encode(const uint8_t* src, const void* tabs, void* coefs, void* info, void* words, uint8_t* slots, uint32_t* lens, void* desc,
                       int n, int H, int W, cudaStream_t s) {
    const JpegEncLayout l = jpeg_enc_layout(H, W);
    const int bw = (W + 7) / 8, nb = (int)l.blocks;
    const uint32_t total = (uint32_t)((size_t)n * nb);
    jpeg_enc_transform_kernel<<<(total + 127) / 128, 128, 0, s>>>(src, (const EncTables*)tabs, (int16_t*)coefs, (EncBlock*)info, H, W, bw, nb, total);
    jpeg_enc_entropy_kernel<<<n, kET, 0, s>>>((const int16_t*)coefs, (const EncBlock*)info, (const EncTables*)tabs, (uint32_t*)words, slots, lens,
                                              (FrameDesc*)desc, nb, l.word_bytes, l.slot_bytes);
    return 2;
}

int launch_jpeg_enc_gather(const uint8_t* slots, size_t slot_bytes, const uint32_t* lens, const uint64_t* offs, uint8_t* dst, int n, uint64_t max_len, cudaStream_t s) {
    const uint32_t gx = (uint32_t)((max_len + 256 * 16 - 1) / (256 * 16));
    jpeg_enc_gather_kernel<<<dim3(gx ? gx : 1, n), 256, 0, s>>>(slots, slot_bytes, lens, offs, dst);
    return 1;
}

}  // namespace dmc
