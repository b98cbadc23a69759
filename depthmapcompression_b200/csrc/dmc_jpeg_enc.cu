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
// With optimised Huffman tables (cv2.IMWRITE_JPEG_OPTIMIZE) the transform kernel also counts each frame's AC symbols,
//   jpeg_enc_table_kernel: one CTA per frame -- counts the DC categories, then one warp per table class builds the
//             frame's optimal table (jpeg_gen_optimal_table, dmc_jpeg_enc_core.h), and writes the frame's code tables and
//             header (EncFrameCode) and, for degradeJPEG, the decoder's HuffTable pair,
// and the entropy kernel recounts the AC bits with the frame's tables and writes the frame's header length.
//
// No host synchronisation between the kernels; the host only reads the lengths back to place the streams.
#include "dmc_common.cuh"
#include "dmc_jpeg_enc_core.h"
#include "dmc_kernels.cuh"

namespace dmc {

using namespace dmcjpeg;

JpegEncLayout jpeg_enc_layout(int rows, int cols, bool optimize) {
    JpegEncLayout l;
    l.blocks = (size_t)((rows + 7) / 8) * (size_t)((cols + 7) / 8);
    l.coef_bytes = l.blocks * 64 * sizeof(int16_t);
    l.info_bytes = l.blocks * sizeof(EncBlock);
    // packed scan of at most blocks * (max block bits) bits; the decoder reuses the region as its de-stuffing scratch,
    // which takes the de-stuffed scan plus up to 12 bytes of padding words
    l.word_bytes = ((l.blocks * (optimize ? kEncMaxBlockBitsOpt : kEncMaxBlockBits) + 7) / 8 + 16 + 15) & ~(size_t)15;
    l.slot_bytes = (jpeg_encode_bound(rows, cols, optimize) + 15) & ~(size_t)15;
    l.opt_bytes = optimize ? ((256 * sizeof(uint32_t) + sizeof(EncFrameCode) + 15) & ~(size_t)15) : 0;
    return l;
}

// hist (kOpt): the AC symbol counts of every frame, 256 per frame, zeroed before the launch.  A CTA's blocks span at
// most two frames when a frame has 128 blocks or more; those two are counted in shared memory, any others directly.
template <bool kOpt>
__global__ void __launch_bounds__(128) jpeg_enc_transform_kernel(const uint8_t* __restrict__ src, const EncTables* __restrict__ tabs, int16_t* __restrict__ coefs,
                                                                 EncBlock* __restrict__ info, uint32_t* __restrict__ hist, int H, int W, int bw, int nb, uint32_t total) {
    __shared__ uint32_t s_qmul[64], s_qhalf[64], s_ac[256], s_hist[kOpt ? 512 : 1];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_ac[i] = tabs->ac[i];
    if (threadIdx.x < 64) { s_qmul[threadIdx.x] = tabs->qmul[threadIdx.x]; s_qhalf[threadIdx.x] = tabs->qhalf[threadIdx.x]; }
    if (kOpt) for (int i = threadIdx.x; i < 512; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x, f_lo = blockIdx.x * blockDim.x / (uint32_t)nb;
    if (!kOpt && g >= total) return;
    if (g < total) {
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
        if (kOpt) {                                   // AC bits are counted by the entropy kernel, with the frame's tables
            uint32_t* h = f - f_lo < 2u ? s_hist + 256 * (f - f_lo) : hist + (size_t)f * 256;
            block_ac_symbols(zz, [h](int sym, int c) { atomicAdd(h + sym, (uint32_t)c); });
            e.ac_bits = 0;
        } else {
            e.ac_bits = block_ac_bits(zz, s_ac);
        }
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
    if (kOpt) {
        __syncthreads();
        const uint32_t n = total / (uint32_t)nb;
        for (int i = threadIdx.x; i < 512; i += blockDim.x)
            if (s_hist[i] && f_lo + i / 256 < n) atomicAdd(hist + (size_t)(f_lo + i / 256) * 256 + (i & 255), s_hist[i]);
    }
}

// One warp builds the optimal table of one class from hist[0 .. nsym) (dmc_jpeg_enc_core.h): BITS, HUFFVAL (n symbols)
// and the code table.  cnt (kOptMaxLen + 1 entries) and code (256) are zero on entry.
__device__ void build_opt_table(const uint32_t* hist, int nsym, uint32_t* cnt, uint32_t* start, uint8_t* bits, uint8_t* vals, int* n_out, uint32_t* code) {
    const int lane = threadIdx.x & 31;
    OptLane L;
    opt_lane_init(L, hist, nsym, lane);
    for (;;) {
        uint32_t f; int s;
        opt_lane_min(L, lane, -1, &f, &s);
        const uint32_t f1 = __reduce_min_sync(0xFFFFFFFFu, f);
        const int c1 = __reduce_max_sync(0xFFFFFFFFu, f == f1 ? s : -1);
        opt_lane_min(L, lane, c1, &f, &s);
        const uint32_t f2 = __reduce_min_sync(0xFFFFFFFFu, f);
        const int c2 = __reduce_max_sync(0xFFFFFFFFu, f == f2 ? s : -1);
        if (c2 < 0) break;
        opt_lane_merge(L, lane, c1, c2, f2);
    }
#pragma unroll
    for (int k = 0; k < kOptPer; k++) if (L.cs[k]) atomicAdd(cnt + L.cs[k], 1u);
    __syncwarp();
    if (lane == 0) {                              // first HUFFVAL position of each codesize, symbols 0..255
        uint32_t acc = 0;
        for (int c = 0; c <= kOptMaxLen; c++) { start[c] = acc; acc += cnt[c] - (c == L.cs[8] ? 1u : 0u); }
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 8; k++) {                 // symbols 32 k + lane in ascending order: rank among equal codesizes
        const int c = L.cs[k];
        const unsigned same = __match_any_sync(0xFFFFFFFFu, c);
        if (c) vals[start[c] + __popc(same & ((1u << lane) - 1u))] = (uint8_t)(32 * k + lane);
        __syncwarp();
        if (c && lane == __ffs(same) - 1) start[c] += __popc(same);
        __syncwarp();
    }
    if (lane == 0) *n_out = opt_fold(cnt, bits);
    __syncwarp();
    const int n = *n_out;
    for (int p = lane; p < n; p += 32) code[vals[p]] = opt_code(bits, p);
}

constexpr int kTT = 1024;                   // threads of the per-frame table CTA

__global__ void __launch_bounds__(kTT) jpeg_enc_table_kernel(const EncBlock* __restrict__ info, const EncTables* __restrict__ tabs, const uint32_t* __restrict__ hist,
                                                             EncFrameCode* __restrict__ code, HuffTable* __restrict__ huff, int nb) {
    __shared__ uint32_t s_hist[2][256], s_cnt[2][kOptMaxLen + 1], s_start[2][kOptMaxLen + 1], s_code[2][256];
    __shared__ uint8_t s_bits[2][16], s_vals[2][256];
    __shared__ int s_n[2];
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const EncBlock* inf = info + (size_t)f * nb;
    for (int i = tid; i < 256; i += kTT) { s_hist[0][i] = 0; s_hist[1][i] = hist[(size_t)f * 256 + i]; s_code[0][i] = 0; s_code[1][i] = 0; }
    for (int i = tid; i < 2 * (kOptMaxLen + 1); i += kTT) (&s_cnt[0][0])[i] = 0;
    __syncthreads();
    {                                             // DC categories: lane c of every warp counts category c
        uint32_t cnt = 0;
        for (int b0 = warp * 32; b0 < nb; b0 += kTT) {
            const int b = b0 + lane;
            const int cat = b < nb ? bit_length((uint32_t)abs(inf[b].dc - (b > 0 ? inf[b - 1].dc : 0))) : 16;
#pragma unroll
            for (int c = 0; c < 12; c++) { const unsigned m = __ballot_sync(0xFFFFFFFFu, cat == c); if (lane == c) cnt += __popc(m); }
        }
        if (lane < 12 && cnt) atomicAdd(&s_hist[0][lane], cnt);
    }
    __syncthreads();
    if (warp < 2) build_opt_table(s_hist[warp], warp ? 256 : 16, s_cnt[warp], s_start[warp], s_bits[warp], s_vals[warp], &s_n[warp], s_code[warp]);
    __syncthreads();
    EncFrameCode* fc = code + f;
    const int n_dc = s_n[0], n_ac = s_n[1], sos = kEncHeaderDhtAt + 42 + n_dc + n_ac;
    for (int i = tid; i < 256; i += kTT) { fc->ac[i] = s_code[1][i]; if (i < 16) fc->dc[i] = s_code[0][i]; }
    for (int i = tid; i < kEncHeaderDhtAt; i += kTT) fc->header[i] = tabs->header[i];
    for (int i = tid; i < kEncSosBytes; i += kTT) fc->header[sos + i] = tabs->header[kEncHeaderBytes - kEncSosBytes + i];
    if (tid == 0) {
        const int dc_len = opt_write_dht(fc->header + kEncHeaderDhtAt, 0, s_bits[0], s_vals[0], n_dc);
        opt_write_dht(fc->header + kEncHeaderDhtAt + dc_len, 1, s_bits[1], s_vals[1], n_ac);
        fc->header_bytes = (uint32_t)(sos + kEncSosBytes);
    }
    if (huff && (tid == 0 || tid == 32)) {        // the decoder's tables for degradeJPEG: DC at 2 f, AC at 2 f + 1
        const int c = tid >> 5;
        uint8_t b17[17];
        b17[0] = 0;
        for (int l = 0; l < 16; l++) b17[l + 1] = s_bits[c][l];
        derive_table(b17, s_vals[c], s_n[c], huff + 2 * (size_t)f + c);
    }
}

constexpr int kET = 1024;                   // lanes of the per-frame entropy CTA

// kOpt: the tables and the header are the frame's own (code[f]) and the AC bits are recounted with them.
template <bool kOpt>
__global__ void __launch_bounds__(kET, 1) jpeg_enc_entropy_kernel(const int16_t* __restrict__ coefs, const EncBlock* __restrict__ info, const EncTables* __restrict__ tabs,
                                                                  const EncFrameCode* __restrict__ code, uint32_t* words_base, uint8_t* __restrict__ slots,
                                                                  uint32_t* __restrict__ lens, FrameDesc* __restrict__ desc, int nb, size_t word_bytes, size_t slot_bytes) {
    __shared__ uint32_t s_dc[16], s_ac[256], warp_tot[32];
    __shared__ uint8_t s_hdr[kEncHeaderBytes];
    const int f = blockIdx.x, tid = threadIdx.x;
    const uint32_t* g_dc = kOpt ? code[f].dc : tabs->dc;
    const uint32_t* g_ac = kOpt ? code[f].ac : tabs->ac;
    const uint8_t* g_hdr = kOpt ? code[f].header : tabs->header;
    const uint32_t hdr_bytes = kOpt ? code[f].header_bytes : (uint32_t)kEncHeaderBytes;
    for (int i = tid; i < 256; i += kET) s_ac[i] = g_ac[i];
    if (tid < 16) s_dc[tid] = g_dc[tid];
    for (int i = tid; i < (int)hdr_bytes; i += kET) s_hdr[i] = g_hdr[i];
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
        for (int b = b0; b < b1; b++) {
            const int dc = inf[b].dc;
            if (kOpt) {
                const int16_t* zz = cf + (size_t)b * 64;
                bits += block_ac_bits_sparse(inf[b].nz, [zz](int k) { return (int)zz[k]; }, s_ac);
            } else {
                bits += inf[b].ac_bits;
            }
            bits += block_dc_bits(dc - prev, s_dc); prev = dc;
        }
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
        if (i0 < L) stuff_write(wv, L, i0, out + hdr_bytes + i0 + stuffed + o);
        stuffed += tile_ff;
    }
    const uint32_t len = hdr_bytes + L + stuffed + 2u;
    for (int i = tid; i < (int)hdr_bytes; i += kET) out[i] = s_hdr[i];
    if (tid == 0) {
        out[len - 2] = 0xFF; out[len - 1] = 0xD9;
        lens[f] = len;
        if (desc) {
            FrameDesc d;
            d.scan_offset = (uint64_t)f * slot_bytes + hdr_bytes;
            d.scan_end = (uint64_t)f * slot_bytes + len;
            d.restart_interval = 0; d.qt = 0; d.dc = kOpt ? 2 * f : 0; d.ac = kOpt ? 2 * f + 1 : 1;
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
                       int n, int H, int W, cudaStream_t s, void* opt, void* huff) {
    const JpegEncLayout l = jpeg_enc_layout(H, W, opt != nullptr);
    const int bw = (W + 7) / 8, nb = (int)l.blocks;
    const uint32_t total = (uint32_t)((size_t)n * nb);
    if (!opt) {
        jpeg_enc_transform_kernel<false><<<(total + 127) / 128, 128, 0, s>>>(src, (const EncTables*)tabs, (int16_t*)coefs, (EncBlock*)info, nullptr, H, W, bw, nb, total);
        jpeg_enc_entropy_kernel<false><<<n, kET, 0, s>>>((const int16_t*)coefs, (const EncBlock*)info, (const EncTables*)tabs, nullptr, (uint32_t*)words, slots, lens,
                                                         (FrameDesc*)desc, nb, l.word_bytes, l.slot_bytes);
        return 2;
    }
    // opt: [n x 256 AC symbol counts][n x EncFrameCode], 16-byte aligned
    uint32_t* hist = (uint32_t*)opt;
    EncFrameCode* code = (EncFrameCode*)((char*)opt + (((size_t)n * 256 * sizeof(uint32_t) + 15) & ~(size_t)15));
    cudaMemsetAsync(hist, 0, (size_t)n * 256 * sizeof(uint32_t), s);
    jpeg_enc_transform_kernel<true><<<(total + 127) / 128, 128, 0, s>>>(src, (const EncTables*)tabs, (int16_t*)coefs, (EncBlock*)info, hist, H, W, bw, nb, total);
    jpeg_enc_table_kernel<<<n, kTT, 0, s>>>((const EncBlock*)info, (const EncTables*)tabs, hist, code, (HuffTable*)huff, nb);
    jpeg_enc_entropy_kernel<true><<<n, kET, 0, s>>>((const int16_t*)coefs, (const EncBlock*)info, (const EncTables*)tabs, code, (uint32_t*)words, slots, lens,
                                                    (FrameDesc*)desc, nb, l.word_bytes, l.slot_bytes);
    return 3;
}

int launch_jpeg_enc_gather(const uint8_t* slots, size_t slot_bytes, const uint32_t* lens, const uint64_t* offs, uint8_t* dst, int n, uint64_t max_len, cudaStream_t s) {
    const uint32_t gx = (uint32_t)((max_len + 256 * 16 - 1) / (256 * 16));
    jpeg_enc_gather_kernel<<<dim3(gx ? gx : 1, n), 256, 0, s>>>(slots, slot_bytes, lens, offs, dst);
    return 1;
}

}  // namespace dmc
