// dmc_stage.cuh -- shared-memory tile staging common to the packed 8-bit kernels (dmc_front8u.cu, dmc_bwrf8u_h2.cu):
// a 128-pixel-wide output tile with a 16-pixel halo on either side, so that every 16-byte load of an interior row
// segment is aligned.
#pragma once
#include "dmc_common.cuh"

namespace dmc {

constexpr int kTW = 128;     // output tile width  (2 warps x 32 lanes x 2 px, or 32 lanes x 4 px)

// Stages rows [ytop, ytop + SH) x columns [X0 - 16, X0 + 128 + 16) of one frame, 16 pixels per thread and step: one 16-byte
// load where the segment lies inside the image and is aligned (`al`: W % 16 == 0 and a 16-byte aligned base), else bytes
// gathered through the border rule.  REFLECT selects BORDER_REFLECT_101 (Gaussian) instead of BORDER_REPLICATE.
//   MODE 0: raw bytes, SW/4 words per row            MODE 1: 0x6400 | byte (fp16 1024 + byte), SW/2 words per row
//   MODE 2: plain fp16 0..255, SW/2 words per row
// SWW_ > 0 pads the row stride to SWW_ words (a multiple of 4).
constexpr int kHalo16 = 16, kSW16 = kTW + 2 * kHalo16, kNV16 = kSW16 / 16;
template <int SH, int MODE, bool REFLECT, int SWW_ = 0>
__device__ __forceinline__ void stage_tile16(uint32_t* __restrict__ sm, const uint8_t* __restrict__ fsrc, int X0, int ytop, int H, int W, bool al, int tid) {
    constexpr int SWW = SWW_ > 0 ? SWW_ : (MODE == 0 ? kSW16 / 4 : kSW16 / 2);
    static_assert(SWW % 4 == 0 && SWW >= (MODE == 0 ? kSW16 / 4 : kSW16 / 2), "16-byte aligned rows");
    for (int idx = tid; idx < SH * kNV16; idx += 256) {
        const int ty = idx / kNV16, tq = idx - ty * kNV16, gx = X0 - kHalo16 + 16 * tq;
        const int gy = REFLECT ? reflect101(ytop + ty, H) : clampi(ytop + ty, 0, H - 1);
        const uint8_t* row = fsrc + (size_t)gy * W;
        uint32_t w[4];
        if (al && gx >= 0 && gx + 15 < W) { const uint4 q = *reinterpret_cast<const uint4*>(row + gx); w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w; }
        else {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                uint32_t v = 0;
#pragma unroll
                for (int b = 0; b < 4; b++) { const int xx = gx + 4 * k + b; v |= (uint32_t)row[REFLECT ? reflect101(xx, W) : clampi(xx, 0, W - 1)] << (8 * b); }
                w[k] = v;
            }
        }
        if constexpr (MODE == 0) *reinterpret_cast<uint4*>(&sm[ty * SWW + 4 * tq]) = make_uint4(w[0], w[1], w[2], w[3]);
        else {
            uint32_t o[8];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                uint32_t a = __byte_perm(w[k], 0x64646464u, 0x4140), b = __byte_perm(w[k], 0x64646464u, 0x4342);
                if (MODE == 2) {
                    const __half2 k1024 = __float2half2_rn(1024.f);
                    __half2 h0 = __hsub2(*reinterpret_cast<__half2*>(&a), k1024), h1 = __hsub2(*reinterpret_cast<__half2*>(&b), k1024);
                    a = *reinterpret_cast<uint32_t*>(&h0); b = *reinterpret_cast<uint32_t*>(&h1);
                }
                o[2 * k] = a; o[2 * k + 1] = b;
            }
            uint4* d = reinterpret_cast<uint4*>(&sm[ty * SWW + 8 * tq]);
            d[0] = make_uint4(o[0], o[1], o[2], o[3]); d[1] = make_uint4(o[4], o[5], o[6], o[7]);
        }
    }
}
__device__ __forceinline__ bool aligned16(const uint8_t* src, int W) { return (W & 15) == 0 && (reinterpret_cast<size_t>(src) & 15) == 0; }

}  // namespace dmc
