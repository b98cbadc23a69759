// dmc_common.cuh -- device-side helpers shared by the sm_100a kernels of libdmc_b200.
//
// Parity rules (SURVEY.md 8a "parity hazards"): this library is compiled with -fmad=false and never with
// --use_fast_math, so every float expression below is a sequence of individually rounded IEEE-754 RN
// operations in source order, exactly like the reference's SSE code built with strict FP.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <float.h>
#include <limits.h>

namespace dmc {

// Entry points that visit several devices leave the calling thread's current device as they found it (the caller may
// be a framework with its own idea of the current device).
struct DeviceGuard {
    int dev = -1;
    DeviceGuard() { if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = -1; } }
    ~DeviceGuard() { if (dev >= 0) cudaSetDevice(dev); }
};

__host__ __device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// cv::borderInterpolate(p, len, BORDER_REFLECT_101)
__host__ __device__ __forceinline__ int reflect101(int p, int len) {
    if ((unsigned)p < (unsigned)len) return p;
    if (len == 1) return 0;
    do { p = p < 0 ? -p : 2 * len - 2 - p; } while ((unsigned)p >= (unsigned)len);
    return p;
}

// cvRound / _mm_cvtps_epi32: round-half-even; NaN or |v| >= 2^31 -> 0x80000000 ("integer indefinite").
__device__ __forceinline__ int cvround(float v) {
    if (!(v >= -2147483648.f && v < 2147483648.f)) return INT_MIN;
    return __float2int_rn(v);
}
__device__ __forceinline__ uint8_t sat_u8(int v) { return (uint8_t)min(max(v, 0), 255); }
__device__ __forceinline__ uint16_t sat_u16(int v) { return (uint16_t)min(max(v, 0), 65535); }
__device__ __forceinline__ int sat_s16(int v) { return min(max(v, -32768), 32767); }

// Circle test of the range filters: tap (i, j) is kept iff sqrt(i*i + j*j) <= rmax, evaluated in double by the
// reference (binalyWeightedRangeFilter.cpp:1070-1072).  For integers that is i*i + j*j <= rmax*rmax.
__host__ __device__ __forceinline__ int circle_halfwidth(int i, int rmax, int rH) {
    int lim = rmax * rmax - i * i, j = 0;
    if (lim < 0) return -1;
    while ((j + 1) * (j + 1) <= lim) j++;
    return j < rH ? j : rH;
}

// Exclusive prefix sum over a CTA of NT threads (all of them call it); *total = sum of all.
template <int NT>
__device__ __forceinline__ uint32_t cta_scan_excl(uint32_t v, uint32_t* warp_tot, uint32_t* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    __syncthreads();                        // warp_tot may still be read by the previous scan
    if (lane == 31) warp_tot[w] = x;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < NT / 32; i++) { const uint32_t t = warp_tot[i]; if (i < w) base += t; tot += t; }
    *total = tot;
    return base + x - v;
}

}  // namespace dmc
