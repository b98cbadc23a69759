// dmc_metrics.cu -- distortion of 8-bit frame batches: the exact per-frame sum of squared differences (SSE) that PSNR
// (dmc_psnr_from_sse, the formula of cv::PSNR) is computed from.
//
// Grid: x = chunk of kCtaVecs 16-byte words of a frame, y = frame.  Every thread loads kVecPerThread words of the
// reference and of each compared frame before it computes, so that a warp has all its loads in flight at once; per 4
// bytes d = |a - b| (__vabsdiffu4) and acc += d . d (__dp4a).  One launch compares the reference batch `a` with one or
// with two batches (b0 -> sse0, b1 -> sse1), so that a rate-distortion sweep reads the source once for the coded and the
// filtered frames.  Integer sums: the result is exact and does not depend on the order of the additions.
#include "dmc_kernels.cuh"

namespace dmc {
namespace {

constexpr int kThreads = 256;
constexpr int kVecPerThread = 4;
constexpr size_t kCtaVecs = (size_t)kThreads * kVecPerThread;    // 16 KB of every frame per CTA
constexpr size_t kCtaBytes = kCtaVecs * 16;
// A thread's 32-bit accumulator takes at most kVecPerThread * 4 words of 4 * 255^2 each, plus one edge byte (< one word):
// the work per thread is bounded by the tiling, no fold into 64 bits is needed before the warp reduction.
static_assert(kVecPerThread * 4 + 1 <= 16512, "per-thread 32-bit accumulator could overflow: floor((2^32 - 1) / (4 * 255^2)) = 16512 words");

__device__ __forceinline__ uint32_t sq_words(uint4 a, uint4 b, uint32_t acc) {
    uint32_t d;
    d = __vabsdiffu4(a.x, b.x); acc = __dp4a(d, d, acc);
    d = __vabsdiffu4(a.y, b.y); acc = __dp4a(d, d, acc);
    d = __vabsdiffu4(a.z, b.z); acc = __dp4a(d, d, acc);
    d = __vabsdiffu4(a.w, b.w); acc = __dp4a(d, d, acc);
    return acc;
}

__device__ __forceinline__ uint32_t sq_byte(uint8_t a, uint8_t b) { const int d = (int)a - (int)b; return (uint32_t)(d * d); }

__device__ __forceinline__ void warp_add(uint32_t acc, unsigned long long* slot) {
    unsigned long long v = acc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(slot, v);
}

// vec: a, b0 (and b1) have the same address modulo 16, so every frame splits into the same unaligned head (< 16 bytes,
// up to the first 16-byte boundary of the frame), aligned 16-byte words and an unaligned tail (< 16 bytes).  The head
// and tail bytes go to the first warp of chunk 0 (lanes 0..15 head, 16..31 tail).  Otherwise the frames are read byte by
// byte, kCtaBytes per CTA.
template <bool kTwo>
__global__ void __launch_bounds__(kThreads) sse_u8_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b0, const uint8_t* __restrict__ b1,
                                                          unsigned long long* __restrict__ sse0, unsigned long long* __restrict__ sse1, size_t frame_bytes, bool vec) {
    const size_t f = blockIdx.y, base = f * frame_bytes;
    const uint8_t* pa = a + base;
    const uint8_t* p0 = b0 + base;
    const uint8_t* p1 = kTwo ? b1 + base : nullptr;
    uint32_t acc0 = 0, acc1 = 0;
    if (vec) {
        const size_t head = min((size_t)((16u - ((uintptr_t)pa & 15u)) & 15u), frame_bytes);
        const size_t nvec = (frame_bytes - head) >> 4, tail = head + nvec * 16;
        const uint4* va = (const uint4*)(pa + head);
        const uint4* v0 = (const uint4*)(p0 + head);
        const uint4* v1 = kTwo ? (const uint4*)(p1 + head) : nullptr;
        const size_t i0 = blockIdx.x * kCtaVecs + threadIdx.x;
        uint4 ra[kVecPerThread], r0[kVecPerThread], r1[kVecPerThread];
        if (i0 + (size_t)(kVecPerThread - 1) * kThreads < nvec) {          // all words in the frame: unpredicated loads
#pragma unroll
            for (int k = 0; k < kVecPerThread; k++) {
                ra[k] = __ldg(va + i0 + k * kThreads); r0[k] = __ldg(v0 + i0 + k * kThreads);
                if (kTwo) r1[k] = __ldg(v1 + i0 + k * kThreads);
            }
        } else {
            const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int k = 0; k < kVecPerThread; k++) {
                const size_t i = i0 + (size_t)k * kThreads;
                const bool in = i < nvec;
                ra[k] = in ? __ldg(va + i) : z; r0[k] = in ? __ldg(v0 + i) : z;
                if (kTwo) r1[k] = in ? __ldg(v1 + i) : z;
            }
        }
#pragma unroll
        for (int k = 0; k < kVecPerThread; k++) {
            acc0 = sq_words(ra[k], r0[k], acc0);
            if (kTwo) acc1 = sq_words(ra[k], r1[k], acc1);
        }
        if (blockIdx.x == 0 && threadIdx.x < 32) {
            const size_t j = threadIdx.x < 16 ? threadIdx.x : tail + threadIdx.x - 16;
            if (threadIdx.x < 16 ? j < head : j < frame_bytes) {
                acc0 += sq_byte(pa[j], p0[j]);
                if (kTwo) acc1 += sq_byte(pa[j], p1[j]);
            }
        }
    } else {
        const size_t i0 = blockIdx.x * kCtaBytes + threadIdx.x;
        for (int k = 0; k < (int)(kCtaBytes / kThreads); k++) {
            const size_t i = i0 + (size_t)k * kThreads;
            if (i < frame_bytes) {
                const uint8_t x = pa[i];
                acc0 += sq_byte(x, p0[i]);
                if (kTwo) acc1 += sq_byte(x, p1[i]);
            }
        }
    }
    warp_add(acc0, sse0 + f);
    if (kTwo) warp_add(acc1, sse1 + f);
}

}  // namespace

int launch_sse_u8(const uint8_t* a, const uint8_t* b0, const uint8_t* b1, uint64_t* sse0, uint64_t* sse1, int n, size_t frame_bytes, cudaStream_t s) {
    if (n <= 0 || frame_bytes == 0) return 0;
    cudaMemsetAsync(sse0, 0, (size_t)n * sizeof(uint64_t), s);
    if (b1) cudaMemsetAsync(sse1, 0, (size_t)n * sizeof(uint64_t), s);
    const uintptr_t m = (uintptr_t)a & 15;
    const bool vec = ((uintptr_t)b0 & 15) == m && (!b1 || ((uintptr_t)b1 & 15) == m);
    const unsigned chunks = (unsigned)((frame_bytes + kCtaBytes - 1) / kCtaBytes);
    int nk = 0;
    for (int f0 = 0; f0 < n; f0 += 65535, nk++) {           // (grid y limit)
        const int nf = n - f0 < 65535 ? n - f0 : 65535;
        const size_t o = (size_t)f0 * frame_bytes;
        if (b1) sse_u8_kernel<true><<<dim3(chunks, nf), kThreads, 0, s>>>(a + o, b0 + o, b1 + o, (unsigned long long*)sse0 + f0, (unsigned long long*)sse1 + f0, frame_bytes, vec);
        else sse_u8_kernel<false><<<dim3(chunks, nf), kThreads, 0, s>>>(a + o, b0 + o, nullptr, (unsigned long long*)sse0 + f0, nullptr, frame_bytes, vec);
    }
    return nk;
}

}  // namespace dmc
