// dmc_metrics.cu -- distortion of 8-bit frame batches: the exact per-frame sum of squared differences (SSE) that PSNR
// (dmc_psnr_from_sse, the formula of cv::PSNR) is computed from, and the structural similarity (SSIM, below).
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

// ---- SSIM (Wang, Bovik, Sheikh, Simoncelli 2004, ssim_index.m) -------------------------------------------------------------
// 11-tap Gaussian window, sigma = 1.5, only the (rows - 10) x (cols - 10) window positions that lie inside the frame;
// interleaved channels are scored apart and their MSSIMs averaged (the definition of include/dmc_c.h, dmc_ssim_batch).
//
// Grid: x, y = tile of kSsimTW x kSsimTH window positions, z = frame.  A CTA stages its tile and the 10-pixel halo of a and b as
// bytes (all channels: interleaved rows are read coalesced once), then per channel: the horizontal pass writes the five moments
// x, y, x^2, y^2, xy of every staged row to FP64 shared memory -- taps paired on integers, g_i (v[-i] + v[i]), exact before the
// multiply --, the vertical pass forms mu, sigma and S at every window position, and a fixed-order CTA reduction writes the
// tile's sum of S to partial[(frame * channels + c) * tiles + tile].  ssim_finish_kernel adds a frame's partials in a fixed
// order (fixed block size, fixed tree) and averages the channels.  No floating-point atomics anywhere: a frame's MSSIM is the
// same bits in any batch, group or launch.  FP64 throughout: in FP32, E[x^2] - mu^2 loses about 4e-3 on sigma^2 near 255.
namespace {

constexpr int kSsimTW = 32, kSsimTH = 16, kSsimThreads = 256, kSsimR = 5;
constexpr int kSsimSW = kSsimTW + 2 * kSsimR, kSsimSH = kSsimTH + 2 * kSsimR;    // staged pixels per channel
constexpr int kFinishThreads = 256;

// g_i = exp(-i^2 / 4.5) / (sum over j = -5..5 of exp(-j^2 / 4.5)) in double, i = 0..5 (g_{-i} = g_i); 17 significant digits
// give back the same doubles
__constant__ double c_ssim_g[kSsimR + 1] = {0.26601172486179436, 0.2130055377112537, 0.10936068950970002, 0.03600077212843083,
                                            0.007598758135239185, 0.00102838008447911};

__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += red[w];
    __syncthreads();
    return t;     // valid in thread 0
}

template <int CN>
__global__ void __launch_bounds__(kSsimThreads) ssim_u8_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, double* __restrict__ partial,
                                                              int rows, int cols) {
    __shared__ uint8_t sa[kSsimSH][kSsimSW * CN], sb[kSsimSH][kSsimSW * CN];
    __shared__ double mom[5][kSsimSH][kSsimTW];
    __shared__ double red[kSsimThreads / 32];
    const size_t frame_bytes = (size_t)rows * cols * CN;
    const uint8_t* pa = a + blockIdx.z * frame_bytes;
    const uint8_t* pb = b + blockIdx.z * frame_bytes;
    const int x0 = blockIdx.x * kSsimTW, y0 = blockIdx.y * kSsimTH;     // first window position (its top-left pixel)
    const int vw = cols - 2 * kSsimR, vh = rows - 2 * kSsimR;            // valid window positions
    const int sw = min(kSsimSW, cols - x0) * CN, sh = min(kSsimSH, rows - y0);
    for (int i = threadIdx.x; i < kSsimSH * kSsimSW * CN; i += kSsimThreads) {
        const int r = i / (kSsimSW * CN), c = i - r * (kSsimSW * CN);
        const bool in = r < sh && c < sw;
        const size_t o = (size_t)(y0 + r) * cols * CN + (size_t)x0 * CN + c;
        sa[r][c] = in ? pa[o] : 0;
        sb[r][c] = in ? pb[o] : 0;
    }
    __syncthreads();
    const double C1 = (0.01 * 255) * (0.01 * 255), C2 = (0.03 * 255) * (0.03 * 255);
    double g[kSsimR + 1];
#pragma unroll
    for (int i = 0; i <= kSsimR; i++) g[i] = c_ssim_g[i];
    const int tile = blockIdx.y * gridDim.x + blockIdx.x, tiles = gridDim.x * gridDim.y;
    for (int ch = 0; ch < CN; ch++) {
        for (int i = threadIdx.x; i < kSsimSH * kSsimTW; i += kSsimThreads) {
            const int r = i / kSsimTW, x = i - r * kSsimTW, cc = (x + kSsimR) * CN + ch;
            const int xa = sa[r][cc], xb = sb[r][cc];
            double m0 = g[0] * xa, m1 = g[0] * xb, m2 = g[0] * (xa * xa), m3 = g[0] * (xb * xb), m4 = g[0] * (xa * xb);
#pragma unroll
            for (int k = 1; k <= kSsimR; k++) {
                const int la = sa[r][cc - k * CN], ra = sa[r][cc + k * CN], lb = sb[r][cc - k * CN], rb = sb[r][cc + k * CN];
                m0 = fma(g[k], (double)(la + ra), m0);
                m1 = fma(g[k], (double)(lb + rb), m1);
                m2 = fma(g[k], (double)(la * la + ra * ra), m2);
                m3 = fma(g[k], (double)(lb * lb + rb * rb), m3);
                m4 = fma(g[k], (double)(la * lb + ra * rb), m4);
            }
            mom[0][r][x] = m0; mom[1][r][x] = m1; mom[2][r][x] = m2; mom[3][r][x] = m3; mom[4][r][x] = m4;
        }
        __syncthreads();
        double acc = 0.0;
        for (int i = threadIdx.x; i < kSsimTH * kSsimTW; i += kSsimThreads) {
            const int r = i / kSsimTW, x = i - r * kSsimTW;
            if (y0 + r >= vh || x0 + x >= vw) continue;
            double v[5];
#pragma unroll
            for (int m = 0; m < 5; m++) {
                double s = g[0] * mom[m][r + kSsimR][x];
#pragma unroll
                for (int k = 1; k <= kSsimR; k++) s = fma(g[k], mom[m][r + kSsimR - k][x] + mom[m][r + kSsimR + k][x], s);
                v[m] = s;
            }
            const double mx = v[0], my = v[1], mxy = mx * my, mxx = mx * mx, myy = my * my;
            const double sxx = v[2] - mxx, syy = v[3] - myy, sxy = v[4] - mxy;
            acc += ((2.0 * mxy + C1) * (2.0 * sxy + C2)) / ((mxx + myy + C1) * (sxx + syy + C2));
        }
        const double t = block_sum(acc, red);      // (its __syncthreads also ends the reads of mom before the next channel)
        if (threadIdx.x == 0) partial[((size_t)blockIdx.z * CN + ch) * tiles + tile] = t;
    }
}

// mssim[f] = mean over the channels of (sum of the channel's tile partials) / positions
__global__ void __launch_bounds__(kFinishThreads) ssim_finish_kernel(const double* __restrict__ partial, double* __restrict__ mssim, int tiles, int cn, double positions) {
    __shared__ double red[kFinishThreads / 32];
    const double* p = partial + (size_t)blockIdx.x * cn * tiles;
    double mean = 0.0;
    for (int ch = 0; ch < cn; ch++) {
        double s = 0.0;
        for (int i = threadIdx.x; i < tiles; i += kFinishThreads) s += p[(size_t)ch * tiles + i];
        const double t = block_sum(s, red);
        mean += t / positions;
    }
    if (threadIdx.x == 0) mssim[blockIdx.x] = cn == 1 ? mean : mean / cn;
}

int ssim_tiles(int rows, int cols) {
    return ((cols - 2 * kSsimR + kSsimTW - 1) / kSsimTW) * ((rows - 2 * kSsimR + kSsimTH - 1) / kSsimTH);
}

}  // namespace

size_t ssim_partial_bytes(int rows, int cols, int channels) { return (size_t)ssim_tiles(rows, cols) * channels * sizeof(double); }

int launch_ssim_u8(const uint8_t* a, const uint8_t* b, double* partial, double* mssim, int n, int rows, int cols, int channels, cudaStream_t s) {
    if (n <= 0) return 0;
    const dim3 grid((cols - 2 * kSsimR + kSsimTW - 1) / kSsimTW, (rows - 2 * kSsimR + kSsimTH - 1) / kSsimTH);
    const int tiles = ssim_tiles(rows, cols);
    const size_t fb = (size_t)rows * cols * channels;
    const double positions = (double)(rows - 2 * kSsimR) * (double)(cols - 2 * kSsimR);
    int nk = 0;
    for (int f0 = 0; f0 < n; f0 += 65535) {                 // (grid z limit)
        const int nf = n - f0 < 65535 ? n - f0 : 65535;
        const dim3 g3(grid.x, grid.y, nf);
        double* part = partial + (size_t)f0 * channels * tiles;
        if (channels == 3) ssim_u8_kernel<3><<<g3, kSsimThreads, 0, s>>>(a + fb * f0, b + fb * f0, part, rows, cols);
        else ssim_u8_kernel<1><<<g3, kSsimThreads, 0, s>>>(a + fb * f0, b + fb * f0, part, rows, cols);
        nk++;
    }
    ssim_finish_kernel<<<n, kFinishThreads, 0, s>>>(partial, mssim, tiles, channels, positions);
    return nk + 1;
}

}  // namespace dmc
