// dmc_kernels_8u.cu -- the integer half of the post filter set on sm_100a:
//   median (cv::medianBlur), small Gaussian (8U through exact FP32), min-max "blur remove", and the 8-bit
//   binary-weighted range filter.  One CTA = one 2-D output tile of one frame; the input tile plus the halo the
//   stage's radius needs is staged in shared memory with the stage's own border rule applied at the IMAGE edge.
#include "dmc_common.cuh"
#include "dmc_kernels.cuh"
#include <math.h>
#include <string.h>

namespace dmc {

// ----------------------------------------------------------------------------------------------------------
// host helpers
// ----------------------------------------------------------------------------------------------------------
RowSpan make_rowspan(int kw, int kh) {
    RowSpan rs; memset(&rs, 0, sizeof rs);
    rs.rH = kw >> 1; rs.rV = kh >> 1;                              // binalyWeightedRangeFilter.cpp:1041-1042
    int rmax = rs.rV > rs.rH ? rs.rV : rs.rH;
    for (int i = -rs.rV; i <= rs.rV; i++) {
        int hw = circle_halfwidth(i, rmax, rs.rH);
        rs.hw[i + rs.rV] = (signed char)hw;
        if (hw >= 0) rs.ntaps += 2 * hw + 1;
    }
    return rs;
}

static const float kSmallGaussianTab[5][9] = {      /* cv::getGaussianKernel: fixed taps for odd n <= 9 when sigma <= 0 (OpenCV 4.13 small_gaussian_tab) */
    {1.f}, {0.25f, 0.5f, 0.25f}, {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f},
    {0.03125f, 0.109375f, 0.21875f, 0.28125f, 0.21875f, 0.109375f, 0.03125f},
    {0.015625f, 0.05078125f, 0.1171875f, 0.19921875f, 0.234375f, 0.19921875f, 0.1171875f, 0.05078125f, 0.015625f}};

bool make_gauss_taps(int d, double sigma, int rows, int cols, GaussTaps* t) {
    // cv::GaussianBlur: a 1-pixel-high (wide) image drops the vertical (horizontal) kernel
    int kw = cols == 1 ? 1 : d, kh = rows == 1 ? 1 : d;
    if (kw > kMaxTapsRow || kh > kMaxTapsRow || d < 1 || (d & 1) == 0) return false;
    for (int pass = 0; pass < 2; pass++) {
        int n = pass ? kh : kw; float* k = pass ? t->ky : t->kx;
        (pass ? t->ry : t->rx) = n / 2;
        if (sigma <= 0 && (n & 1) && n <= 9) { for (int i = 0; i < n; i++) k[i] = kSmallGaussianTab[n >> 1][i]; continue; }   // dyadic taps, sum exactly 1
        double tmp[kMaxTapsRow], sum = 0, sx = sigma > 0 ? sigma : ((n - 1) * 0.5 - 1) * 0.3 + 0.8, s2 = -0.5 / (sx * sx);
        for (int i = 0; i < n; i++) { double x = i - (n - 1) * 0.5; tmp[i] = exp(s2 * x * x); sum += tmp[i]; }
        sum = 1. / sum;
        for (int i = 0; i < n; i++) k[i] = (float)(tmp[i] * sum);
    }
    return true;
}

// ----------------------------------------------------------------------------------------------------------
// tile staging
// ----------------------------------------------------------------------------------------------------------
enum { B_REPLICATE = 0, B_REFLECT101 = 1 };

// Copies the (tw x th) window whose top-left image coordinate is (x0, y0) into shared memory, mapping
// out-of-image coordinates with the border rule.  Interior tiles take the unclamped path.
template <typename T, int BORDER>
__device__ __forceinline__ void stage_tile(T* sm, int tw, int th, const T* __restrict__ src, int H, int W, int x0, int y0) {
    const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
    for (int idx = tid; idx < tw * th; idx += nt) {
        int ty = idx / tw, tx = idx - ty * tw;
        int gx = x0 + tx, gy = y0 + ty;
        if (BORDER == B_REPLICATE) { gx = clampi(gx, 0, W - 1); gy = clampi(gy, 0, H - 1); }
        else { gx = reflect101(gx, W); gy = reflect101(gy, H); }
        sm[idx] = src[(size_t)gy * W + gx];
    }
}

// ----------------------------------------------------------------------------------------------------------
// median: every supported radius (1..10) runs in dmc_front8u.cu (shared-sort circuits for 3x3 / 5x5, packed bisection
// for 7x7 .. 21x21)
// ----------------------------------------------------------------------------------------------------------
constexpr int kTX = 32, kTY = 16;   // output tile of the generic stage kernels (256 threads, 2 rows each)

int launch_median8u(const uint8_t* src, uint8_t* dst, int n, int H, int W, int r, cudaStream_t s) {
    return launch_median8u_fast(src, dst, n, H, W, r, s);       // 0 for a radius outside 1..10 (the C ABI rejects those before)
}

// ----------------------------------------------------------------------------------------------------------
// small Gaussian: u8 -> f32 -> separable blur (rows, then columns) -> RNE + saturate u8
//   d <= 5 : x0*k0 + sum_i (x[-i] + x[+i]) * k_i   on both passes
//   d >= 7 : the row pass is a left-to-right running sum, the column pass stays symmetric
// ----------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gauss8u_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int H, int W, GaussTaps t) {
    extern __shared__ unsigned char smraw[];
    const int rx = t.rx, ry = t.ry, TW = kTX + 2 * rx, TH = kTY + 2 * ry;
    uint8_t* sin = smraw;                                        // TH x TW input tile
    float* srow = (float*)(smraw + ((TW * TH + 15) & ~15));      // TH x kTX row-pass results
    const size_t fo = (size_t)blockIdx.z * H * W;
    const int x0 = blockIdx.x * kTX, y0 = blockIdx.y * kTY;
    stage_tile<uint8_t, B_REFLECT101>(sin, TW, TH, src + fo, H, W, x0 - rx, y0 - ry);
    __syncthreads();
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    for (int idx = tid; idx < TH * kTX; idx += 256) {
        int ty = idx / kTX, tx = idx - ty * kTX;
        const uint8_t* p = sin + ty * TW + tx + rx;
        float acc;
        if (2 * rx + 1 <= 5) {
            acc = (float)p[0] * t.kx[rx];
            for (int i = 1; i <= rx; i++) acc = acc + ((float)p[-i] + (float)p[i]) * t.kx[rx + i];
        } else {
            acc = t.kx[0] * (float)p[-rx];
            for (int i = 1; i <= 2 * rx; i++) acc = acc + t.kx[i] * (float)p[i - rx];
        }
        srow[idx] = acc;
    }
    __syncthreads();
    for (int ly = threadIdx.y; ly < kTY; ly += blockDim.y) {
        int x = x0 + threadIdx.x, y = y0 + ly;
        if (x >= W || y >= H) continue;
        const float* p = srow + (ly + ry) * kTX + threadIdx.x;
        float acc = p[0] * t.ky[ry];
        for (int i = 1; i <= ry; i++) acc = acc + (p[-i * kTX] + p[i * kTX]) * t.ky[ry + i];
        dst[fo + (size_t)y * W + x] = sat_u8(cvround(acc));
    }
}

int launch_gauss8u(const uint8_t* src, uint8_t* dst, int n, int H, int W, const GaussTaps& t, cudaStream_t s) {
    if (int nk = launch_gauss8u_fast(src, dst, n, H, W, t, s)) return nk;
    dim3 grid((W + kTX - 1) / kTX, (H + kTY - 1) / kTY, n), block(32, 8);
    int TW = kTX + 2 * t.rx, TH = kTY + 2 * t.ry;
    size_t smem = ((TW * TH + 15) & ~15) + (size_t)TH * kTX * sizeof(float);
    gauss8u_kernel<<<grid, block, smem, s>>>(src, dst, H, W, t);
    return 1;
}

// ----------------------------------------------------------------------------------------------------------
// min-max: dilate / erode over (2r+1)^2 with out-of-image taps ignored (== clamped coordinates), then the
// "blur remove" select  out = (|src-mn| == min(|src-mn|, |src-mx|)) ? mn : mx   (minmaxFilter.cpp:63-65, :83-89)
// ----------------------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ T absdiff_cv(T a, T b) { return a > b ? (T)(a - b) : (T)(b - a); }
template <> __device__ __forceinline__ int16_t absdiff_cv<int16_t>(int16_t a, int16_t b) { int d = (int)a - (int)b; d = d < 0 ? -d : d; return (int16_t)min(d, 32767); }
template <> __device__ __forceinline__ float absdiff_cv<float>(float a, float b) { return fabsf(a - b); }
template <> __device__ __forceinline__ double absdiff_cv<double>(double a, double b) { return fabs(a - b); }

// MODE 0: blur-remove select; 1: max only; 2: min only.  The channel is blockIdx.z % cn (planes are filtered
// independently, minmaxFilter.cpp:189-213).
// Visiting order (cv::dilate / cv::erode as the reference build's cv:: stand-in states them, DESIGN.md §2): each pass
// starts at the window's centre and then folds every tap in order (left to right, top to bottom) with m = v > m ? v : m.
// For ordered values the order is free, but a NaN sticks only where the fold starts and of +0 / -0 the first one seen
// wins, so float results follow the reference only in this order.  Clamped border taps repeat a neighbour and change
// nothing.
template <typename T, int MODE>
__global__ void __launch_bounds__(256) minmax_kernel(const T* __restrict__ src, T* __restrict__ dst, int H, int W, int cn, int rx, int ry) {
    extern __shared__ unsigned char smraw[];
    const int TW = kTX + 2 * rx, TH = kTY + 2 * ry;
    T* sin = (T*)smraw;                       // TH x TW
    T* smx = sin + TW * TH;                   // TH x kTX row maxima
    T* smn = smx + TH * kTX;                  // TH x kTX row minima
    const int frame = blockIdx.z / cn, c = blockIdx.z - frame * cn;
    const T* fsrc = src + (size_t)frame * H * W * cn; T* fdst = dst + (size_t)frame * H * W * cn;
    const int x0 = blockIdx.x * kTX, y0 = blockIdx.y * kTY;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    for (int idx = tid; idx < TW * TH; idx += 256) {
        int ty = idx / TW, tx = idx - ty * TW;
        int gx = clampi(x0 - rx + tx, 0, W - 1), gy = clampi(y0 - ry + ty, 0, H - 1);
        sin[idx] = fsrc[((size_t)gy * W + gx) * cn + c];
    }
    __syncthreads();
    for (int idx = tid; idx < TH * kTX; idx += 256) {
        int ty = idx / kTX, tx = idx - ty * kTX;
        const T* p = sin + ty * TW + tx;
        T mx = p[rx], mn = p[rx];                 // centre first: see the visiting order above
        for (int i = 0; i <= 2 * rx; i++) { T v = p[i]; mx = v > mx ? v : mx; mn = v < mn ? v : mn; }
        smx[idx] = mx; smn[idx] = mn;
    }
    __syncthreads();
    for (int ly = threadIdx.y; ly < kTY; ly += blockDim.y) {
        int x = x0 + threadIdx.x, y = y0 + ly;
        if (x >= W || y >= H) continue;
        T mx = smx[(ly + ry) * kTX + threadIdx.x], mn = smn[(ly + ry) * kTX + threadIdx.x];
        for (int i = 0; i <= 2 * ry; i++) {
            T a = smx[(ly + i) * kTX + threadIdx.x], b = smn[(ly + i) * kTX + threadIdx.x];
            mx = a > mx ? a : mx; mn = b < mn ? b : mn;
        }
        T out;
        if (MODE == 1) out = mx;
        else if (MODE == 2) out = mn;
        else {
            T v = sin[(ly + ry) * TW + threadIdx.x + rx];
            T mind = absdiff_cv<T>(v, mn), maxd = absdiff_cv<T>(v, mx);
            T mask = maxd < mind ? maxd : mind;             // cv::min
            out = (mind == mask) ? mn : mx;
        }
        fdst[((size_t)y * W + x) * cn + c] = out;
    }
}

template <typename T, int MODE>
static int launch_minmax_t(const void* src, void* dst, int n, int H, int W, int cn, int rx, int ry, cudaStream_t s) {
    dim3 grid((W + kTX - 1) / kTX, (H + kTY - 1) / kTY, n * cn), block(32, 8);
    int TW = kTX + 2 * rx, TH = kTY + 2 * ry;
    size_t smem = ((size_t)TW * TH + 2 * (size_t)TH * kTX) * sizeof(T);
    minmax_kernel<T, MODE><<<grid, block, smem, s>>>((const T*)src, (T*)dst, H, W, cn, rx, ry);
    return 1;
}

template <int MODE>
static int launch_minmax_mode(const void* src, void* dst, int n, int H, int W, int depth, int cn, int rx, int ry, cudaStream_t s) {
    switch (depth) {
    case 0: return launch_minmax_t<uint8_t, MODE>(src, dst, n, H, W, cn, rx, ry, s);
    case 2: return launch_minmax_t<uint16_t, MODE>(src, dst, n, H, W, cn, rx, ry, s);
    case 3: return launch_minmax_t<int16_t, MODE>(src, dst, n, H, W, cn, rx, ry, s);
    case 5: return launch_minmax_t<float, MODE>(src, dst, n, H, W, cn, rx, ry, s);
    case 6: return launch_minmax_t<double, MODE>(src, dst, n, H, W, cn, rx, ry, s);
    }
    return 0;
}

int launch_minmax(const void* src, void* dst, int n, int H, int W, int depth, int cn, int r, cudaStream_t s) {
    if (depth == 0 && cn == 1) if (int nk = launch_minmax8u_fast((const uint8_t*)src, (uint8_t*)dst, n, H, W, r, s)) return nk;
    return launch_minmax_mode<0>(src, dst, n, H, W, depth, cn, r, r, s);
}
int launch_morph(const void* src, void* dst, int n, int H, int W, int depth, int kw, int kh, int is_max, cudaStream_t s) {
    return is_max ? launch_minmax_mode<1>(src, dst, n, H, W, depth, 1, kw / 2, kh / 2, s)
                  : launch_minmax_mode<2>(src, dst, n, H, W, depth, 1, kw / 2, kh / 2, s);
}

// maxFilter / minFilter on 32F: the reference seeds its sliding window with FLT_MIN (max) / FLT_MAX (min)
// (minmaxFilter.cpp:332, :412) and the seed leaks into the output data-dependently, so the row-serial
// recurrence is reproduced literally: one thread per row, horizontal pass then the same pass on columns.
__global__ void minmax_filter_f32_seeded_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols,
                                                int sstride_row, int sstride_col, int width, float seed, int is_max) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    const float* s = src + (size_t)i * sstride_row; float* d = dst + (size_t)i * sstride_row;
    if (width == 1) { for (int j = 0; j < cols; j++) d[(size_t)j * sstride_col] = s[(size_t)j * sstride_col]; return; }
    const int rx = width / 2, st = width - 1;
#define SIM(k) s[(size_t)clampi((k) - rx, 0, cols - 1) * sstride_col]       /* copyMakeBorder(REPLICATE) row */
    float prev = seed;
    for (int k = 0; k < width; k++) { float v = SIM(k); prev = is_max ? (v > prev ? v : prev) : (v < prev ? v : prev); }
    d[0] = prev; float ed = SIM(0);
    for (int j = 1; j < cols; j++) {
        float nv = SIM(j + st);
        if (is_max ? (prev <= nv) : (prev >= nv)) { prev = nv; d[(size_t)j * sstride_col] = prev; }
        else if (ed != prev) { d[(size_t)j * sstride_col] = prev; ed = SIM(j); }
        else {
            float m = seed;
            for (int k = 0; k < width; k++) { float v = SIM(j + k); m = is_max ? (v > m ? v : m) : (v < m ? v : m); }
            d[(size_t)j * sstride_col] = m; prev = m; ed = SIM(j);
        }
    }
#undef SIM
}

int launch_minmax_filter_f32_seeded(const float* src, float* dst, float* tmp, int H, int W, int kw, int kh, int is_max, cudaStream_t s) {
    float seed = is_max ? FLT_MIN : FLT_MAX;
    minmax_filter_f32_seeded_kernel<<<(H + 127) / 128, 128, 0, s>>>(src, tmp, H, W, W, 1, kw, seed, is_max);       // rows
    minmax_filter_f32_seeded_kernel<<<(W + 127) / 128, 128, 0, s>>>(tmp, dst, W, H, 1, W, kh, seed, is_max);       // columns
    return 2;
}

// ----------------------------------------------------------------------------------------------------------
// 8-bit binary-weighted range filter (binalyWeightedRangeFilter.cpp:131-236 C1, :237-462 C3)
//   w = |v - c| <= th (C3: saturating L1 over the three channels); out = RNE(float(sum w*v) / float(sum w)).
// The sums are exact integers (< 2^24 for r <= 10), so their order is free; the one FP32 divide and the
// round-half-even conversion are done exactly as _mm_div_ps / _mm_cvtps_epi32 do.
// ----------------------------------------------------------------------------------------------------------
constexpr int kBX = 64, kBY = 16;   // output tile of the generic range-filter kernels

template <int CN>
__global__ void __launch_bounds__(256) bwrf8u_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int H, int W, RowSpan rs, int th) {
    extern __shared__ unsigned char smraw[];
    const int rH = rs.rH, rV = rs.rV, TW = kBX + 2 * rH, TH = kBY + 2 * rV;
    uint8_t* sm = smraw;                                            // TH x TW x CN, interleaved
    const size_t fo = (size_t)blockIdx.z * H * W * CN;
    const int x0 = blockIdx.x * kBX, y0 = blockIdx.y * kBY;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    for (int idx = tid; idx < TW * TH; idx += 256) {
        int ty = idx / TW, tx = idx - ty * TW;
        int gx = clampi(x0 - rH + tx, 0, W - 1), gy = clampi(y0 - rV + ty, 0, H - 1);
        const uint8_t* p = src + fo + ((size_t)gy * W + gx) * CN;
#pragma unroll
        for (int c = 0; c < CN; c++) sm[idx * CN + c] = p[c];
    }
    __syncthreads();
    for (int ly = threadIdx.y; ly < kBY; ly += blockDim.y)
        for (int lx = threadIdx.x; lx < kBX; lx += blockDim.x) {
            int x = x0 + lx, y = y0 + ly;
            if (x >= W || y >= H) continue;
            const uint8_t* pc = sm + ((ly + rV) * TW + lx + rH) * CN;
            int c0[CN], sum[CN], cnt = 0;
#pragma unroll
            for (int c = 0; c < CN; c++) { c0[c] = pc[c]; sum[c] = 0; }
            for (int i = -rV; i <= rV; i++) {
                int hw = rs.hw[i + rV];
                const uint8_t* pr = pc + i * TW * CN;
                for (int j = -hw; j <= hw; j++) {
                    int v[CN], d = 0;
#pragma unroll
                    for (int c = 0; c < CN; c++) { v[c] = pr[j * CN + c]; d += abs(v[c] - c0[c]); }
                    if (CN > 1) d = min(d, 255);
                    int w = d <= th;
#pragma unroll
                    for (int c = 0; c < CN; c++) sum[c] += w ? v[c] : 0;
                    cnt += w;
                }
            }
            float fw = (float)cnt;
#pragma unroll
            for (int c = 0; c < CN; c++)
                dst[fo + ((size_t)y * W + x) * CN + c] = sat_u8(sat_s16(cvround(__fdiv_rn((float)sum[c], fw))));
        }
}

int launch_bwrf8u(const uint8_t* src, uint8_t* dst, int n, int H, int W, int cn, const RowSpan& rs, int th, cudaStream_t s) {
    dim3 grid((W + kBX - 1) / kBX, (H + kBY - 1) / kBY, n), block(32, 8);
    size_t smem = (size_t)(kBX + 2 * rs.rH) * (kBY + 2 * rs.rV) * cn;
    if (cn == 1) bwrf8u_kernel<1><<<grid, block, smem, s>>>(src, dst, H, W, rs, th);
    else bwrf8u_kernel<3><<<grid, block, smem, s>>>(src, dst, H, W, rs, th);
    return 1;
}

}  // namespace dmc
