// dmc_prepare.cu -- pointcloudTest's preparation of sensor depth on frame batches (main.cpp:254-260):
// depth16U2disp8U -> fillOcclusion(0, FILL_DISPARITY) [-> transpose -> fillOcclusion -> transpose].
//
// Closed form of the row loop of fill_occlusion_kernel (fillOcclusion_<uchar>, depthmapUtil.cpp:548-590) for invalid = 0,
// edge = 255 and MAX_LENGTH = (int)(cols * 0.5), which are the only values this path takes.  Let e be the row after the
// edge setting (e[0] = e[cols-1] = 255) and call a pixel valid when e[p] != 0; both ends are valid.
//  1. A maximal run of invalid pixels [i, t) has valid neighbours e[i-1] and e[t], which no earlier step changed: filling
//     an earlier run writes dd = min of two valid values, itself nonzero, into that run only.  So as long as no run is
//     over-long, every run fills independently with min(e[i-1], e[t]), and the next-row read (t == cols) never happens,
//     because e[cols-1] = 255 is valid.
//  2. The first run with t - i > MAX_LENGTH blanks the whole row to 0.  Every later step then sees s[i-1] == 0, so its
//     dd = min(st, 0) = 0 whatever st is (the next row's first pixel included): it writes 0 or blanks again.  The
//     closing s[0] = s[1], s[cols-1] = s[cols-2] copy 0.  The row is all 0, independent of where the run lies.
//  3. Otherwise the closing copies give s[0] = f[1] and s[cols-1] = f[cols-2] of the filled row f (for cols = 2 both
//     are the edge value 255).
// So a row is: all 0 if any run of zeros between its ends is longer than MAX_LENGTH, else every zero replaced by the
// min of its nearest nonzero neighbours (ends counted as 255), then the two end copies.  The next row's first pixel
// never matters, so no kernel here reads a neighbouring row, column or frame.  tests/test_prepare_closed_form.py checks
// this statement against the serial CPU loop on every row over a small alphabet.
//
// The column pass of pointcloudTest (transpose, fillOcclusion, transpose) is the same closed form down each column with
// MAX_LENGTH = (int)(rows * 0.5).
#include "dmc_common.cuh"
#include "dmc_kernels.cuh"

namespace dmc {

namespace {

constexpr int kRowWarps = 8;         // rows per CTA of the row kernel, one warp each
constexpr int kColThreads = 128;     // columns per CTA of the column kernel, one thread each

// depth16U2disp8U of one pixel (convert_kernel, kind 2): the SSE body [0, sse) of a frame sign-extends and saturates,
// the scalar tail adds b and truncates.
__device__ __forceinline__ int disp_of_depth16(uint16_t v, bool body, float maf, float b) {
    const float s = body ? (float)(int)(int16_t)v : (float)(int)v;
    float r = __fdiv_rn(maf, s);
    if (!body || b != 0.f) r = __fadd_rn(r, b);
    const int iv = cvround(r);
    return body ? sat_u8(sat_s16(iv)) : (uint8_t)iv;
}

// Converted and row-filled frames: one warp per row of rows_total = frames * rows, pixels x0 + lane in tiles of 32.
// Pass 1 (left to right) writes each pixel's value, or for a zero the value of its nearest nonzero pixel to the left,
// and finds over-long runs; pass 2 (right to left) replaces each zero by the min of that and its nearest nonzero pixel
// to the right.  Both passes read the same source, so each lane rereads the pixels it wrote.
__global__ void __launch_bounds__(kRowWarps * 32) prepare_row_kernel(const uint16_t* __restrict__ src, uint8_t* __restrict__ dst, int rows_total,
                                                                     int rows, int cols, long sse, float fb, float a, float b) {
    const int w = blockIdx.x * kRowWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= rows_total) return;
    const uint16_t* s = src + (size_t)w * cols;
    uint8_t* d = dst + (size_t)w * cols;
    const long base = (long)(w % rows) * cols;          // index of the row's first pixel in its frame
    const int max_len = (int)(cols * 0.5);
    const float maf = __fmul_rn(a, fb);
    auto value = [&](int x) { return x == 0 || x == cols - 1 ? 255 : disp_of_depth16(s[x], base + x < sse, maf, b); };
    int lpos = 0, lval = 255;
    bool over = false;
    for (int x0 = 0; x0 < cols; x0 += 32) {
        const int x = x0 + lane;
        const int v = x < cols ? value(x) : 0;
        const unsigned m = __ballot_sync(0xffffffffu, v != 0);
        const unsigned below = m & ((1u << lane) - 1);
        const int src_lane = below ? 31 - __clz(below) : lane;
        const int pv = __shfl_sync(0xffffffffu, v, src_lane);
        const int ppos = below ? x0 + src_lane : lpos, pval = below ? pv : lval;
        if (v != 0 && x - ppos - 1 > max_len) over = true;
        if (x < cols) d[x] = (uint8_t)(v != 0 ? v : pval);
        const int hi = m ? 31 - __clz(m) : 0;
        const int hv = __shfl_sync(0xffffffffu, v, hi);
        if (m) { lpos = x0 + hi; lval = hv; }
    }
    if (__any_sync(0xffffffffu, over)) {
        for (int x = lane; x < cols; x += 32) d[x] = 0;
        return;
    }
    int rval = 255;
    for (int x0 = (cols - 1) & ~31; x0 >= 0; x0 -= 32) {
        const int x = x0 + lane;
        const int v = x < cols ? value(x) : 0;
        const unsigned m = __ballot_sync(0xffffffffu, v != 0);
        const unsigned above = m & ~((2u << lane) - 1);
        const int nv = __shfl_sync(0xffffffffu, v, above ? __ffs(above) - 1 : lane);
        if (x < cols && v == 0) { const int nval = above ? nv : rval; d[x] = (uint8_t)min((int)d[x], nval); }
        const int lv = __shfl_sync(0xffffffffu, v, m ? __ffs(m) - 1 : 0);
        if (m) rval = lv;
    }
    __syncwarp();
    if (lane == 0) { d[0] = d[1]; d[cols - 1] = d[cols - 2]; }
}

// The same fill down every column of frames of rows x cols (first-pass output src -> dst): one thread per column, so a
// warp reads 32 adjacent pixels of a row at a time.  frame = blockIdx.y.
__global__ void __launch_bounds__(kColThreads) prepare_col_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int rows, int cols) {
    const int x = blockIdx.x * kColThreads + threadIdx.x;
    if (x >= cols) return;
    const size_t off = (size_t)blockIdx.y * rows * cols + x;
    const uint8_t* s = src + off;
    uint8_t* d = dst + off;
    const int max_len = (int)(rows * 0.5);
    int lpos = 0, lval = 255;
    bool over = false;
#pragma unroll 4
    for (int y = 0; y < rows; y++) {
        const int v = y == 0 || y == rows - 1 ? 255 : s[(size_t)y * cols];
        if (v != 0) { over |= y - lpos - 1 > max_len; lpos = y; lval = v; }
        d[(size_t)y * cols] = (uint8_t)(v != 0 ? v : lval);
    }
    if (over) {
        for (int y = 0; y < rows; y++) d[(size_t)y * cols] = 0;
        return;
    }
    int rval = 255;
#pragma unroll 4
    for (int y = rows - 1; y >= 0; y--) {
        const int v = y == 0 || y == rows - 1 ? 255 : s[(size_t)y * cols];
        if (v != 0) rval = v;
        else d[(size_t)y * cols] = (uint8_t)min((int)d[(size_t)y * cols], rval);
    }
    d[0] = d[cols];
    d[(size_t)(rows - 1) * cols] = d[(size_t)(rows - 2) * cols];
}

}  // namespace

int launch_prepare_disp(const uint16_t* src, uint8_t* dst, uint8_t* scratch, int nf, int rows, int cols, float fb, float a, float b, int passes, cudaStream_t s) {
    if (nf <= 0) return 0;
    const long area = (long)rows * cols;
    const int rows_total = nf * rows;
    prepare_row_kernel<<<(rows_total + kRowWarps - 1) / kRowWarps, kRowWarps * 32, 0, s>>>(src, passes == 2 ? scratch : dst, rows_total, rows, cols,
                                                                                        (area / 16) * 16, fb, a, b);
    if (passes == 1) return 1;
    prepare_col_kernel<<<dim3((cols + kColThreads - 1) / kColThreads, nf), kColThreads, 0, s>>>(scratch, dst, rows, cols);
    return 2;
}

}  // namespace dmc
