// dmc_render.cu -- point-cloud render (SURVEY.md 8f-3): projectPointsSimple (ref:depthmapUtil.cpp:10-156),
// projectImagefromXYZ (:285-448), fillSmallHole (:187-283); call sites ref:main.cpp:341-373.
//
// The reference splats the points SERIALLY in raster order into a z-buffer: a point writes its pixel if it is nearer than
// what is there at that moment, and only then tries up to six neighbour pixels (isSub), two of which colour a different
// pixel than the one they z-test (:366-379, :409-422).  The result therefore depends on the visiting order.  It is
// reproduced here EXACTLY, in parallel:
//
//   * an "attempt" is (time = point index * 8 + ordinal, z, z-tested pixel q, coloured pixel c).  An attempt fires iff it
//     is considered and its z is below every considered attempt on q with an earlier time (the z values that fire on a
//     pixel decrease strictly, so "below all earlier considered" == "below the buffer at that moment").  Primary attempts
//     are always considered; a neighbour attempt is considered iff the primary attempt of its point fired.
//   * attempts are binned per z-tested pixel (count / exclusive scan / fill / per-pixel sort by time), then the fired bits
//     of the primaries are iterated to their fixed point: one thread per pixel walks its time-sorted list with a running
//     minimum.  Whether a primary fires depends only on attempts of EARLIER points, so the fixed point is unique and an
//     iteration that changes nothing has reached it.  Natural scenes settle in 3-5 iterations, but the count has no such
//     bound: point k's primary can depend on point k-1's through a neighbour attempt that z-tests k's pixel, and each such
//     link of a chain can cost an iteration (a 3 x W image can chain W/2 points).  So after max(32, n / 1024) iterations
//     (n pixels a frame) the frames that still changed are finished by splat_serial_kernel, one thread per frame replaying
//     the serial loop to get `fired`.  The cap is a choice: n / 1024 sweeps cost less than one serial replay of the frame
//     (DESIGN.md section 6 has the times), and 32 alone would send some coded 1080p views, which need more, to the replay.
//   * the colour of a pixel is that of the LATEST fired attempt that colours it (atomicMax on time), its depth the final
//     running minimum.
//   * a batch of F frames (one camera) is rendered at once: the kernels take the frame from the grid, a pixel's global
//     index is frame * n + local, while times, coloured pixels and the `fired` bits stay frame-local.  Only interior points
//     make attempts, so no attempt reaches into another frame.  One scan covers all F * n counters, and the fixed point
//     is iterated until no frame changed (one host read per iteration for the whole batch); the last iteration before the
//     serial finish also reports each frame's own change, so the finish replays only the frames that have not settled.
//
// The projection uses the reference's reciprocal: _mm_rcp_ps (:78) is a 2048-entry look-up on Intel CPUs, carried here as
// a table (dmc_rcp_intel.inc, verified against the instruction on all 2^32 operands by tools/gen_rcp_table.c); the last
// n%4 points take the reference's scalar tail with a true division (:88-97), as do all points when `exact_divide` is set.
#include "dmc_common.cuh"
#include "dmc_kernels.cuh"

namespace dmc {

__constant__ uint16_t c_rcp_tab[2048] = {
#include "dmc_rcp_intel.inc"
};

__device__ __forceinline__ float rcp_intel(float x) {
    const uint32_t b = __float_as_uint(x), s = b & 0x80000000u, E = (b >> 23) & 0xffu, m = b & 0x7fffffu;
    if (E == 0xffu) return __uint_as_float(m ? (b | 0x400000u) : s);
    if (E == 0u) return __uint_as_float(s | 0x7f800000u);
    if (E >= 253u) return __uint_as_float(s);
    return __uint_as_float(s | ((253u - E) << 23) | ((uint32_t)c_rcp_tab[m >> 12] << 11));
}

// (int)v as cvttss2si does it: out of range / NaN -> INT_MIN ("integer indefinite")
__device__ __forceinline__ int f2i_x86(float v) {
    if (!(v > -2147483904.f && v < 2147483648.f)) return (int)0x80000000u;
    return (int)v;
}
__device__ __forceinline__ int sub_wrap(int a, int b) { return (int)((unsigned)a - (unsigned)b); }

struct RenderCam { float r[3][3]; float t[3]; };

// F frames of n points, frame = blockIdx.y; the rcp / exact split is per frame (the reference's tail is per call)
__global__ void project_points_kernel(const float* __restrict__ xyz, float2* __restrict__ pt, long n, long n_rcp, RenderCam cam) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long g = (long)blockIdx.y * n + i;
    const float x = __fadd_rn(xyz[3 * g], cam.t[0]), y = __fadd_rn(xyz[3 * g + 1], cam.t[1]), z = __fadd_rn(xyz[3 * g + 2], cam.t[2]);
    auto dot = [&](int k) { return __fadd_rn(__fadd_rn(__fmul_rn(cam.r[k][0], x), __fmul_rn(cam.r[k][1], y)), __fmul_rn(cam.r[k][2], z)); };
    const float den = dot(2);
    const float div = i < n_rcp ? rcp_intel(den) : __fdiv_rn(1.f, den);
    pt[g] = make_float2(__fmul_rn(dot(0), div), __fmul_rn(dot(1), div));
}

// The attempts of interior point p of one frame (pt: that frame's points): calls f(ordinal, z-tested pixel index,
// coloured pixel index), all frame-local.  p +- 1 and p +- cols stay inside the frame because p is interior.
template <class F>
__device__ __forceinline__ void for_each_attempt(const float2* __restrict__ pt, long p, int rows, int cols, int is_sub, F f) {
    const float2 me = pt[p];
    const int x = f2i_x86(me.x), y = f2i_x86(me.y);
    if (!(x >= 1 && x < cols - 1 && y >= 1 && y < rows - 1)) return;
    const long q0 = (long)y * cols + x;
    f(0, q0, q0);
    if (!is_sub) return;
    int ord = 1;
    const bool down = sub_wrap(f2i_x86(pt[p + cols].y), y) > 1, right = sub_wrap(f2i_x86(pt[p + 1].x), x) > 1;
    if (down && right) { f(ord++, q0 + 1, q0 + 1); f(ord++, q0 + cols + 1, q0 + cols); f(ord++, q0 + cols, q0 + cols + 1); }      // (the last two colour each other's pixel)
    else if (right) f(ord++, q0 + 1, q0 + 1);
    else if (down) f(ord++, q0 + cols, q0 + cols);
    const bool up = sub_wrap(f2i_x86(pt[p - cols].y), y) < -1, left = sub_wrap(f2i_x86(pt[p - 1].x), x) < -1;
    if (up && left) { f(ord++, q0 - 1, q0 - 1); f(ord++, q0 - cols - 1, q0 - cols); f(ord++, q0 - cols, q0 - cols - 1); }
    else if (left) f(ord++, q0 - 1, q0 - 1);
    else if (up) f(ord++, q0 - cols, q0 - cols);
}

// time = frame-local point * 8 + ordinal; c = frame-local coloured pixel.  Pixel lists hold one frame's attempts only.
struct Attempt { uint32_t time; float z; uint32_t c; };

// The kernels over interior points take row j = j0 + blockIdx.y + 1 (gridDim.y is at most 65535: launch_interior splits
// taller images into several launches) and frame = blockIdx.z.  Counters, cursors and offsets are indexed by the global
// pixel frame * n + q.
__global__ void attempts_count_kernel(const float2* __restrict__ pt, uint32_t* __restrict__ cnt, int rows, int cols, int is_sub, int j0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x + 1, j = j0 + blockIdx.y + 1;
    if (i >= cols - 1 || j >= rows - 1) return;
    const long base = (long)blockIdx.z * rows * cols;
    for_each_attempt(pt + base, (long)j * cols + i, rows, cols, is_sub, [&](int, long q, long) { atomicAdd(&cnt[base + q], 1u); });
}

__global__ void attempts_fill_kernel(const float2* __restrict__ pt, const float* __restrict__ xyz, const uint32_t* __restrict__ offs, uint32_t* __restrict__ cursor,
                                     Attempt* __restrict__ att, int rows, int cols, int is_sub, int j0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x + 1, j = j0 + blockIdx.y + 1;
    if (i >= cols - 1 || j >= rows - 1) return;
    const long base = (long)blockIdx.z * rows * cols, p = (long)j * cols + i;
    const float z = xyz[3 * (base + p) + 2];
    for_each_attempt(pt + base, p, rows, cols, is_sub, [&](int ord, long q, long c) {
        const uint32_t slot = offs[base + q] + atomicAdd(&cursor[base + q], 1u);
        Attempt a; a.time = (uint32_t)p * 8u + (uint32_t)ord; a.z = z; a.c = (uint32_t)c;
        att[slot] = a;
    });
}

// kernel<<<...>>>(args..., j0) over the interior rows of `frames` frames, at most 65535 rows a launch -> launches
template <class Kernel, class... Args>
int launch_interior(Kernel kernel, int frames, int rows, int cols, cudaStream_t s, Args... args) {
    int nk = 0;
    for (int j0 = 0; j0 < rows - 2; j0 += 65535, nk++)
        kernel<<<dim3((cols + 255) / 256, rows - 2 - j0 < 65535 ? rows - 2 - j0 : 65535, frames), 256, 0, s>>>(args..., j0);
    return nk;
}

// exclusive scan of n counters: per-block sums, scan of the sums by one block, add
constexpr int kScanT = 256, kScanPer = 8;
__global__ void scan_blocks_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t* __restrict__ sums, long n) {
    __shared__ uint32_t warp_tot[kScanT / 32];
    const long base = ((long)blockIdx.x * kScanT + threadIdx.x) * kScanPer;
    uint32_t v[kScanPer], s = 0;
#pragma unroll
    for (int k = 0; k < kScanPer; k++) { v[k] = base + k < n ? in[base + k] : 0u; s += v[k]; }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t x = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) warp_tot[w] = x;
    __syncthreads();
    uint32_t wbase = 0, tot = 0;
#pragma unroll
    for (int k = 0; k < kScanT / 32; k++) { if (k < w) wbase += warp_tot[k]; tot += warp_tot[k]; }
    uint32_t run = wbase + x - s;
#pragma unroll
    for (int k = 0; k < kScanPer; k++) { if (base + k < n) out[base + k] = run; run += v[k]; }
    if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}
__global__ void scan_sums_kernel(uint32_t* __restrict__ sums, int nb) {      // one block; nb is small (n / 2048)
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < nb; b0 += 1024) {
        const int i = b0 + threadIdx.x;
        const uint32_t v = i < nb ? sums[i] : 0u;
        __shared__ uint32_t tmp[1024];
        tmp[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) { uint32_t y = threadIdx.x >= o ? tmp[threadIdx.x - o] : 0u; __syncthreads(); tmp[threadIdx.x] += y; __syncthreads(); }
        if (i < nb) sums[i] = carry + tmp[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry += tmp[1023];
        __syncthreads();
    }
}
__global__ void scan_add_kernel(uint32_t* __restrict__ out, const uint32_t* __restrict__ sums, long n) {
    const long base = ((long)blockIdx.x * kScanT + threadIdx.x) * kScanPer;
    const uint32_t add = sums[blockIdx.x];
#pragma unroll
    for (int k = 0; k < kScanPer; k++) if (base + k < n) out[base + k] += add;
}

// Pixel q of frame blockIdx.y (global pixel index frame * n + q) in the kernels below.
__global__ void attempts_sort_kernel(const uint32_t* __restrict__ offs, const uint32_t* __restrict__ cnt, Attempt* __restrict__ att, long n) {
    const long q = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const long g = (long)blockIdx.y * n + q;
    const uint32_t m = cnt[g];
    if (m < 2) return;
    Attempt* a = att + offs[g];
    if (m <= 48) {                                      // the usual case: a handful of entries
        for (uint32_t i = 1; i < m; i++) {
            const Attempt key = a[i]; uint32_t k = i;
            while (k > 0 && a[k - 1].time > key.time) { a[k] = a[k - 1]; k--; }
            a[k] = key;
        }
        return;
    }
    // a view that collapses many points onto one pixel: heap sort keeps the worst case at m log m
    auto sift = [&](uint32_t root, uint32_t end) {
        for (;;) {
            uint32_t child = 2 * root + 1;
            if (child >= end) return;
            if (child + 1 < end && a[child].time < a[child + 1].time) child++;
            if (a[root].time >= a[child].time) return;
            const Attempt t = a[root]; a[root] = a[child]; a[child] = t; root = child;
        }
    };
    for (uint32_t i = m / 2; i-- > 0;) sift(i, m);
    for (uint32_t end = m; end-- > 1;) { const Attempt t = a[0]; a[0] = a[end]; a[end] = t; sift(0, end); }
}

// One sweep of the fixed-point iteration over every frame; FINAL: also emits colours and depth.  `changed` is shared by
// the frames: the batch iterates until no frame changed.  frame_changed (the last sweep before the serial finish only,
// NULL in the others) receives each frame's own flag.
template <bool FINAL>
__global__ void attempts_sweep_kernel(const uint32_t* __restrict__ offs, const uint32_t* __restrict__ cnt, const Attempt* __restrict__ att, uint8_t* fired,
                                      int* __restrict__ changed, int* __restrict__ frame_changed, uint32_t* __restrict__ ckey, float* __restrict__ depth, long n) {
    const long q = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const long base = (long)blockIdx.y * n, g = base + q;
    const uint32_t m = cnt[g];
    const Attempt* a = att + offs[g];
    uint8_t* fr = fired + base;
    float cur = 10000.f;                                // depth.setTo(10000.f) :306
    for (uint32_t i = 0; i < m; i++) {
        const Attempt e = a[i];
        const uint32_t p = e.time >> 3, ord = e.time & 7u;
        const bool considered = ord == 0u || fr[p] != 0;
        const bool fires = considered && cur > e.z;     // `*zbuff > z` :325 (false for NaN)
        if (fires) { cur = e.z; if (FINAL) atomicMax(&ckey[base + e.c], e.time + 1u); }
        if (!FINAL && ord == 0u && (fr[p] != 0) != fires) { fr[p] = fires ? 1 : 0; *changed = 1; if (frame_changed) frame_changed[blockIdx.y] = 1; }
    }
    if (FINAL && depth) depth[g] = cur;
}

// The serial splat (ref:depthmapUtil.cpp:320-445) of the frames whose last sweep still changed, one thread per frame: a
// point's primary fires iff it is below the z-buffer at that moment, and only then do its neighbour attempts write.  Only
// `fired` is kept: the FINAL sweep then emits colours and depth from it as after a settled iteration.  zbuf: n floats a
// frame.
__global__ void splat_serial_kernel(const float2* __restrict__ pt, const float* __restrict__ xyz, const int* __restrict__ frame_changed,
                                    uint8_t* __restrict__ fired, float* __restrict__ zbuf, int frames, int rows, int cols, int is_sub) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= frames || !frame_changed[f]) return;
    const long n = (long)rows * cols, base = (long)f * n;
    float* zb = zbuf + base;
    uint8_t* fr = fired + base;
    for (long q = 0; q < n; q++) zb[q] = 10000.f;
    for (int j = 1; j < rows - 1; j++)
        for (int i = 1; i < cols - 1; i++) {
            const long p = (long)j * cols + i;
            const float z = xyz[3 * (base + p) + 2];
            bool won = false;
            for_each_attempt(pt + base, p, rows, cols, is_sub, [&](int ord, long q, long) {
                if (ord == 0) { won = zb[q] > z; fr[p] = won ? 1 : 0; if (won) zb[q] = z; }
                else if (won && zb[q] > z) zb[q] = z;
            });
        }
}

__global__ void render_resolve_kernel(const uint8_t* __restrict__ image, const uint32_t* __restrict__ ckey, uint8_t* __restrict__ dest, long n) {
    const long q = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const long base = (long)blockIdx.y * n, g = base + q;
    const uint32_t k = ckey[g];
    uint8_t b = 0, gr = 0, r = 0;                       // destimage.setTo(0) :288
    if (k) { const uint8_t* c = image + 3 * (base + (long)((k - 1u) >> 3)); b = c[0]; gr = c[1]; r = c[2]; }
    dest[3 * g] = b; dest[3 * g + 1] = gr; dest[3 * g + 2] = r;
}

// fillSmallHole :187-283: a pixel whose GREEN is 0 becomes the mean of the neighbours whose BLUE is not 0 (s[lstep+1-1]);
// cvRound of a double quotient; border pixels and non-holes keep dst's previous content.  Row j0 + blockIdx.y + 1, frame =
// blockIdx.z.
__global__ void fill_small_hole_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int rows, int cols, int j0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x + 1, j = j0 + blockIdx.y + 1;
    if (i >= cols - 1 || j >= rows - 1) return;
    const long step = (long)cols * 3, frame = (long)blockIdx.z * rows * step;
    const uint8_t* s = src + frame + j * step + 3 * i;
    if (s[1] != 0) return;
    int count = 0, b = 0, g = 0, r = 0;
#pragma unroll
    for (int dy = -1; dy <= 1; dy++)
#pragma unroll
        for (int dx = -1; dx <= 1; dx++) {
            if (!dy && !dx) continue;
            const uint8_t* q = s + dy * step + 3 * dx;
            if (q[0] != 0) { b += q[0]; g += q[1]; r += q[2]; count++; }
        }
    uint8_t* d = dst + frame + j * step + 3 * i;
    d[0] = count ? (uint8_t)__double2int_rn(__ddiv_rn((double)b, (double)count)) : 0;
    d[1] = count ? (uint8_t)__double2int_rn(__ddiv_rn((double)g, (double)count)) : 0;
    d[2] = count ? (uint8_t)__double2int_rn(__ddiv_rn((double)r, (double)count)) : 0;
}

// splitBGRLineInterleave (ref:split.cpp:167-177): interleaved 3-channel rows -> a B row, a G row and an R row per image row
template <typename T>
__global__ void split_line_interleave_kernel(const T* __restrict__ src, T* __restrict__ dst, int rows, int cols) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= cols) return;
    const T* s = src + ((size_t)y * cols + x) * 3;
    T* d = dst + (size_t)3 * y * cols + x;
    d[0] = s[0]; d[cols] = s[1]; d[2 * (size_t)cols] = s[2];
}
int launch_split_line_interleave(const void* src, void* dst, int rows, int cols, int elem, cudaStream_t s) {
    dim3 grid((cols + 255) / 256, rows);
    if (elem == 1) split_line_interleave_kernel<uint8_t><<<grid, 256, 0, s>>>((const uint8_t*)src, (uint8_t*)dst, rows, cols);
    else split_line_interleave_kernel<float><<<grid, 256, 0, s>>>((const float*)src, (float*)dst, rows, cols);
    return 1;
}

// ---- launchers ----------------------------------------------------------------------------------------------------
int launch_project_points(const float* xyz, float* pt, int frames, long n, const float kr[9], const float t[3], int exact_divide, cudaStream_t s) {
    if (frames <= 0 || n <= 0) return 0;
    RenderCam cam;
    for (int i = 0; i < 3; i++) { for (int j = 0; j < 3; j++) cam.r[i][j] = kr[3 * i + j]; cam.t[i] = t[i]; }
    project_points_kernel<<<dim3((unsigned)((n + 255) / 256), frames), 256, 0, s>>>(xyz, (float2*)pt, n, exact_divide ? 0 : 4 * (n / 4), cam);
    return 1;
}

size_t render_scratch_bytes(int frames, int rows, int cols) {
    const size_t n = (size_t)frames * rows * cols, nb = (n + kScanT * kScanPer - 1) / (kScanT * kScanPer);
    return n * 4 * 3 + nb * 4 + 256 + n * 7 * sizeof(Attempt) + n + 64;      // cnt, offs, cursor/ckey, block sums, attempts, fired
}

// Everything after the projection, up to the fixed point, for `frames` frames of rows x cols at once (one scan over all
// their counters: the caller keeps frames * rows * cols * 7 below 2^32).  `changed_host` is pinned memory the sweeps report
// through: one read per iteration for the whole batch; changed_dev holds 1 + frames ints (the shared flag, then the
// frames' own).  After render_sweep_cap(rows * cols) iterations the frames that still changed are finished by the serial
// splat (see the header), so the work is bounded whatever the input.  Returns the number of kernels launched, or -1 on a
// CUDA error.
int render_sweep_cap(long n) { return n / 1024 > 32 ? (int)(n / 1024) : 32; }
int launch_render(const uint8_t* image, const float* xyz, const float* pt, int frames, int rows, int cols, int is_sub, uint8_t* dest, float* depth,
                  void* scratch, int* changed_dev, int* changed_host, cudaStream_t s) {
    const long n = (long)rows * cols, nt = n * frames;
    if (nt <= 0) return 0;
    const int nb = (int)((nt + kScanT * kScanPer - 1) / (kScanT * kScanPer));
    uint32_t* cnt = (uint32_t*)scratch; uint32_t* offs = cnt + nt; uint32_t* cursor = offs + nt; uint32_t* sums = cursor + nt;
    Attempt* att = (Attempt*)(((uintptr_t)(sums + nb) + 63) & ~(uintptr_t)63);
    uint8_t* fired = (uint8_t*)(att + (size_t)nt * 7);
    int nk = 0;
    cudaMemsetAsync(cnt, 0, (size_t)nt * 4, s); cudaMemsetAsync(cursor, 0, (size_t)nt * 4, s); cudaMemsetAsync(fired, 1, (size_t)nt, s);
    if (cols > 2) nk += launch_interior(attempts_count_kernel, frames, rows, cols, s, (const float2*)pt, cnt, rows, cols, is_sub);
    scan_blocks_kernel<<<nb, kScanT, 0, s>>>(cnt, offs, sums, nt);
    scan_sums_kernel<<<1, 1024, 0, s>>>(sums, nb);
    scan_add_kernel<<<nb, kScanT, 0, s>>>(offs, sums, nt);
    nk += 3;
    if (cols > 2) nk += launch_interior(attempts_fill_kernel, frames, rows, cols, s, (const float2*)pt, xyz, offs, cursor, att, rows, cols, is_sub);
    const dim3 gq((unsigned)((n + 255) / 256), frames);
    attempts_sort_kernel<<<gq, 256, 0, s>>>(offs, cnt, att, n); nk++;
    if (is_sub) {
        const int cap = render_sweep_cap(n);
        for (int it = 0;; it++) {
            if (it == cap) {                        // not settled: the serial splat finishes the frames that still changed
                splat_serial_kernel<<<(frames + 31) / 32, 32, 0, s>>>((const float2*)pt, xyz, changed_dev + 1, fired, (float*)cursor, frames, rows, cols, is_sub); nk++;
                break;
            }
            int* frame_changed = it == cap - 1 ? changed_dev + 1 : nullptr;
            cudaMemsetAsync(changed_dev, 0, sizeof(int) * (frame_changed ? 1 + (size_t)frames : 1), s);
            attempts_sweep_kernel<false><<<gq, 256, 0, s>>>(offs, cnt, att, fired, changed_dev, frame_changed, nullptr, nullptr, n); nk++;
            cudaMemcpyAsync(changed_host, changed_dev, sizeof(int), cudaMemcpyDeviceToHost, s);
            if (cudaStreamSynchronize(s) != cudaSuccess) return -1;
            if (!*changed_host) break;
        }
    }
    uint32_t* ckey = cursor;                            // the fill cursors (and the serial splat's z-buffer) are no longer needed
    cudaMemsetAsync(ckey, 0, (size_t)nt * 4, s);
    attempts_sweep_kernel<true><<<gq, 256, 0, s>>>(offs, cnt, att, fired, nullptr, nullptr, ckey, depth, n);
    render_resolve_kernel<<<gq, 256, 0, s>>>(image, ckey, dest, n);
    return nk + 2;
}

int launch_fill_small_hole(const uint8_t* src, uint8_t* dst, int frames, int rows, int cols, cudaStream_t s) {
    if (rows <= 2 || cols <= 2 || frames <= 0) return 0;
    return launch_interior(fill_small_hole_kernel, frames, rows, cols, s, src, dst, rows, cols);
}

}  // namespace dmc
