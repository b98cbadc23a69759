// dmc_bwrf8u_h2.cu -- the hot kernel of the chain: 8-bit binary-weighted range filter, square window (circular tap
// set), in packed half-precision SIMD.
//
// Formulation.  For a centre c and a tap v (both 0..255):  w = [|v-c| <= th],  sum w*v = c * sum w + sum w*(v-c).
// With d = v-c, |w*d| <= th, so  S = sum w*d  and  N = sum w  stay integers of magnitude <= ntaps*th and <= ntaps.
// When ntaps*th <= 2048 every partial sum is exactly representable in fp16, so S and N can be accumulated with
// HFMA2 on two pixels at once -- 4 instructions per pixel pair per tap, spread over two pipes (measured on B200 with
// tools/ubench_pipes.cu: HFMA2/HADD2 issue at 2 warp-instructions/clk/SM on the FMA pipe, HSET2/LEA/PRMT at 2/clk/SM
// on the ALU pipe, so two of each per tap keeps both pipes and the 4/clk issue port equally busy):
//     d = v - c (HFMA2)   w = (|d| <= th) ? 1.0 : 0.0 (HSET2.BF)   S += w*d (HFMA2)   N15 += bits(w) >> 10 (LEA.HI)
// (bits(1.0h) >> 10 = 15 in each 16-bit lane, so N15 counts 15 per accepted tap: 15*317 < 65536, no lane overflow)
// and the result  RNE(float(c*N + S) / float(N))  is bit-identical to the reference's FP32 sums (which are exact
// integers as well) followed by _mm_div_ps / _mm_cvtps_epi32 (binalyWeightedRangeFilter.cpp:165-216).
//
// Data layout.  The CTA stages its input tile (+halo) in shared memory as fp16 with a +1024 bias (0x6400 | byte):
// the bias makes the byte->half conversion a byte permute and cancels in v - c.  A thread owns a 2-pixel-wide, R-row
// tall block of outputs; for every input row it loads 7 aligned half2 words, funnel-shifts the odd offsets, and
// reuses each tap vector for all the output rows whose window contains it (register tiling: ~0.5 LDS per 2x81 taps).
// R = 4 at radius >= 4 keeps the fully unrolled body near the 32 KB instruction cache (R = 8, 56 KB, ran 5x slower;
// R = 4 with the flat-strip path below, 2328 instructions = 36.4 KB at radius 5: uniform noise, which never leaves
// the tap loop, runs about 2 % slower than the tap loop alone, centre pre-test included).  A variant with a run-time loop over the horizontal offset, R = 8 and two shifted shared-memory copies was measured
// too: fewer loads per tap but more staging/loop instructions, 17.9 ms vs 16.0 ms per 1000 frames -- not kept.
#include "dmc_common.cuh"
#include "dmc_kernels.cuh"
#include "dmc_stage.cuh"

namespace dmc {

namespace {

constexpr int kHalo = kHalo16;    // staged halo in pixels (>= radius + 1; 16 keeps the staging loads aligned)
constexpr int kTileW = kTW;       // output tile width: 4 warps x 16 lanes x 2 pixels

__host__ __device__ constexpr int hw_of(int rad, int dy) {      // circle_halfwidth as a constant expression
    int lim = rad * rad - dy * dy, j = 0;
    while ((j + 1) * (j + 1) <= lim) j++;
    return j;
}

__host__ __device__ constexpr int ntaps_of(int rad) {
    int n = 0;
    for (int dy = -rad; dy <= rad; dy++) n += 2 * hw_of(rad, dy < 0 ? -dy : dy) + 1;
    return n;
}

// RNE(t / n) for integers 0 <= t <= 255 * n, n >= 1, t < 2^24, in place of an IEEE division (FCHK plus a subroutine call
// for the slow case).  q = RNE(t * rcp.approx(n)) is within 1 of the answer; e = t - q*n is exact (integers below
// 2^24), and q moves by one when |e| > n/2, or when |e| == n/2 and q is odd (round half to even).  For such t and n the
// result equals RNE(float(t) / float(n)); test_bwrf8_epilogue.py checks that for every t and n the filter can reach
// and for each reciprocal within one ulp of 1/n.  Returns 1.5 * 2^23 + result as float bits: the low byte is the result.
__device__ __forceinline__ uint32_t rne_div(float t, float n) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(n));
    const float qm = fmaf(t, r, 12582912.f);
    const float e = fmaf(12582912.f - qm, n, t), hn = 0.5f * n;
    const uint32_t q = __float_as_uint(qm), odd = q & 1u;
    return q + (uint32_t)(e > hn || (e == hn && odd)) - (uint32_t)(e < -hn || (e == -hn && odd));
}

// Row stride of the staged tile in words: a warp's two lane-rows read rows R apart, so R * stride = 16 (mod 32) puts
// them on disjoint banks.  No multiple of 4 (16-byte staging stores) satisfies that for R = 8, which keeps 80.
__host__ __device__ constexpr int stride_of(int R) {
    for (int s = kSW16 / 2; s < kSW16 / 2 + 32; s += 4)
        if ((R * s) % 32 == 16) return s;
    return kSW16 / 2;
}

// FLUSH: for thresholds with ntaps*th > 2048 the half accumulator S is folded into an FP32 accumulator after every
// input row (a row contributes at most 2*RAD+1 taps, so |S| <= (2*RAD+1)*th <= 2048 stays exact); +5 instructions
// per output row and input row.
//
// Strips.  A thread computes one strip of 2 x R outputs; the CTA's 256 strips tile its 128 x 4R outputs, strip id
// s = 32 * (4 * wy + wx) + lane at pixels (32 * wx + 2 * (lane % 16), 2R * wy + R * (lane / 16)), so that with the
// identity assignment a warp owns a 32 x 2R block, lanes 0-15 the upper R rows, lanes 16-31 the lower.
//
// Flat strips.  Let F be a strip's footprint in the staged tile: the NW words the tap loop reads (pixels x - E .. x + E + 1)
// over its R + 2*RAD input rows.  The staged tile already holds the REPLICATE border values, so F holds every value a
// tap of the strip can read.  Let m and M be the min and max over F, cmin and cmax over the strip's centres.  If
// M - cmin <= th and cmax - m <= th, every tap of every pixel of the strip is within th of its centre: N = ntaps and
// the filter is the disc mean RNE(sum v / ntaps).  cmax - cmin <= th is necessary for that and costs little, so F is
// read only in CTAs where some strip passes it (uniform noise never does).  F is taken separably: the CTA first writes
// the column min / max of every word column over the input rows of each strip row to shared memory (strip rows 2p and
// 2p+1 share all but R of their rows, so one thread takes both), then each thread folds its NW columns.
// The CTA then reassigns strips to threads: flat strips first, tap strips after, each in id order, and the one warp
// that would hold both runs the tap loop for all of its strips, so no warp pays for both paths.  On the chain's real
// input (bench.py, radius 5, th 10) 75 % of the 2 x 4 strips pass, against 39 % of 32 x 8 warps under the warp-wide
// test this replaced, and 29 % of the warps run the tap loop after regrouping.  Measured on a B200 (1000 W), range
// filter alone on 8 stacked frames of that input: 0.1022 -> 0.0801 ms; a constant frame 0.0414 -> 0.0433 ms (the
// strip test costs more than the warp test); uniform noise 0.1237 -> 0.1233 ms.  The timings imply that 54 % of the warps take the
// flat path, not 71 %: a CTA keeps its slot until its last tap warp ends, so flat warps beside tap warps free nothing
// (25 % tap strips cost 0.0739 ms as two tap warps in every CTA, 0.0674 ms as a quarter of the CTAs all tap).  Tap
// warps of scattered strips read shared memory with bank conflicts and store 2 bytes per lane at scattered rows; both
// measured at about 1 % (coalescing the stores through shared memory was slower).
// The flat path adds, per input row, the packed segment sums for every half-width (2 pixels per 32-bit word, 16-bit
// fields) into the R output rows.  The fields hold sum (v - m) <= ntaps * (M - m) <= ntaps * 2 * th < 2^16
// (static_assert below), so 32-bit adds of the biased words, wrapping, and one subtraction of ntaps * (0x6400 + m) per
// field at the end give them exactly.  ntaps is odd, so sum / ntaps is never a half-integer; it is at least
// 1 / (2 * ntaps) >= 1/634 away from one, more than the float spacing below 256 (2^-16), so the reference's float
// division cannot round it onto or across one either: RNE(float(sum) / float(ntaps)) equals
// m + (sum(v - m) + ntaps / 2) / ntaps  in integers.
template <int RAD, int R, bool FLUSH, bool EVEN>     // EVEN: W and dst allow 2-byte stores
__global__ void __launch_bounds__(256) bwrf8u_h2_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int H, int W, int th) {
    constexpr int TILE_H = 4 * R;                         // 4 strip rows of R
    constexpr int SH = TILE_H + 2 * RAD;
    constexpr int SWW = stride_of(R);                     // row stride in 32-bit words
    constexpr int NT = ntaps_of(RAD);
    constexpr int E = RAD <= 6 ? 6 : (RAD <= 8 ? 8 : 10), NW = E + 1;     // words (x-E, x-E+1) .. (x+E, x+E+1) cover offsets -E .. E+1
    constexpr int NC = 64 + E;                            // word columns any strip's footprint touches, from word (kHalo - E) / 2
    static_assert(NT % 2 == 1 && (long)NT * 2 * (2048 / (2 * RAD + 1)) < 65536, "flat-path fields must not overflow");
    __shared__ __align__(16) uint32_t sm[SH * SWW];
    __shared__ uint2 colmm[4][NC];                        // per strip row and word column: packed (min, max) over its input rows
    __shared__ uint32_t order[256];                       // thread -> strip id | footprint min << 8
    __shared__ uint32_t wflat[8];

    const size_t fo = (size_t)blockIdx.z * H * W;
    const int X0 = blockIdx.x * kTileW, Y0 = blockIdx.y * TILE_H;
    const int tid = threadIdx.y * 32 + threadIdx.x, lane = threadIdx.x;
    stage_tile16<SH, 1, false, SWW>(sm, src + fo, X0, Y0 - RAD, H, W, aligned16(src, W), tid);      // biased half2 words (0x6400 | byte)
    __syncthreads();

    int xl, yl;                                           // first pixel and first output row of this thread's strip inside the tile
    const uint32_t* base;                                 // word holding pixels (x-E, x-E+1) of the strip's first input row
    __half2 c[R];
    auto take_strip = [&](int s) {
        xl = 32 * ((s >> 5) & 3) + 2 * (s & 15);
        yl = R * (s >> 7 << 1 | (s >> 4 & 1));
        base = sm + yl * SWW + (xl + kHalo - E) / 2;
#pragma unroll
        for (int r = 0; r < R; r++) {
            uint32_t cw = base[(r + RAD) * SWW + E / 2];  // pixels (x, x+1) of output row r
            c[r] = *reinterpret_cast<__half2*>(&cw);
        }
    };
    take_strip(tid);

    // ---- flat-strip test.  The biased halves 0x6400 | byte order like their bit patterns: min / max of 16-bit fields ----
    auto h2u = [](__half2 h) { return *reinterpret_cast<const uint32_t*>(&h); };
    __half2 cmn = c[0], cmx = c[0];
#pragma unroll
    for (int r = 1; r < R; r++) { cmn = __hmin2(cmn, c[r]); cmx = __hmax2(cmx, c[r]); }
    const uint32_t cmin = min(h2u(cmn) & 0xFFFFu, h2u(cmn) >> 16), cmax = max(h2u(cmx) & 0xFFFFu, h2u(cmx) >> 16);
    const bool outside = X0 + xl >= W || Y0 + yl >= H;    // never stored: counted with the flat strips
    bool flat = false;
    uint32_t m = 0;
    if (__syncthreads_or(!outside && (int)(cmax - cmin) <= th)) {
        if (tid < 2 * NC) {
            // strip rows 2p and 2p+1 read input rows 2pR .. 2pR + R + 2RAD - 1 and (2p+1)R .. (2p+1)R + R + 2RAD - 1
            const int p = tid / NC, j = tid - p * NC;
            const uint32_t* col = sm + 2 * p * R * SWW + (kHalo - E) / 2 + j;
            uint32_t mn = col[R * SWW], mx = mn;
#pragma unroll
            for (int y = R + 1; y < R + 2 * RAD; y++) { mn = __vminu2(mn, col[y * SWW]); mx = __vmaxu2(mx, col[y * SWW]); }
            uint32_t amn = mn, amx = mx, bmn = mn, bmx = mx;
#pragma unroll
            for (int y = 0; y < R; y++) { amn = __vminu2(amn, col[y * SWW]); amx = __vmaxu2(amx, col[y * SWW]); }
#pragma unroll
            for (int y = R + 2 * RAD; y < 2 * R + 2 * RAD; y++) { bmn = __vminu2(bmn, col[y * SWW]); bmx = __vmaxu2(bmx, col[y * SWW]); }
            colmm[2 * p][j] = make_uint2(amn, amx);
            colmm[2 * p + 1][j] = make_uint2(bmn, bmx);
        }
        __syncthreads();
        const uint2* cm = &colmm[yl / R][xl / 2];
        uint32_t fmn = cm[0].x, fmx = cm[0].y;
#pragma unroll
        for (int i = 1; i < NW; i++) { const uint2 q = cm[i]; fmn = __vminu2(fmn, q.x); fmx = __vmaxu2(fmx, q.y); }
        m = min(fmn & 0xFFFFu, fmn >> 16);
        const uint32_t M = max(fmx & 0xFFFFu, fmx >> 16);
        flat = outside || ((int)(M - cmin) <= th && (int)(cmax - m) <= th);

        // ---- regroup: flat strips to the first threads, tap strips after them, both in id order.  The warp that would
        // hold both runs the tap loop for all its strips (exact for any strip): no warp runs both paths ----
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, flat);
        if (lane == 0) wflat[threadIdx.y] = __popc(bal);
        const int nflat = __syncthreads_count(flat);
        if (nflat >= 32 && nflat < 256) {                 // otherwise every thread keeps its own strip
            uint32_t before = 0;
#pragma unroll
            for (int w = 0; w < 8; w++) before += w < (int)threadIdx.y ? wflat[w] : 0u;
            const uint32_t rank = __popc(bal & ((1u << lane) - 1u));
            order[flat ? before + rank : nflat + 32 * threadIdx.y - before + lane - rank] = (uint32_t)tid | (m & 0xFFu) << 8;
            __syncthreads();
            const uint32_t o = order[tid];
            m = o >> 8;
            take_strip(o & 0xFFu);
        }
        flat = tid < (nflat & ~31);
    }
    uint32_t o0[R], o1[R];                                // results, in the low byte
    if (flat) {
        // ---- flat strip: disc mean from packed per-row segment sums ----
        uint32_t acc[R];
#pragma unroll
        for (int r = 0; r < R; r++) acc[r] = 0u;
#pragma unroll
        for (int yy = 0; yy < R + 2 * RAD; yy++) {
            uint32_t wd[NW];
#pragma unroll
            for (int i = 0; i < NW; i++) wd[i] = base[yy * SWW + i];
            auto tv = [&](int dx) { return (dx & 1) == 0 ? wd[(dx + E) / 2] : __byte_perm(wd[(dx + E - 1) / 2], wd[(dx + E + 1) / 2], 0x5432); };
            uint32_t seg[RAD + 1];                        // seg[h]: taps -h .. h of this row
            seg[0] = tv(0);
#pragma unroll
            for (int h = 1; h <= RAD; h++) seg[h] = seg[h - 1] + tv(-h) + tv(h);
#pragma unroll
            for (int r = 0; r < R; r++) {
                const int dy = yy - r - RAD, ady = dy < 0 ? -dy : dy;
                if (ady <= RAD) acc[r] += seg[hw_of(RAD, ady)];
            }
        }
        const uint32_t mb = m & 0xFFu, bias = (uint32_t)NT * ((0x6400u + mb) * 0x10001u);
#pragma unroll
        for (int r = 0; r < R; r++) {
            const uint32_t f = acc[r] - bias;
            o0[r] = mb + ((f & 0xFFFFu) + NT / 2) / NT; o1[r] = mb + ((f >> 16) + NT / 2) / NT;
        }
    } else {
        const __half2 th2 = __half2half2(__int2half_rn(th));
        __half2 S[R]; uint32_t N15[R]; float Sf0[FLUSH ? R : 1], Sf1[FLUSH ? R : 1];
#pragma unroll
        for (int r = 0; r < R; r++) {
            S[r] = __float2half2_rn(0.f); N15[r] = 0u;
            if (FLUSH) { Sf0[r] = 0.f; Sf1[r] = 0.f; }
        }
#pragma unroll
        for (int yy = 0; yy < R + 2 * RAD; yy++) {
            uint32_t wd[NW];
#pragma unroll
            for (int i = 0; i < NW; i++) wd[i] = base[yy * SWW + i];
#pragma unroll
            for (int dx = -RAD; dx <= RAD; dx++) {
                // tap vector for offset dx: pixels (x+dx, x+dx+1)
                uint32_t vb;
                if ((dx & 1) == 0) vb = wd[(dx + E) / 2];
                else vb = __byte_perm(wd[(dx + E - 1) / 2], wd[(dx + E + 1) / 2], 0x5432);
                const __half2 v = *reinterpret_cast<__half2*>(&vb);
                const int adx = dx < 0 ? -dx : dx;
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int dy = yy - r - RAD, ady = dy < 0 ? -dy : dy;
                    if (ady <= RAD && adx <= hw_of(RAD, ady)) {
                        const __half2 d = __hsub2(v, c[r]);
                        const __half2 w = __hle2(__habs2(d), th2);
                        S[r] = __hfma2(w, d, S[r]);
                        N15[r] += (*reinterpret_cast<const uint32_t*>(&w)) >> 10;
                    }
                }
            }
            if (FLUSH) {
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int dy = yy - r - RAD;
                    if (dy >= -RAD && dy <= RAD) { const float2 f = __half22float2(S[r]); Sf0[r] += f.x; Sf1[r] += f.y; S[r] = __float2half2_rn(0.f); }
                }
            }
        }
        // ---- out = RNE(float(c*N + S) / float(N)), as RNE(15*(c*N + S) / (15*N)): the factor 15 of the packed
        // counter leaves the quotient unchanged, so N15 is never divided by 15 ----
#pragma unroll
        for (int r = 0; r < R; r++) {
            const float2 cf = __half22float2(c[r]);
            const float2 sf = FLUSH ? make_float2(Sf0[r], Sf1[r]) : __half22float2(S[r]);
            const float n0 = (float)(N15[r] & 0xFFFFu), n1 = (float)(N15[r] >> 16);
            o0[r] = rne_div((cf.x - 1024.f) * n0 + 15.f * sf.x, n0); o1[r] = rne_div((cf.y - 1024.f) * n1 + 15.f * sf.y, n1);
        }
    }

    const int x = X0 + xl;
    if (x >= W) return;
    uint8_t* op = dst + fo + (size_t)(Y0 + yl) * W + x;
    const int yrem = H - (Y0 + yl);
#pragma unroll
    for (int r = 0; r < R; r++) {
        if (r < yrem) {
            if (EVEN) *reinterpret_cast<uint16_t*>(op) = (uint16_t)__byte_perm(o0[r], o1[r], 0x4440);
            else { op[0] = (uint8_t)o0[r]; if (x + 1 < W) op[1] = (uint8_t)o1[r]; }
        }
        op += W;
    }
}

template <int RAD, int R>
void launch_rr(const uint8_t* src, uint8_t* dst, int n, int H, int W, int th, bool flush, cudaStream_t s) {
    dim3 block(32, 8), grid((W + kTileW - 1) / kTileW, (H + 4 * R - 1) / (4 * R), n);
    const bool even = (W & 1) == 0 && (reinterpret_cast<size_t>(dst) & 1) == 0;
    if (flush) { if (even) bwrf8u_h2_kernel<RAD, R, true, true><<<grid, block, 0, s>>>(src, dst, H, W, th); else bwrf8u_h2_kernel<RAD, R, true, false><<<grid, block, 0, s>>>(src, dst, H, W, th); }
    else { if (even) bwrf8u_h2_kernel<RAD, R, false, true><<<grid, block, 0, s>>>(src, dst, H, W, th); else bwrf8u_h2_kernel<RAD, R, false, false><<<grid, block, 0, s>>>(src, dst, H, W, th); }
}

template <int RAD>
int launch_rad(const uint8_t* src, uint8_t* dst, int n, int H, int W, int th, bool flush, cudaStream_t s) {
    constexpr int R = RAD <= 3 ? 8 : (RAD <= 6 ? 4 : (RAD <= 8 ? 2 : 1));     // keeps the unrolled body (ntaps * R * 4 instructions) under the 32 KB instruction cache (R = 8 at RAD = 5 ran 5x slower)
    static_assert(RAD <= 10, "11 words per row cover offsets -10..11 only");
    if (R > 2 && (long)((W + kTileW - 1) / kTileW) * ((H + 4 * R - 1) / (4 * R)) * n < 2 * 148) launch_rr<RAD, 2>(src, dst, n, H, W, th, flush, s);   // few tiles (single small frame): shorter tiles fill the GPU
    else launch_rr<RAD, R>(src, dst, n, H, W, th, flush, s);
    return 1;
}

}  // namespace

int launch_bwrf8u_h2(const uint8_t* src, uint8_t* dst, int n, int H, int W, int radius, int th, int ntaps, cudaStream_t s) {
    if (radius < 1 || radius > 10 || th < 0 || (long)(2 * radius + 1) * th > 2048) return 0;
    const bool flush = (long)ntaps * th > 2048;
    switch (radius) {
    case 1: return launch_rad<1>(src, dst, n, H, W, th, flush, s);
    case 2: return launch_rad<2>(src, dst, n, H, W, th, flush, s);
    case 3: return launch_rad<3>(src, dst, n, H, W, th, flush, s);
    case 4: return launch_rad<4>(src, dst, n, H, W, th, flush, s);
    case 5: return launch_rad<5>(src, dst, n, H, W, th, flush, s);
    case 6: return launch_rad<6>(src, dst, n, H, W, th, flush, s);
    case 7: return launch_rad<7>(src, dst, n, H, W, th, flush, s);
    case 8: return launch_rad<8>(src, dst, n, H, W, th, flush, s);
    case 9: return launch_rad<9>(src, dst, n, H, W, th, flush, s);
    case 10: return launch_rad<10>(src, dst, n, H, W, th, flush, s);
    }
    return 0;
}

}  // namespace dmc
