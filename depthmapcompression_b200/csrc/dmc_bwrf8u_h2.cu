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
// R = 4 with the flat path below, 2224 instructions = 34.8 KB at radius 5: uniform noise, which never leaves the tap
// loop, runs 2.3 % slower, flat test included).  A
// variant with a run-time loop over the horizontal offset, R = 8 and two shifted shared-memory copies was measured
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
// Warps.  A warp owns a 32 x 2R pixel block of the 128 x 4R tile: lanes 0-15 the upper R rows, lanes 16-31 the lower.
// On the chain's real input 32 x 8 blocks pass the flat test below about 10 points more often than 64 x 4 blocks.
//
// Flat warps.  Let F be a warp's square footprint in the staged tile (its block plus RAD on every side, widened to whole
// 4-pixel chunks; the staged tile already holds the REPLICATE border values, so F holds every value a tap of the warp can
// read), m and M the min and max over F, cmin and cmax over the warp's centres.  If M - cmin <= th and cmax - m <= th,
// every tap of every pixel of the warp is within th of its centre: N = ntaps and the filter is the disc mean
// RNE(sum v / ntaps).  cmax - cmin <= th is necessary for that and costs little, so F is read only when it holds.
// The flat path adds, per input row, the packed segment sums for every half-width (2 pixels per 32-bit word, 16-bit
// fields) into the R output rows.  The fields hold sum (v - m) <= ntaps * (M - m) <= ntaps * 2 * th < 2^16
// (static_assert below), so 32-bit adds of the biased words, wrapping, and one subtraction of ntaps * (0x6400 + m) per
// field at the end give them exactly.  ntaps is odd, so sum / ntaps is never a half-integer; it is at least
// 1 / (2 * ntaps) >= 1/634 away from one, more than the float spacing below 256 (2^-16), so the reference's float
// division cannot round it onto or across one either: RNE(float(sum) / float(ntaps)) equals
// m + (sum(v - m) + ntaps / 2) / ntaps  in integers.
template <int RAD, int R, bool FLUSH, bool EVEN>     // EVEN: W and dst allow 2-byte stores
__global__ void __launch_bounds__(256) bwrf8u_h2_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int H, int W, int th) {
    constexpr int TILE_H = 4 * R;                         // 2 warp rows of 2R
    constexpr int SH = TILE_H + 2 * RAD;
    constexpr int SWW = stride_of(R);                     // row stride in 32-bit words
    constexpr int NT = ntaps_of(RAD);
    static_assert(NT % 2 == 1 && (long)NT * 2 * (2048 / (2 * RAD + 1)) < 65536, "flat-path fields must not overflow");
    __shared__ __align__(16) uint32_t sm[SH * SWW];

    const size_t fo = (size_t)blockIdx.z * H * W;
    const int X0 = blockIdx.x * kTileW, Y0 = blockIdx.y * TILE_H;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    stage_tile16<SH, 1, false, SWW>(sm, src + fo, X0, Y0 - RAD, H, W, aligned16(src, W), tid);      // biased half2 words (0x6400 | byte)
    __syncthreads();

    const int lane = threadIdx.x, wx = threadIdx.y & 3, wy = threadIdx.y >> 2;
    const int xl = 32 * wx + 2 * (lane & 15);             // first pixel of this thread's pair inside the tile
    const int yl = 2 * R * wy + R * (lane >> 4);          // first output row of this thread inside the tile
    constexpr int E = RAD <= 6 ? 6 : (RAD <= 8 ? 8 : 10), NW = E + 1;     // words (x-E, x-E+1) .. (x+E, x+E+1) cover offsets -E .. E+1
    const uint32_t* base = sm + yl * SWW + (xl + kHalo - E) / 2;      // word holding pixels (x-E, x-E+1)

    __half2 c[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
        uint32_t cw = base[(r + RAD) * SWW + E / 2];      // pixels (x, x+1) of output row r
        c[r] = *reinterpret_cast<__half2*>(&cw);
    }

    // ---- flat-warp test.  The biased halves 0x6400 | byte order like their bit patterns: min / max of 16-bit fields ----
    auto h2u = [](__half2 h) { return *reinterpret_cast<const uint32_t*>(&h); };
    __half2 cmn = c[0], cmx = c[0];
#pragma unroll
    for (int r = 1; r < R; r++) { cmn = __hmin2(cmn, c[r]); cmx = __hmax2(cmx, c[r]); }
    const uint32_t cmin = __reduce_min_sync(0xFFFFFFFFu, min(h2u(cmn) & 0xFFFFu, h2u(cmn) >> 16));
    const uint32_t cmax = __reduce_max_sync(0xFFFFFFFFu, max(h2u(cmx) & 0xFFFFu, h2u(cmx) >> 16));
    bool flat = (int)(cmax - cmin) <= th;
    uint32_t m = 0;
    if (flat) {
        // F: rows 2R*wy .. 2R*wy + 2R + 2*RAD - 1, 4-pixel chunks Q0 .. Q0 + NQ - 1 of the warp's columns; lane l reads
        // chunk l % NQ of rows l / NQ, l / NQ + RPI, ... (lanes from RPI * NQ on read none)
        constexpr int Q0 = (kHalo - RAD) >> 2, NQ = ((kHalo + 31 + RAD) >> 2) - Q0 + 1, RPI = 32 / NQ, FR = 2 * R + 2 * RAD;
        __half2 fmn = c[0], fmx = c[0];
        const int fr = lane / NQ;
        const uint2* fp = reinterpret_cast<const uint2*>(sm + (2 * R * wy + fr) * SWW) + 8 * wx + Q0 + lane % NQ;
#pragma unroll
        for (int k = 0; k < (FR + RPI - 1) / RPI; k++) {
            if (fr < RPI && fr + k * RPI < FR) {
                const uint2 q = fp[k * RPI * (SWW / 2)];
                const __half2 a = *reinterpret_cast<const __half2*>(&q.x), b = *reinterpret_cast<const __half2*>(&q.y);
                fmn = __hmin2(fmn, __hmin2(a, b)); fmx = __hmax2(fmx, __hmax2(a, b));
            }
        }
        m = __reduce_min_sync(0xFFFFFFFFu, min(h2u(fmn) & 0xFFFFu, h2u(fmn) >> 16));
        const uint32_t M = __reduce_max_sync(0xFFFFFFFFu, max(h2u(fmx) & 0xFFFFu, h2u(fmx) >> 16));
        flat = (int)(M - cmin) <= th && (int)(cmax - m) <= th;
    }

    uint32_t o0[R], o1[R];                                // results, in the low byte
    if (flat) {
        // ---- flat warp: disc mean from packed per-row segment sums ----
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
