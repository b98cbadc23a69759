// dmc_brf.cu -- boundary reconstruction filter (ref: boundaryReconstructionFilter.cpp:12-131) on sm_100a, and the fused
// min-max -> boundary-reconstruction extension (filter_ext.h; ref: minmaxFilter.cpp:48-174 followed by the same filter).
//
// What the reference computes per pixel: the list of distinct values in a circular window in first-encounter (raster tap)
// order, with a count and a sequential FP32 sum of tap distances per value; then two passes over that list (normalise,
// score) and the best-scoring value wins.  The sums are FP32 additions in tap order, so every (pixel, value) pair is a
// dependent chain and nothing slides from one pixel to the next.  The cost is finding the value's entry for every tap.
//
// Formulation here ("tile ranks"): a CTA stages its tile + halo once, gives every distinct value of the STAGED TILE a
// dense id (8-bit: direct table of 256; 16-bit / float / double: open-addressing hash in shared memory, compacted by a
// block scan), and rewrites the tile as ids.  A tap's id then addresses the thread's own (distance-sum, count) entry
// directly: [id][thread] in shared memory, one 8-byte load and store per tap, no search, no divergence, conflict-free
// (a half-warp touches 16 consecutive 8-byte words whatever the ids are).  First-encounter order is kept in a byte list
// [slot][thread] for the scoring passes.  Shared memory is a fixed pool of 8192 entries per 256-pixel tile; a tile with M
// distinct values runs P = min(256, 8192 / M) pixels at a time (whole warps), so tiles with up to 32 values (the usual case
// on decoded depth maps) keep every thread busy and a noisy tile with up to 256 values still runs out of shared memory,
// 32 pixels per pass.  Tiles with more than 256 distinct values, or float tiles holding NaN / -0 (whose `==` is not bit
// equality), fall back to the per-thread list of the reference inside the same kernel.
#include "dmc_common.cuh"
#include "dmc_kernels.cuh"

namespace dmc {

constexpr int kBrfMaxTaps = 320;    // circle of radius 10 has 317 taps
struct BrfTap { int off; float dist; };                  // off = di * TW + dj for the kernel's tile pitch; one 8-byte constant load per tap
struct alignas(16) BrfTaps { int n; int pad[3]; BrfTap t[kBrfMaxTaps]; };     // t is 16-byte aligned: two taps per constant load

// shared memory through 32-bit addresses: the tap loop below is scheduled by hand (ids of four taps, entries of two taps in
// flight) and must not be re-serialised by generic-pointer alias analysis
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint2 lds_v2(uint32_t a) { uint2 v; asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_v2(uint32_t a, uint2 v) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(a), "r"(v.x), "r"(v.y) : "memory"); }

constexpr int kTX = 32;             // tile width = one warp
constexpr int kPoolPerPixel = 32;    // (dist, count) entries per tile pixel: CTA pool = 32 * TY * 32 entries
constexpr int kMaxRanks = 256;
constexpr int kMaxTile = (kTX + 2 * kMaxRadius) * (8 + 2 * kMaxRadius);

template <typename T> struct BrfT;
template <> struct BrfT<uint8_t>  { typedef uint32_t key_t; static constexpr int kSlots = 256;  static constexpr bool kDirect = true;
    static __device__ float sub(uint8_t a, uint8_t b) { return (float)abs((int)a - (int)b); } static __device__ uint8_t cast(float f) { return (uint8_t)(int)f; }
    static __device__ float rangef(uint8_t mx, uint8_t mn) { return (float)((int)mx - (int)mn); }
    static __device__ bool plain(uint8_t) { return true; } static __device__ key_t key(uint8_t v) { return v; } static __device__ uint8_t val(key_t k) { return (uint8_t)k; } };
template <> struct BrfT<uint16_t> { typedef uint32_t key_t; static constexpr int kSlots = 2048; static constexpr bool kDirect = false;
    static __device__ float sub(uint16_t a, uint16_t b) { return (float)abs((int)a - (int)b); } static __device__ uint16_t cast(float f) { return (uint16_t)(int)f; }
    static __device__ float rangef(uint16_t mx, uint16_t mn) { return (float)((int)mx - (int)mn); }
    static __device__ bool plain(uint16_t) { return true; } static __device__ key_t key(uint16_t v) { return v; } static __device__ uint16_t val(key_t k) { return (uint16_t)k; } };
template <> struct BrfT<int16_t>  { typedef uint32_t key_t; static constexpr int kSlots = 2048; static constexpr bool kDirect = false;
    static __device__ float sub(int16_t a, int16_t b) { return (float)abs((int)a - (int)b); } static __device__ int16_t cast(float f) { return (int16_t)(int)f; }
    static __device__ float rangef(int16_t mx, int16_t mn) { return (float)((int)mx - (int)mn); }
    static __device__ bool plain(int16_t) { return true; } static __device__ key_t key(int16_t v) { return (uint16_t)v; } static __device__ int16_t val(key_t k) { return (int16_t)(uint16_t)k; } };
template <> struct BrfT<float>    { typedef uint32_t key_t; static constexpr int kSlots = 2048; static constexpr bool kDirect = false;
    static __device__ float sub(float a, float b) { return fabsf(__fsub_rn(a, b)); } static __device__ float cast(float f) { return f; }
    static __device__ float rangef(float mx, float mn) { return __fsub_rn(mx, mn); }
    static __device__ bool plain(float v) { return !(v != v) && __float_as_uint(v) != 0x80000000u; }
    static __device__ key_t key(float v) { return __float_as_uint(v); } static __device__ float val(key_t k) { return __uint_as_float(k); } };
template <> struct BrfT<double>   { typedef unsigned long long key_t; static constexpr int kSlots = 2048; static constexpr bool kDirect = false;
    static __device__ float sub(double a, double b) { return (float)fabs(__dsub_rn(a, b)); } static __device__ double cast(float f) { return (double)f; }
    static __device__ float rangef(double mx, double mn) { return (float)__dsub_rn(mx, mn); }
    static __device__ bool plain(double v) { return !(v != v) && (unsigned long long)__double_as_longlong(v) != 0x8000000000000000ull; }
    static __device__ key_t key(double v) { return (unsigned long long)__double_as_longlong(v); } static __device__ double val(key_t k) { return __longlong_as_double((long long)k); } };

// scoring passes of the reference (:80-125) over the thread's list; cnt(q) / dsum(q) / value(q) address entry q of the list
template <typename T, typename FC, typename FD, typename FSD, typename FV>
__device__ __forceinline__ T brf_score(int nd, int ntaps, T val0, float frec, float color, float space, FC cnt, FD dsum, FSD set_dsum, FV value) {
    if (nd == 1) return value(0);                                   // :80-84
    float maxDis = 0.f, minDis = FLT_MAX; int maxOcc = 0, minOcc = ntaps; T maxDiff = (T)0, minDiff = (T)255;
    for (int q = 0; q < nd; q++) {                                  // :93-103
        // the reference divides in double and narrows (:96).  With a 24-bit dividend and a count < 2^9 the exact quotient is
        // either a float midpoint or at least 2^-20 ulp away from one, so the double rounding cannot change the result:
        // the correctly rounded FP32 quotient is the same number.
        const int c = cnt(q);
        const float dq = __fdiv_rn(dsum(q), (float)c);
        set_dsum(q, dq);
        const float sq = BrfT<T>::sub(value(q), val0);
        maxDis = fmaxf(dq, maxDis); minDis = fminf(dq, minDis);
        maxOcc = max(c, maxOcc); minOcc = min(c, minOcc);
        const T s = BrfT<T>::cast(fabsf(sq));
        maxDiff = s > maxDiff ? s : maxDiff; minDiff = s < minDiff ? s : minDiff;
    }
    const float divOcc = (maxOcc == minOcc) ? 0.00000001f : __fdiv_rn(1.0f, (float)(maxOcc - minOcc));
    const float divDiff = (maxDiff == minDiff) ? 0.00000001f : __fdiv_rn(1.0f, BrfT<T>::rangef(maxDiff, minDiff));
    const float divDis = (maxDis == minDis) ? 0.00000001f : __fdiv_rn(1.0f, __fsub_rn(maxDis, minDis));
    float maxE = 0.f; T mind = val0; const float fmaxDiff = (float)maxDiff;
    for (int q = 0; q < nd; q++) {                                  // :113-125
        const T v = value(q);
        const float sq = BrfT<T>::sub(v, val0);
        float J = __fmul_rn(__fmul_rn(frec, (float)(cnt(q) - minOcc)), divOcc);
        J = __fadd_rn(J, __fmul_rn(__fmul_rn(color, __fsub_rn(fmaxDiff, sq)), divDiff));
        J = __fadd_rn(J, __fmul_rn(__fmul_rn(space, __fsub_rn(maxDis, dsum(q))), divDis));
        if (J > maxE) { maxE = J; mind = v; }
    }
    return mind;
}

// the reference's own per-pixel list with a linear search per value change (fallback for tiles the ranks cannot serve)
template <typename T, typename FTap>
__device__ __noinline__ T brf_pixel_list(const BrfTaps& taps, T val0, float frec, float color, float space, FTap tap) {
    T val[kBrfMaxTaps]; short cnt[kBrfMaxTaps]; float dist[kBrfMaxTaps];
    int nd = 1, rq = 0, rcnt = 1; T rv = tap(0); float rdist = taps.t[0].dist;
    val[0] = rv;
    for (int k = 1; k < taps.n; k++) {                              // :54-78; the entry of the current run stays in registers
        const T v = tap(k);
        if (v == rv) { rcnt++; rdist = __fadd_rn(rdist, taps.t[k].dist); continue; }
        cnt[rq] = (short)rcnt; dist[rq] = rdist;
        int q = 0;
        for (; q < nd; q++) if (v == val[q]) break;
        if (q < nd) { rcnt = cnt[q] + 1; rdist = __fadd_rn(dist[q], taps.t[k].dist); }
        else { val[nd] = v; nd++; rcnt = 1; rdist = taps.t[k].dist; }
        rq = q; rv = v;
    }
    cnt[rq] = (short)rcnt; dist[rq] = rdist;
    return brf_score<T>(nd, taps.n, val0, frec, color, space, [&](int q) { return (int)cnt[q]; }, [&](int q) { return dist[q]; },
                        [&](int q, float d) { dist[q] = d; }, [&](int q) { return val[q]; });
}

// blurRemoveMinMax_ select (ref: minmaxFilter.cpp:63-65, :83-89, :160-172): the window minimum if |v-min| == min(|v-min|, |v-max|),
// else the maximum; cv::absdiff saturates for 16S.  Used by the fused kernel while it stages the BRF tile.
template <typename T> __device__ __forceinline__ T brf_absdiff(T a, T b) { return a > b ? (T)(a - b) : (T)(b - a); }
template <> __device__ __forceinline__ int16_t brf_absdiff<int16_t>(int16_t a, int16_t b) { int d = (int)a - (int)b; d = d < 0 ? -d : d; return (int16_t)min(d, 32767); }
template <typename T> __device__ __forceinline__ T minmax_pick(T v, T mn, T mx) {
    const T mind = brf_absdiff<T>(v, mn), maxd = brf_absdiff<T>(v, mx);
    const T mask = maxd < mind ? maxd : mind;
    return (mind == mask) ? mn : mx;
}

// Shared memory (dynamic): [pool: kPool x 8 B][order: kPool B][ids: tile bytes][vals: 256 x sizeof(key)]
//   while ranking, the pool area holds the hash keys (kSlots x sizeof(key)) followed by slot -> id (kSlots x 2 B), and the
//   order area holds the tile as slot numbers (2 B each).
// A launch covers a batch of dense H x W frames: blockIdx.z is the frame.  Everything else is per CTA (staged tile, rank
// table, flat-tile exit, list fallback), so frames of one launch may take different paths.
template <typename T, int TY, bool FUSED>
__global__ void __launch_bounds__(kTX * TY) brf_rank_kernel(const T* __restrict__ src, T* __restrict__ dst, int H, int W, int rw, int rh, int mr,
                                                        const __grid_constant__ BrfTaps taps, float frec, float color, float space) {
    typedef typename BrfT<T>::key_t key_t;
    constexpr int NS = BrfT<T>::kSlots;
    constexpr int kNT = kTX * TY, kPool = kNT * kPoolPerPixel;
    constexpr key_t EMPTY = ~(key_t)0;
    extern __shared__ __align__(16) unsigned char smraw[];
    uint2* pool = (uint2*)smraw;
    uint8_t* order = smraw + (size_t)kPool * 8;
    uint8_t* ids = order + kPool;
    const int TW = kTX + 2 * rw, TH = TY + 2 * rh, NTILE = TW * TH;
    key_t* vals = (key_t*)(ids + ((NTILE + 15) & ~15));
    key_t* keys = (key_t*)smraw;                                    // ranking phase only
    uint16_t* slot_id = (uint16_t*)(keys + NS + 2);                 // keys[NS] is the reserved slot of a value whose bits equal EMPTY (an all-ones NaN)
    uint16_t* slot_tile = (uint16_t*)order;
    __shared__ int s_warp[kNT / 32], s_m, s_odd;
    // Frame 0 keeps the parameters as they are, and the fused kernel rebases dst only once its min-max tile is staged: both
    // keep register pressure at the single-image kernel's (rebasing unconditionally costs 1-8 registers, profiles/r09_brf_ptxas.md)
    if (blockIdx.z) { const size_t fo = (size_t)blockIdx.z * H * W; src += fo; if constexpr (!FUSED) dst += fo; }
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * kTX, y0 = blockIdx.y * TY;

    const int warp = tid >> 5, lane = tid & 31;
    constexpr int NW = TY;                                          // warps per CTA
    constexpr int RPW = (TY + 2 * kMaxRadius + NW - 1) / NW;        // tile rows per warp (upper bound)

    for (int i = tid; i < NS; i += kNT) keys[i] = EMPTY;
    if (tid == 0) s_odd = 0;
    if constexpr (FUSED) {
        // The BRF input is blurRemoveMinMax(src, mr): REPLICATE border for the min/max window (cv::dilate / erode ignore
        // out-of-image taps), then REFLECT_101 of that image.  Produced for the whole staged tile into `mm` (order area).
        T* mm = (T*)order;
        T* raw = (T*)(smraw + ((((size_t)NS + 2) * (sizeof(key_t) + 2) + 15) & ~(size_t)15));
        const int RW = TW + 2 * mr, RH = TH + 2 * mr;
        T* hmn = raw + RW * RH; T* hmx = hmn + RH * TW;
        const int gx0 = x0 - rw - mr, gy0 = y0 - rh - mr;
        if (gx0 >= 0 && gy0 >= 0 && gx0 + RW <= W && gy0 + RH <= H) {            // interior tile: separable min / max out of shared memory
            for (int idx = tid; idx < RW * RH; idx += kNT) { const int ry = idx / RW, rx = idx - ry * RW; raw[idx] = src[(size_t)(gy0 + ry) * W + gx0 + rx]; }
            __syncthreads();
            for (int idx = tid; idx < RH * TW; idx += kNT) {
                const int ry = idx / TW, tx = idx - ry * TW;
                const T* r = raw + ry * RW + tx;
                T mn = r[0], mx = mn;
                for (int j = 1; j <= 2 * mr; j++) { const T u = r[j]; mn = u < mn ? u : mn; mx = u > mx ? u : mx; }
                hmn[idx] = mn; hmx[idx] = mx;
            }
            __syncthreads();
            for (int idx = tid; idx < NTILE; idx += kNT) {
                const int ty = idx / TW, tx = idx - ty * TW;
                T mn = hmn[idx], mx = hmx[idx];
                for (int i = 1; i <= 2 * mr; i++) { const T a = hmn[idx + i * TW], c = hmx[idx + i * TW]; mn = a < mn ? a : mn; mx = c > mx ? c : mx; }
                mm[idx] = minmax_pick<T>(raw[(ty + mr) * RW + tx + mr], mn, mx);
            }
        } else {
            for (int idx = tid; idx < NTILE; idx += kNT) {
                const int ty = idx / TW, tx = idx - ty * TW;
                const int cy = reflect101(y0 - rh + ty, H), cx = reflect101(x0 - rw + tx, W);
                T mn = src[(size_t)cy * W + cx], mx = mn; const T c = mn;
                for (int i = -mr; i <= mr; i++) {
                    const T* row = src + (size_t)clampi(cy + i, 0, H - 1) * W;
                    for (int j = -mr; j <= mr; j++) { const T u = row[clampi(cx + j, 0, W - 1)]; mn = u < mn ? u : mn; mx = u > mx ? u : mx; }
                }
                mm[idx] = minmax_pick<T>(c, mn, mx);
            }
        }
    }
    __syncthreads();
    // ---- stage: copyMakeBorder(BORDER_DEFAULT = REFLECT_101) :19.  A warp takes whole tile rows (coalesced); all of a
    // thread's loads are issued before the first one is used, and the values / table slots stay in registers.
    T v[RPW][2]; uint16_t slot[RPW][2];
    {
        const int gx[2] = { reflect101(x0 - rw + lane, W), reflect101(x0 - rw + lane + 32, W) };
        #pragma unroll
        for (int rr = 0; rr < RPW; rr++) {
            const int ty = warp + rr * NW;
            if (ty < TH) {
                const int gy = reflect101(y0 - rh + ty, H);
                #pragma unroll
                for (int h = 0; h < 2; h++) if (lane + 32 * h < TW) {
                    if constexpr (FUSED) v[rr][h] = ((const T*)order)[ty * TW + lane + 32 * h];
                    else v[rr][h] = src[(size_t)gy * W + gx[h]];
                }
            }
        }
    }
    if constexpr (FUSED) __syncthreads();                           // `mm` shares the order area with the slot tile of the fallback path
    #pragma unroll
    for (int rr = 0; rr < RPW; rr++) {
        #pragma unroll
        for (int h = 0; h < 2; h++) if (warp + rr * NW < TH && lane + 32 * h < TW) {
            const key_t k = BrfT<T>::key(v[rr][h]);
            int sl;
            if constexpr (BrfT<T>::kDirect) { sl = (int)k; keys[sl] = k; }
            else {
                if (!BrfT<T>::plain(v[rr][h])) s_odd = 1;
                uint32_t hh = (uint32_t)k ^ (uint32_t)((unsigned long long)k >> 32);
                hh *= 0x9E3779B1u; sl = (int)(hh >> 21);            // top 11 bits: NS == 2048 (a tile holds at most 1456 elements)
                if (k == EMPTY) { sl = NS; keys[NS] = k; }          // (a NaN: the tile takes the list path, which reads the value back from here)
                else while (true) {
                    const key_t old = atomicCAS(&keys[sl], EMPTY, k);
                    if (old == EMPTY || old == k) break;
                    sl = (sl + 1) & (NS - 1);
                }
            }
            slot[rr][h] = (uint16_t)sl;
        }
    }
    __syncthreads();
    // ---- dense ids: block scan over the occupied slots
    {
        constexpr int SPT = NS / kNT;
        int n = 0;
        #pragma unroll
        for (int i = 0; i < SPT; i++) n += keys[tid * SPT + i] != EMPTY;
        int incl = n;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int base = 0, total = 0;
        #pragma unroll
        for (int w = 0; w < NW; w++) { const int c = s_warp[w]; if (w < warp) base += c; total += c; }
        if (tid == 0) s_m = total;
        int id = base + incl - n;
        #pragma unroll
        for (int i = 0; i < SPT; i++) {
            const key_t k = keys[tid * SPT + i];
            if (k != EMPTY) { slot_id[tid * SPT + i] = (uint16_t)id; if (id < kMaxRanks) vals[id] = k; id++; }
        }
    }
    __syncthreads();
    if constexpr (FUSED) if (blockIdx.z) dst += (size_t)blockIdx.z * H * W;
    const int M = s_m;
    const bool ranked = M <= kMaxRanks && M * 32 <= kPool && s_odd == 0;     // at least one warp of pixels per pass
    if (M == 1) {                                                   // a flat tile: every window holds that one value
        const T fv = BrfT<T>::val(vals[0]);
        for (int p = tid; p < kTX * TY; p += kNT) { const int x = x0 + (p & 31), y = y0 + (p >> 5); if (x < W && y < H) dst[(size_t)y * W + x] = fv; }
        return;
    }
    if (!ranked) {
        // per-thread lists on the staged values (keys[] still holds them: the pool is not used on this path)
        #pragma unroll
        for (int rr = 0; rr < RPW; rr++) {
            #pragma unroll
            for (int h = 0; h < 2; h++) if (warp + rr * NW < TH && lane + 32 * h < TW) slot_tile[(warp + rr * NW) * TW + lane + 32 * h] = slot[rr][h];
        }
        __syncthreads();
        for (int p = tid; p < kTX * TY; p += kNT) {
            const int px = p & 31, py = p >> 5, x = x0 + px, y = y0 + py;
            if (x >= W || y >= H) continue;
            const uint16_t* pc = slot_tile + (py + rh) * TW + px + rw;
            const T val0 = BrfT<T>::val(keys[pc[0]]);
            dst[(size_t)y * W + x] = brf_pixel_list<T>(taps, val0, frec, color, space, [&](int k) { return BrfT<T>::val(keys[pc[taps.t[k].off]]); });
        }
        return;
    }
    #pragma unroll
    for (int rr = 0; rr < RPW; rr++) {
        #pragma unroll
        for (int h = 0; h < 2; h++) if (warp + rr * NW < TH && lane + 32 * h < TW) ids[(warp + rr * NW) * TW + lane + 32 * h] = (uint8_t)slot_id[slot[rr][h]];
    }
    __syncthreads();                                                // keys / slot tables are dead from here: the pool takes over

    // ---- main passes: P pixels at a time, entry of id r for thread t at pool[r * P + t]
    const int P = min(kTX * TY, (kPool / M) & ~31);
    if (tid >= P) return;
    const uint32_t my = (uint32_t)__cvta_generic_to_shared(pool + tid);          // entry of id r: my + r * P8
    const uint32_t ord0 = (uint32_t)__cvta_generic_to_shared(order + tid);       // list slot q: ord0 + q * P
    const uint32_t ids0 = (uint32_t)__cvta_generic_to_shared(ids);
    const int P8 = P * 8;
    for (int r = 0; r < M; r++) sts_v2(my + r * P8, make_uint2(0u, 0u));      // later pixels of this thread: entries are cleared by their last reader
    for (int p0 = 0; p0 < kTX * TY; p0 += P) {
        const int p = p0 + tid, px = p & 31, py = p >> 5, x = x0 + px, y = y0 + py;
        if (py >= TY || y >= H) break;                              // later passes only hold rows further down
        if (x >= W) continue;
        const uint32_t pc = ids0 + (py + rh) * TW + px + rw;
        uint32_t ord = ord0;
        // :54-78, the same few instructions for every lane and tap.  0 + d == d, so the first tap of a value is no special case.
        // Four entries are in flight; a tap whose id equals an earlier one of the group continues from that one's registers
        // (the stores go out in tap order, so the last one wins).  The ids of the next group are fetched before the current
        // group's read-modify-write chain starts.
        auto upd = [&](uint2& e, uint32_t r, float d) {
            if (e.y == 0u) { sts_u8(ord, r); ord += P; }
            e.x = __float_as_uint(__fadd_rn(__uint_as_float(e.x), d)); e.y++;
        };
        const int n4 = taps.n & ~3;
        uint32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0;
        if (n4) { const uint4 c01 = *(const uint4*)&taps.t[0], c23 = *(const uint4*)&taps.t[2];
                  r0 = lds_u8(pc + c01.x); r1 = lds_u8(pc + c01.z); r2 = lds_u8(pc + c23.x); r3 = lds_u8(pc + c23.z); }
        for (int k = 0; k < n4; k += 4) {
            const uint4 c01 = *(const uint4*)&taps.t[k], c23 = *(const uint4*)&taps.t[k + 2];       // (off, dist) x 2
            const uint32_t a0 = my + r0 * P8, a1 = my + r1 * P8, a2 = my + r2 * P8, a3 = my + r3 * P8;
            uint2 e0 = lds_v2(a0), e1 = lds_v2(a1), e2 = lds_v2(a2), e3 = lds_v2(a3);
            const uint32_t q0 = r0, q1 = r1, q2 = r2, q3 = r3;
            if (k + 4 < n4) { const uint4 n01 = *(const uint4*)&taps.t[k + 4], n23 = *(const uint4*)&taps.t[k + 6];
                              r0 = lds_u8(pc + n01.x); r1 = lds_u8(pc + n01.z); r2 = lds_u8(pc + n23.x); r3 = lds_u8(pc + n23.z); }
            upd(e0, q0, __uint_as_float(c01.y));
            if (q1 == q0) e1 = e0;
            upd(e1, q1, __uint_as_float(c01.w));
            if (q2 == q0) e2 = e0;
            if (q2 == q1) e2 = e1;
            upd(e2, q2, __uint_as_float(c23.y));
            if (q3 == q0) e3 = e0;
            if (q3 == q1) e3 = e1;
            if (q3 == q2) e3 = e2;
            upd(e3, q3, __uint_as_float(c23.w));
            sts_v2(a0, e0); sts_v2(a1, e1); sts_v2(a2, e2); sts_v2(a3, e3);
        }
        for (int k = n4; k < taps.n; k++) {
            const uint32_t r = lds_u8(pc + taps.t[k].off), a = my + r * P8;
            uint2 e = lds_v2(a);
            upd(e, r, taps.t[k].dist);
            sts_v2(a, e);
        }
        const int nd = (int)(ord - ord0) / P;
        const uint32_t id0 = lds_u8(pc);
        const T val0 = BrfT<T>::val(vals[id0]);
        if constexpr (sizeof(T) <= 2) {
            // integer types: |val - val0| is an exact integer < 2^16, so the first pass leaves (mean distance, count | absdiff << 16)
            // in the entry and the second pass reads each entry once
            if (nd == 1) { const uint32_t id = lds_u8(ord0); sts_v2(my + id * P8, make_uint2(0u, 0u)); dst[(size_t)y * W + x] = BrfT<T>::val(vals[id]); continue; }      // :80-84
            // Both passes fetch the next list entry before they work on the current one (entries of a list are distinct, so the
            // early load never passes a store to the same entry).
            float maxDis = 0.f, minDis = FLT_MAX; int maxOcc = 0, minOcc = taps.n; T maxDiff = (T)0, minDiff = (T)255;
            uint32_t idn = lds_u8(ord0); uint2 en = lds_v2(my + idn * P8);
            for (int q = 0; q < nd; q++) {                              // :93-103 (the division: see brf_score)
                const uint32_t id = idn, a = my + id * P8; const uint2 e = en;
                if (q + 1 < nd) { idn = lds_u8(ord0 + (q + 1) * P); en = lds_v2(my + idn * P8); }
                const int c = (int)e.y;
                // x / 1 == x; keeping a zero numerator (the centre tap alone) out of the divider keeps it on its fast path
                const float num = __uint_as_float(e.x);
                const float dq = c == 1 ? num : __fdiv_rn(num, (float)c);
                const int ad = abs((int)BrfT<T>::val(vals[id]) - (int)val0);
                sts_v2(a, make_uint2(__float_as_uint(dq), e.y | ((uint32_t)ad << 16)));
                maxDis = fmaxf(dq, maxDis); minDis = fminf(dq, minDis);
                maxOcc = max(c, maxOcc); minOcc = min(c, minOcc);
                const T sd = BrfT<T>::cast((float)ad);
                maxDiff = sd > maxDiff ? sd : maxDiff; minDiff = sd < minDiff ? sd : minDiff;
            }
            const float divOcc = (maxOcc == minOcc) ? 0.00000001f : __fdiv_rn(1.0f, (float)(maxOcc - minOcc));
            const float divDiff = (maxDiff == minDiff) ? 0.00000001f : __fdiv_rn(1.0f, BrfT<T>::rangef(maxDiff, minDiff));
            const float divDis = (maxDis == minDis) ? 0.00000001f : __fdiv_rn(1.0f, __fsub_rn(maxDis, minDis));
            float maxE = 0.f; uint32_t best = id0; const float fmaxDiff = (float)maxDiff;
            idn = lds_u8(ord0); en = lds_v2(my + idn * P8);
            for (int q = 0; q < nd; q++) {                              // :113-125
                const uint32_t id = idn, a = my + id * P8; const uint2 e = en;
                if (q + 1 < nd) { idn = lds_u8(ord0 + (q + 1) * P); en = lds_v2(my + idn * P8); }
                sts_v2(a, make_uint2(0u, 0u));
                float J = __fmul_rn(__fmul_rn(frec, (float)((int)(e.y & 0xffffu) - minOcc)), divOcc);
                J = __fadd_rn(J, __fmul_rn(__fmul_rn(color, __fsub_rn(fmaxDiff, (float)(e.y >> 16))), divDiff));
                J = __fadd_rn(J, __fmul_rn(__fmul_rn(space, __fsub_rn(maxDis, __uint_as_float(e.x))), divDis));
                if (J > maxE) { maxE = J; best = id; }
            }
            dst[(size_t)y * W + x] = BrfT<T>::val(vals[best]);
        } else {
            uint2* const myp = pool + tid; const uint8_t* const ordp = order + tid;
            auto ent = [&](int q) { return myp + (int)ordp[q * P] * P; };
            dst[(size_t)y * W + x] = brf_score<T>(nd, taps.n, val0, frec, color, space,
                [&](int q) { return (int)ent(q)->y; }, [&](int q) { return __uint_as_float(ent(q)->x); },
                [&](int q, float d) { ent(q)->x = __float_as_uint(d); }, [&](int q) { return BrfT<T>::val(vals[ordp[q * P]]); });
            for (int q = 0; q < nd; q++) *ent(q) = make_uint2(0u, 0u);
        }
    }
}

template <typename T, int TY, bool FUSED>
static int launch_brf_rank(const void* src, void* dst, int nf, int H, int W, int rw, int rh, int mr, const BrfTaps& taps, float frec, float color, float space, cudaStream_t s) {
    typedef typename BrfT<T>::key_t key_t;
    const int ntile = (kTX + 2 * rw) * (TY + 2 * rh);
    constexpr int kNT = kTX * TY, kPool = kNT * kPoolPerPixel;
    const size_t smem = (size_t)kPool * 9 + ((ntile + 15) & ~15) + kMaxRanks * sizeof(key_t);
    static_assert(((size_t)BrfT<T>::kSlots + 2) * (sizeof(key_t) + 2) <= (size_t)kPool * 8, "hash tables must fit the pool area");
    auto kern = brf_rank_kernel<T, TY, FUSED>;
    // (the attribute is per function AND per device: set on every call, ~1 us, so that every GPU of a scheduler gets it)
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kPool * 9 + kMaxTile + 16 + kMaxRanks * sizeof(key_t))) != cudaSuccess) return 0;
    dim3 grid((W + kTX - 1) / kTX, (H + TY - 1) / TY, nf);
    kern<<<grid, kNT, smem, s>>>((const T*)src, (T*)dst, H, W, rw, rh, mr, taps, frec, color, space);
    return 1;
}

static bool make_brf_taps(int kw, int kh, BrfTaps* taps) {
    const int rw = kw / 2, rh = kh / 2, TW = kTX + 2 * rw;
    taps->n = 0;
    for (int i = -rh; i <= rh; i++) for (int j = -rw; j <= rw; j++) {                      // :26-38
        const double r = sqrt((double)i * i + (double)j * j);
        if (r > rw) continue;
        if (taps->n >= kBrfMaxTaps) return false;
        taps->t[taps->n].off = i * TW + j; taps->t[taps->n].dist = (float)r; taps->n++;
    }
    return taps->n > 0;
}

constexpr int kBrfTY8 = 4;          // 8-bit tile height (a direct 256-slot table: small CTAs are cheap); hashed types keep 8 rows

template <bool FUSED>
static int launch_brf_any(const void* src, void* dst, int nf, int H, int W, int depth, int kw, int kh, int mr, float frec, float color, float space, cudaStream_t s) {
    BrfTaps taps;
    if (!make_brf_taps(kw, kh, &taps)) return 0;
    const int rw = kw / 2, rh = kh / 2;
    if (nf < 1 || nf > 65535) return 0;                                                   // grid z
    switch (depth) {
    case 0: return launch_brf_rank<uint8_t, FUSED ? 8 : kBrfTY8, FUSED>(src, dst, nf, H, W, rw, rh, mr, taps, frec, color, space, s);      // fused: taller tiles, less halo to min-max
    case 2: return launch_brf_rank<uint16_t, 8, FUSED>(src, dst, nf, H, W, rw, rh, mr, taps, frec, color, space, s);
    case 3: return launch_brf_rank<int16_t, 8, FUSED>(src, dst, nf, H, W, rw, rh, mr, taps, frec, color, space, s);
    case 5: if (FUSED) return 0; return launch_brf_rank<float, 8, false>(src, dst, nf, H, W, rw, rh, mr, taps, frec, color, space, s);
    case 6: if (FUSED) return 0; return launch_brf_rank<double, 8, false>(src, dst, nf, H, W, rw, rh, mr, taps, frec, color, space, s);
    }
    return 0;
}

int launch_brf(const void* src, void* dst, int nf, int H, int W, int depth, int kw, int kh, float frec, float color, float space, cudaStream_t s) {
    return launch_brf_any<false>(src, dst, nf, H, W, depth, kw, kh, 0, frec, color, space, s);
}

int launch_minmax_brf(const void* src, void* dst, int nf, int H, int W, int depth, int minmax_r, int kw, int kh, float frec, float color, float space, cudaStream_t s) {
    return launch_brf_any<true>(src, dst, nf, H, W, depth, kw, kh, minmax_r, frec, color, space, s);
}

}  // namespace dmc
