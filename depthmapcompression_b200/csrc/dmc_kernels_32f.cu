// dmc_kernels_32f.cu -- the floating-point half of the path on sm_100a: the 32-bit binary-weighted range
// filter (with the disparity->depth / integer conversions of the PostFilterSet entry points fused into its
// tile load and store), the disparity<->depth converters, fillOcclusion
// and reprojectXYZ.  Every float operation is written with an explicit round-to-nearest intrinsic so that no
// FMA contraction can change a bit (SURVEY.md 8a "parity hazards").
#include "dmc_common.cuh"
#include "dmc_kernels.cuh"

namespace dmc {

constexpr int kFX = 64, kFY = 16;   // output tile of the float range filter

template <int LOAD> __device__ __forceinline__ float load_as_f32(const void* p, size_t i, float maf);
template <> __device__ __forceinline__ float load_as_f32<LOAD_F32>(const void* p, size_t i, float) { return ((const float*)p)[i]; }
template <> __device__ __forceinline__ float load_as_f32<LOAD_U16>(const void* p, size_t i, float) { return (float)((const uint16_t*)p)[i]; }
template <> __device__ __forceinline__ float load_as_f32<LOAD_S16>(const void* p, size_t i, float) { return (float)((const int16_t*)p)[i]; }
template <> __device__ __forceinline__ float load_as_f32<LOAD_U8>(const void* p, size_t i, float) { return (float)((const uint8_t*)p)[i]; }
// disp8U2depth32F with b == 0 (depthmapUtil.cpp:935-968): depth = (a * focal_baseline) / disp, disp 0 -> +inf
template <> __device__ __forceinline__ float load_as_f32<LOAD_U8_DISP2DEPTH>(const void* p, size_t i, float maf) { return __fdiv_rn(maf, (float)((const uint8_t*)p)[i]); }

template <int STORE> __device__ __forceinline__ void store_from_f32(void* p, size_t i, float v);
template <> __device__ __forceinline__ void store_from_f32<STORE_F32>(void* p, size_t i, float v) { ((float*)p)[i] = v; }
template <> __device__ __forceinline__ void store_from_f32<STORE_U16>(void* p, size_t i, float v) { ((uint16_t*)p)[i] = sat_u16(cvround(v)); }   // convertTo(CV_16U)
template <> __device__ __forceinline__ void store_from_f32<STORE_S16>(void* p, size_t i, float v) { ((int16_t*)p)[i] = (int16_t)sat_s16(cvround(v)); }

// binalyWeightedRangeFilter_32f + BinalyWeightedRangeFilter_32f_InvokerSSE4 (binalyWeightedRangeFilter.cpp:471-663,
// :978-1029).  Taps in raster order, sequential FP32 accumulation  t += w*v, W += w  with w in {0.f, 1.f}; the
// product is a real multiply so that 0*inf = NaN propagates as in the SSE code (:525-526).
//
// `quirk`: for rH % 8 == 5 and cols % 4 == 0 the reference pads one column too few on the right (rpad = -1,
// :993-997), so the tap (i, +rH) of the LAST column reads the first element of the next line of its padded
// buffer.  That element is staged into the halo column W-1+rH here, which only that tap ever reads.
template <int CN, int LOAD, int STORE>
__global__ void __launch_bounds__(256) bwrf32f_kernel(const void* __restrict__ src, void* __restrict__ dst, int H, int W,
                                                      RowSpan rs, float th, float maf, int quirk) {
    extern __shared__ float smf[];
    const int rH = rs.rH, rV = rs.rV, TW = kFX + 2 * rH, TH = kFY + 2 * rV;
    const size_t fo = (size_t)blockIdx.z * H * W * CN;
    const int x0 = blockIdx.x * kFX, y0 = blockIdx.y * kFY;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    for (int idx = tid; idx < TW * TH; idx += 256) {
        int ty = idx / TW, tx = idx - ty * TW;
        int ux = x0 - rH + tx, uy = y0 - rV + ty;                  // unclamped (padded-buffer) coordinates
        int gx = clampi(ux, 0, W - 1), gy = clampi(uy, 0, H - 1);
        size_t base = fo + ((size_t)gy * W + gx) * CN;
#pragma unroll
        for (int c = 0; c < CN; c++) smf[idx * CN + c] = load_as_f32<LOAD>(src, base + c, maf);
        if (quirk && ux == W - 1 + rH) {
            bool has_next = uy + 1 <= H - 1 + rV;                  // next line of the padded buffer exists
            size_t same0 = fo + ((size_t)gy * W) * CN, next0 = fo + ((size_t)clampi(uy + 1, 0, H - 1) * W) * CN;
            if (CN == 1) { if (has_next) smf[idx] = load_as_f32<LOAD>(src, next0, maf); }
            else {
                smf[idx * CN + 0] = load_as_f32<LOAD>(src, same0 + 1, maf);
                smf[idx * CN + 1] = load_as_f32<LOAD>(src, same0 + 2, maf);
                if (has_next) smf[idx * CN + 2] = load_as_f32<LOAD>(src, next0, maf);
            }
        }
    }
    __syncthreads();
    for (int ly = threadIdx.y; ly < kFY; ly += blockDim.y)
        for (int lx = threadIdx.x; lx < kFX; lx += blockDim.x) {
            int x = x0 + lx, y = y0 + ly;
            if (x >= W || y >= H) continue;
            const float* pc = smf + ((ly + rV) * TW + lx + rH) * CN;
            float c0[CN], t[CN], wsum = 0.f;
#pragma unroll
            for (int c = 0; c < CN; c++) { c0[c] = pc[c]; t[c] = 0.f; }
            for (int i = -rV; i <= rV; i++) {
                int hw = rs.hw[i + rV];
                const float* pr = pc + i * TW * CN;
                for (int j = -hw; j <= hw; j++) {
                    float v[CN], d;
#pragma unroll
                    for (int c = 0; c < CN; c++) v[c] = pr[j * CN + c];
                    if (CN == 1) d = fabsf(__fsub_rn(c0[0], v[0]));
                    else d = __fadd_rn(__fadd_rn(fabsf(__fsub_rn(c0[CN - 1], v[CN - 1])), fabsf(__fsub_rn(c0[CN > 1 ? 1 : 0], v[CN > 1 ? 1 : 0]))),
                                       fabsf(__fsub_rn(c0[0], v[0])));
                    float w = d <= th ? 1.f : 0.f;
#pragma unroll
                    for (int c = 0; c < CN; c++) t[c] = __fmaf_rn(w, v[c], t[c]);      // exact product (w is 0 or 1): one rounding, as mul then add
                    wsum = __fadd_rn(wsum, w);
                }
            }
#pragma unroll
            for (int c = 0; c < CN; c++) store_from_f32<STORE>(dst, fo + ((size_t)y * W + x) * CN + c, __fdiv_rn(t[c], wsum));
        }
}

template <int CN, int LOAD>
static int launch_bwrf32f_ls(const void* src, void* dst, dim3 grid, size_t smem, int H, int W, const RowSpan& rs, float th, float maf, int quirk, int store_op, cudaStream_t s) {
    dim3 block(32, 8);
    switch (store_op) {
    case STORE_F32: bwrf32f_kernel<CN, LOAD, STORE_F32><<<grid, block, smem, s>>>(src, dst, H, W, rs, th, maf, quirk); return 1;
    case STORE_U16: bwrf32f_kernel<CN, LOAD, STORE_U16><<<grid, block, smem, s>>>(src, dst, H, W, rs, th, maf, quirk); return 1;
    case STORE_S16: bwrf32f_kernel<CN, LOAD, STORE_S16><<<grid, block, smem, s>>>(src, dst, H, W, rs, th, maf, quirk); return 1;
    }
    return 0;
}

int launch_bwrf32f(const void* src, void* dst, int n, int H, int W, int cn, const RowSpan& rs, float th,
                   int load_op, float maf, int store_op, cudaStream_t s) {
    if (cn == 1 && rs.rH == rs.rV && rs.rH >= 1 && rs.rH <= 10)
        if (int nk = launch_bwrf32f_tiled(src, dst, n, H, W, rs.rH, th, load_op, maf, store_op, s)) return nk;
    if (cn == 3 && rs.rH == rs.rV && rs.rH >= 1 && rs.rH <= 10)
        if (int nk = launch_bwrf32f_c3_tiled(src, dst, n, H, W, rs.rH, th, load_op, store_op, s)) return nk;
    dim3 grid((W + kFX - 1) / kFX, (H + kFY - 1) / kFY, n);
    size_t smem = (size_t)(kFX + 2 * rs.rH) * (kFY + 2 * rs.rV) * cn * sizeof(float);
    int quirk = (rs.rH % 8 == 5) && (W % 4 == 0);
    if (cn == 1) {
        switch (load_op) {
        case LOAD_F32: return launch_bwrf32f_ls<1, LOAD_F32>(src, dst, grid, smem, H, W, rs, th, maf, quirk, store_op, s);
        case LOAD_U16: return launch_bwrf32f_ls<1, LOAD_U16>(src, dst, grid, smem, H, W, rs, th, maf, quirk, store_op, s);
        case LOAD_S16: return launch_bwrf32f_ls<1, LOAD_S16>(src, dst, grid, smem, H, W, rs, th, maf, quirk, store_op, s);
        case LOAD_U8: return launch_bwrf32f_ls<1, LOAD_U8>(src, dst, grid, smem, H, W, rs, th, maf, quirk, store_op, s);
        case LOAD_U8_DISP2DEPTH: return launch_bwrf32f_ls<1, LOAD_U8_DISP2DEPTH>(src, dst, grid, smem, H, W, rs, th, maf, quirk, store_op, s);
        }
    } else if (cn == 3) {
        switch (load_op) {
        case LOAD_F32: return launch_bwrf32f_ls<3, LOAD_F32>(src, dst, grid, smem, H, W, rs, th, maf, quirk, store_op, s);
        case LOAD_U16: return launch_bwrf32f_ls<3, LOAD_U16>(src, dst, grid, smem, H, W, rs, th, maf, quirk, store_op, s);
        case LOAD_S16: return launch_bwrf32f_ls<3, LOAD_S16>(src, dst, grid, smem, H, W, rs, th, maf, quirk, store_op, s);
        }
    }
    return 0;
}

// ----------------------------------------------------------------------------------------------------------
// converters (depthmapUtil.cpp:685-1014).  Elements [0, sse) follow the SSE body (saturating packs), the last
// n % 16 the scalar tail (truncating casts).
// ----------------------------------------------------------------------------------------------------------
__global__ void convert_kernel(int kind, const void* __restrict__ src, void* __restrict__ dst, long n, long sse, float fb, float a, float b) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float maf = __fmul_rn(a, fb);
    if (kind == 0) {                                           // disp8U2depth32F :923-1014
        float s = (float)((const uint8_t*)src)[i];
        if (b == 0.f) ((float*)dst)[i] = i < sse ? __fdiv_rn(maf, s) : __fadd_rn(__fdiv_rn(maf, s), b);
        else if (i < n - sse) ((float*)dst)[i] = __fadd_rn(__fdiv_rn(maf, s), b);   // SSE body commented out: only the first n%16
        return;
    }
    float s;
    if (kind == 1) s = ((const float*)src)[i];                 // depth32F2disp8U :768-838
    else if (kind == 2) s = i < sse ? (float)(int)(int16_t)((const uint16_t*)src)[i] : (float)(int)((const uint16_t*)src)[i];   // :858-859 sign extension
    else s = (float)(int)((const int16_t*)src)[i];             // disp16S2depth16U :685-765
    float v = __fdiv_rn(maf, s);
    if (i >= sse || b != 0.f) v = __fadd_rn(v, b);
    int iv = cvround(v);
    if (kind == 3) ((uint16_t*)dst)[i] = i < sse ? (uint16_t)(int16_t)sat_s16(iv) : (uint16_t)iv;
    else ((uint8_t*)dst)[i] = i < sse ? sat_u8(sat_s16(iv)) : (uint8_t)iv;
}

int launch_convert(int kind, const void* src, void* dst, long n, float fb, float a, float b, cudaStream_t s) {
    if (n <= 0) return 0;
    convert_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(kind, src, dst, n, (n / 16) * 16, fb, a, b);
    return 1;
}

__global__ void f32_to_u16_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, long n) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = sat_u16(cvround(src[i]));
}
int launch_f32_to_u16(const float* src, uint16_t* dst, long n, cudaStream_t s) {
    if (n <= 0) return 0;
    f32_to_u16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, dst, n);
    return 1;
}

// ----------------------------------------------------------------------------------------------------------
// fillOcclusion_<T> / fillOcclusionInv_<T> (depthmapUtil.cpp:548-636): row-serial run filling, one thread/row.
// ----------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void fill_occlusion_kernel(T* __restrict__ img, const T* __restrict__ pristine, int rows, int cols, T invalid, T edge, int inv) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= rows) return;
    const int MAX_LENGTH = inv ? cols : (int)(cols * 0.5);
    T* s = img + (size_t)j * cols;
    s[0] = edge; s[cols - 1] = edge;
    for (int i = 1; i < cols - 1; i++) {
        if (s[i] == invalid) {
            int t = i;
            do { t++; if (t > cols - 1) break; } while (s[t] == invalid);
            // t == cols: the reference reads one element past the row = the (not yet processed) next row's first pixel
            T st = t <= cols - 1 ? s[t] : (j + 1 < rows ? pristine[(size_t)(j + 1) * cols] : invalid);
            const T dd = inv ? (s[i - 1] > st ? s[i - 1] : st) : (st < s[i - 1] ? st : s[i - 1]);
            if (t - i > MAX_LENGTH) { for (int n = 0; n < cols; n++) s[n] = invalid; }
            else { for (; i < t && i < cols; i++) s[i] = dd; }
        }
    }
    s[0] = s[1]; s[cols - 1] = s[cols - 2];
}

int launch_fill_occlusion(void* img, const void* pristine, int H, int W, int depth, double invalid, int inv, cudaStream_t s) {
    int blocks = (H + 63) / 64;
    switch (depth) {
    case 0: fill_occlusion_kernel<uint8_t><<<blocks, 64, 0, s>>>((uint8_t*)img, (const uint8_t*)pristine, H, W, (uint8_t)(int)invalid, inv ? 0 : 255, inv); return 1;
    case 3: fill_occlusion_kernel<int16_t><<<blocks, 64, 0, s>>>((int16_t*)img, (const int16_t*)pristine, H, W, (int16_t)(int)invalid, inv ? 0 : SHRT_MAX, inv); return 1;
    case 2: fill_occlusion_kernel<uint16_t><<<blocks, 64, 0, s>>>((uint16_t*)img, (const uint16_t*)pristine, H, W, (uint16_t)(int)invalid, inv ? 0 : USHRT_MAX, inv); return 1;
    case 5: fill_occlusion_kernel<float><<<blocks, 64, 0, s>>>((float*)img, (const float*)pristine, H, W, (float)(int)invalid, inv ? 0.f : FLT_MAX, inv); return 1;
    }
    return 0;
}

// ----------------------------------------------------------------------------------------------------------
// reprojectXYZ_<T> (depthmapUtil.cpp:450-481): xyz = (x*z, y*z, z==0 ? 10000 : z); x is the reference's running
// FP32 sum along the row (xtab, built by the host with the same serial adds), y = (j - ch) * fyinv.  Frame = blockIdx.z.
// ----------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void reproject_kernel(const T* __restrict__ depth, float* __restrict__ xyz, const float* __restrict__ xtab, int H, int W, float fyinv, float ch) {
    int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i >= W) return;
    const size_t g = ((size_t)blockIdx.z * H + j) * W + i;
    float y = __fmul_rn(__fsub_rn((float)j, ch), fyinv);
    float z = (float)depth[g];
    float* o = xyz + g * 3;
    o[0] = __fmul_rn(xtab[i], z); o[1] = __fmul_rn(y, z); o[2] = (z == 0) ? 10000.f : z;
}

int launch_reproject(const void* depth, float* xyz, const float* xtab, int frames, int H, int W, int dtype, float fyinv, float ch, cudaStream_t s) {
    if (frames <= 0) return 0;
    dim3 grid((W + 255) / 256, H, frames), block(256);
    switch (dtype) {
    case 0: reproject_kernel<uint8_t><<<grid, block, 0, s>>>((const uint8_t*)depth, xyz, xtab, H, W, fyinv, ch); return 1;
    case 3: reproject_kernel<int16_t><<<grid, block, 0, s>>>((const int16_t*)depth, xyz, xtab, H, W, fyinv, ch); return 1;
    case 2: reproject_kernel<uint16_t><<<grid, block, 0, s>>>((const uint16_t*)depth, xyz, xtab, H, W, fyinv, ch); return 1;
    case 5: reproject_kernel<float><<<grid, block, 0, s>>>((const float*)depth, xyz, xtab, H, W, fyinv, ch); return 1;
    }
    return 0;
}

// ----------------------------------------------------------------------------------------------------------
// cv::transpose (main.cpp:258, :260 between the two fillOcclusion passes): 32x32 shared-memory tiles
// ----------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void transpose_kernel(const T* __restrict__ src, T* __restrict__ dst, int H, int W) {
    __shared__ T t[32][33];
    int x = blockIdx.x * 32 + threadIdx.x, y0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) if (x < W && y0 + j < H) t[j][threadIdx.x] = src[(size_t)(y0 + j) * W + x];
    __syncthreads();
    int ox = blockIdx.y * 32 + threadIdx.x, oy0 = blockIdx.x * 32;          // dst is W rows x H cols
    for (int j = threadIdx.y; j < 32; j += blockDim.y) if (ox < H && oy0 + j < W) dst[(size_t)(oy0 + j) * H + ox] = t[threadIdx.x][j];
}

int launch_transpose(const void* src, void* dst, int H, int W, int elem_size, cudaStream_t s) {
    dim3 grid((W + 31) / 32, (H + 31) / 32), block(32, 8);
    switch (elem_size) {
    case 1: transpose_kernel<uint8_t><<<grid, block, 0, s>>>((const uint8_t*)src, (uint8_t*)dst, H, W); return 1;
    case 2: transpose_kernel<uint16_t><<<grid, block, 0, s>>>((const uint16_t*)src, (uint16_t*)dst, H, W); return 1;
    case 4: transpose_kernel<uint32_t><<<grid, block, 0, s>>>((const uint32_t*)src, (uint32_t*)dst, H, W); return 1;
    case 8: transpose_kernel<uint64_t><<<grid, block, 0, s>>>((const uint64_t*)src, (uint64_t*)dst, H, W); return 1;
    }
    return 0;
}

}  // namespace dmc
