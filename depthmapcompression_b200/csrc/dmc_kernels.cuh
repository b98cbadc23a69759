// dmc_kernels.cuh -- host-side launchers of the sm_100a kernels (implemented in dmc_kernels_*.cu).
// All images are dense device buffers; `n` frames of H x W (x cn) lie back to back and are processed by one
// launch (frame = blockIdx.z).  Launchers return the number of kernels they launched (0 = nothing to do).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dmc {

constexpr int kMaxRadius = 10;
constexpr int kMaxTapsRow = 2 * kMaxRadius + 1;

struct GaussTaps { float kx[kMaxTapsRow]; float ky[kMaxTapsRow]; int rx, ry; };   // getGaussianKernel taps (host computed)
struct RowSpan { signed char hw[kMaxTapsRow]; int rV, rH, ntaps; };               // circular window: half-width per row

RowSpan make_rowspan(int kw, int kh);                    // binalyWeightedRangeFilter.cpp:1066-1076
bool make_gauss_taps(int d, double sigma, int rows, int cols, GaussTaps* t);   // cv::getGaussianKernel (OpenCV 4.x)

// cv::medianBlur, 8UC1, BORDER_REPLICATE (postFilterSet.cpp:23,36,47,59)
int launch_median8u(const uint8_t* src, uint8_t* dst, int n, int H, int W, int r, cudaStream_t s);
// smallGaussianBlur on 8UC1: 8U -> 32F -> GaussianBlur(REFLECT_101) -> RNE/saturate 8U (postFilterSet.cpp:4-16)
int launch_gauss8u(const uint8_t* src, uint8_t* dst, int n, int H, int W, const GaussTaps& t, cudaStream_t s);
// blurRemoveMinMax_<T> (minmaxFilter.cpp:48-174); depth in {8U,16U,16S,32F,64F}, cn channels interleaved
int launch_minmax(const void* src, void* dst, int n, int H, int W, int depth, int cn, int r, cudaStream_t s);
// windowed max / min with out-of-image taps ignored (cv::dilate/erode; maxFilter/minFilter for integer types)
int launch_morph(const void* src, void* dst, int n, int H, int W, int depth, int kw, int kh, int is_max, cudaStream_t s);
// maxFilter/minFilter 32F with the reference's FLT_MIN / FLT_MAX seeds (minmaxFilter.cpp:256-414), row-serial
int launch_minmax_filter_f32_seeded(const float* src, float* dst, float* tmp, int H, int W, int kw, int kh, int is_max, cudaStream_t s);

// binalyWeightedRangeFilter_8u (binalyWeightedRangeFilter.cpp:1031-1082), C1 and C3
int launch_bwrf8u(const uint8_t* src, uint8_t* dst, int n, int H, int W, int cn, const RowSpan& rs, int th, cudaStream_t s);

// binalyWeightedRangeFilter_32f (:978-1029) with fused input / output conversions
enum LoadOp { LOAD_F32 = 0, LOAD_U16 = 1, LOAD_S16 = 2, LOAD_U8 = 3, LOAD_U8_DISP2DEPTH = 4 };
enum StoreOp { STORE_F32 = 0, STORE_U16 = 1, STORE_S16 = 2 };
int launch_bwrf32f(const void* src, void* dst, int n, int H, int W, int cn, const RowSpan& rs, float th,
                   int load_op, float maf, int store_op, cudaStream_t s);

// boundaryReconstructionFilter_<T> (boundaryReconstructionFilter.cpp:12-131) on nf dense H x W frames (1..65535, one launch);
// returns 0 (nothing launched) for a window or frame count the kernel cannot take
int launch_brf(const void* src, void* dst, int nf, int H, int W, int depth, int kw, int kh, float frec, float color, float space, cudaStream_t s);
// extension (filter_ext.h): blurRemoveMinMax(minmax_r) fused into the tile staging of the boundary reconstruction filter; 8U / 16U / 16S
int launch_minmax_brf(const void* src, void* dst, int nf, int H, int W, int depth, int minmax_r, int kw, int kh, float frec, float color, float space, cudaStream_t s);

// converters (depthmapUtil.cpp:685-1014); kind: 0 disp8U2depth32F, 1 depth32F2disp8U, 2 depth16U2disp8U, 3 disp16S2depth16U
int launch_convert(int kind, const void* src, void* dst, long n, float fb, float a, float b, cudaStream_t s);
int launch_f32_to_u16(const float* src, uint16_t* dst, long n, cudaStream_t s);   // Mat::convertTo(CV_16U)
// fillOcclusion_<T> / Inv_ (depthmapUtil.cpp:548-636): `pristine` is an untouched copy of `img`
int launch_fill_occlusion(void* img, const void* pristine, int H, int W, int depth, double invalid, int inv, cudaStream_t s);
int launch_transpose(const void* src, void* dst, int H, int W, int elem_size, cudaStream_t s);   // cv::transpose, single channel
// pointcloudTest's preparation of nf frames (dmc_prepare.cu): depth16U2disp8U -> fillOcclusion(0, FILL_DISPARITY), and with
// passes = 2 the column fill (transpose -> fillOcclusion -> transpose) from `scratch` (nf frames of 8 bits) into dst
int launch_prepare_disp(const uint16_t* src, uint8_t* dst, uint8_t* scratch, int nf, int rows, int cols, float fb, float a, float b, int passes, cudaStream_t s);
// reprojectXYZ_<T> (depthmapUtil.cpp:450-481) of `frames` frames: xtab[i] = running FP32 sum along the row, computed by the
// host and shared by the frames
int launch_reproject(const void* depth, float* xyz, const float* xtab, int frames, int H, int W, int dtype, float fyinv, float ch, cudaStream_t s);

}  // namespace dmc

namespace dmc {
// Fast path of the 8UC1 range filter for square kernels (radius 1..6): packed half2 arithmetic, two pixels per
// instruction, register-tiled over rows.  Exact (all intermediate values are integers below 2048), taken when
// ntaps * th <= 2048; returns 0 if the configuration is not covered (the caller then uses the generic kernel).
int launch_bwrf8u_h2(const uint8_t* src, uint8_t* dst, int n, int H, int W, int radius, int th, int ntaps, cudaStream_t s);
}

namespace dmc {
// Packed-SIMD fast paths of the three 8-bit front stages (dmc_front8u.cu); each returns 0 when the configuration is
// not covered and the caller falls back to the generic kernel of dmc_kernels_8u.cu.
int launch_median8u_fast(const uint8_t* src, uint8_t* dst, int n, int H, int W, int r, cudaStream_t s);          // r = 1, 2
int launch_gauss8u_fast(const uint8_t* src, uint8_t* dst, int n, int H, int W, const GaussTaps& t, cudaStream_t s);   // d = 3, 5
int launch_minmax8u_fast(const uint8_t* src, uint8_t* dst, int n, int H, int W, int r, cudaStream_t s);          // r = 1..5
}

namespace dmc {
// Register-tiled fast path of the single-channel 32-bit range filter, square window radius 1..7 (0 = not covered).
int launch_bwrf32f_tiled(const void* src, void* dst, int n, int H, int W, int radius, float th, int load_op, float maf, int store_op, cudaStream_t s);
int launch_bwrf32f_c3_tiled(const void* src, void* dst, int n, int H, int W, int radius, float th, int load_op, int store_op, cudaStream_t s);
}

#include "dmc_jpeg_parse.h"
namespace dmc {
// Baseline grayscale JPEG decoding (dmc_jpeg.cu).  `scratch`: sum of jpeg_scratch_bytes over the frames (FrameDesc::ds_offset
// points into it); `coefs` (n * blocks * 64 int16) is only needed when n_restart > 0 frames carry restart intervals.
size_t jpeg_scratch_bytes(uint64_t scan_bytes);
int launch_jpeg_decode(const uint8_t* blob, const void* desc, const void* hts, const void* qts, uint8_t* scratch, int16_t* coefs, uint8_t* dst,
                       int n, int n_restart, int H, int W, cudaStream_t s);
// Baseline colour JPEG decoding (dmc_jpeg_color.cu) to dense BGR in dst.  desc: n ColorFrameDescs whose ds_offset points
// into `scratch` (jpeg_scratch_bytes per frame), plane_offset into `planes` (color_plane_bytes) and, for the n_restart
// frames with restart intervals, coef_offset into `coefs` (color_blocks * 64 int16, zero on entry); max_blocks: the
// largest color_blocks of those frames.  ycc: the YccTables.
int launch_jpeg_color_decode(const uint8_t* blob, const void* desc, const void* hts, const void* qts, const void* ycc, uint8_t* scratch, uint8_t* planes,
                             int16_t* coefs, uint8_t* dst, int n, int n_restart, uint32_t max_blocks, int H, int W, cudaStream_t s);
// Baseline grayscale JPEG encoding (dmc_jpeg_enc.cu).  Per-frame scratch of a rows x cols frame: int16 coefficients, block
// records, packed scan words (reused by the decoder as de-stuffing scratch) and the slot the frame's stream is written to.
// optimize: optimised Huffman tables, which take opt_bytes more per frame (symbol counts, the frame's code tables and header).
struct JpegEncLayout { size_t blocks, coef_bytes, info_bytes, word_bytes, slot_bytes, opt_bytes; };
JpegEncLayout jpeg_enc_layout(int rows, int cols, bool optimize = false);
// n frames of src -> one stream per slot (slots + f * slot_bytes), its length in lens[f]; with desc != nullptr also the
// FrameDesc that decodes slot f in place (scan_offset / scan_end relative to `slots`, ds_offset relative to `words`).
// opt != nullptr (n x opt_bytes of a layout with optimize): optimised Huffman tables, every frame its own; the FrameDescs
// then refer to the HuffTable pair huff[2 f], huff[2 f + 1], which the encoder writes when huff != nullptr.
int launch_jpeg_encode(const uint8_t* src, const void* tabs, void* coefs, void* info, void* words, uint8_t* slots, uint32_t* lens, void* desc,
                       int n, int H, int W, cudaStream_t s, void* opt = nullptr, void* huff = nullptr);
// Baseline colour JPEG encoding (dmc_jpeg_color_enc.cu) of n dense 8UC3 BGR frames with luma factors hy x vy: the per-frame
// scratch has the gray encoder's parts (opt_bytes = 0), sized by jpeg_color_enc_layout.  tabs: a device EncColorTables.
// With desc != nullptr the encoder also writes the ColorFrameDesc that decodes slot f in place: *tmpl (the header's
// parse: geometry and table indices) with scan_offset / scan_end relative to `slots`, ds_offset relative to `words` and
// plane_offset = f * plane_bytes.
JpegEncLayout jpeg_color_enc_layout(int rows, int cols, int hy, int vy);
int launch_jpeg_color_encode(const uint8_t* src, const void* tabs, void* coefs, void* info, void* words, uint8_t* slots, uint32_t* lens,
                             void* desc, const dmcjpeg::ColorFrameDesc* tmpl, uint64_t plane_bytes, int n, int H, int W, int hy, int vy, cudaStream_t s);
// copies stream f (lens[f] bytes of slot f) to dst + offs[f]; max_len >= every lens[f]
int launch_jpeg_enc_gather(const uint8_t* slots, size_t slot_bytes, const uint32_t* lens, const uint64_t* offs, uint8_t* dst, int n, uint64_t max_len, cudaStream_t s);
}

namespace dmc {
// Exact per-frame sum of squared differences of n dense 8-bit frames of frame_bytes each (dmc_metrics.cu): sse0[f] = SSE(a, b0)
// and, when b1 != nullptr, sse1[f] = SSE(a, b1) in the same launch (a is read once).  Zeroes the outputs first.
int launch_sse_u8(const uint8_t* a, const uint8_t* b0, const uint8_t* b1, uint64_t* sse0, uint64_t* sse1, int n, size_t frame_bytes, cudaStream_t s);
// SSIM of n dense rows x cols 8-bit frames of `channels` (1 or 3, interleaved) channels, rows and cols >= 11 (dmc_metrics.cu):
// mssim[f] = MSSIM(a_f, b_f), the definition of dmc_ssim_batch.  `partial` holds n x ssim_partial_bytes(rows, cols, channels)
// bytes of per-tile sums; mssim (device, n doubles) is written in stream order.  Deterministic: no floating-point atomics.
size_t ssim_partial_bytes(int rows, int cols, int channels);
int launch_ssim_u8(const uint8_t* a, const uint8_t* b, double* partial, double* mssim, int n, int rows, int cols, int channels, cudaStream_t s);
}

namespace dmc {
// point-cloud render (dmc_render.cu), `frames` dense frames of n = rows x cols points / pixels back to back, one camera
int launch_project_points(const float* xyz, float* pt, int frames, long n, const float kr[9], const float t[3], int exact_divide, cudaStream_t s);
size_t render_scratch_bytes(int frames, int rows, int cols);
int launch_render(const uint8_t* image, const float* xyz, const float* pt, int frames, int rows, int cols, int is_sub, uint8_t* dest, float* depth,
                  void* scratch, int* changed_dev, int* changed_host, cudaStream_t s);
int launch_fill_small_hole(const uint8_t* src, uint8_t* dst, int frames, int rows, int cols, cudaStream_t s);
int launch_split_line_interleave(const void* src, void* dst, int rows, int cols, int elem, cudaStream_t s);
}

namespace dmc {
// Packed-half fast path of the 8UC3 range filter, square window radius 1..5, exact while ntaps*th <= 2048 (0 = not covered).
int launch_bwrf8u_c3_h2(const uint8_t* src, uint8_t* dst, int n, int H, int W, int radius, int th, int ntaps, cudaStream_t s);
// joint (guided) range filter: 8UC1 image averaged with weights from a guide of gcn = 1 or 3 channels (dmc_joint_bwrf.cu)
int launch_joint_bwrf8u(const uint8_t* src, const uint8_t* guide, uint8_t* dst, int n, int H, int W, int gcn, const RowSpan& rs, int th, cudaStream_t s);
}
