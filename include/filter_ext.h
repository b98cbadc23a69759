// filter_ext.h -- operators of libdmc_b200 that have NO counterpart in the reference's filter.h.  They live in their
// own header so that include/filter.h stays a truthful drop-in of the reference API (SURVEY.md section 8f-4).
#pragma once
#include "filter.h"
#include "util.h"
#include <cstring>

// Joint ("colour-guided") binary-weighted range filter: `src` (CV_8UC1 depth / disparity) is averaged over the window
// of binalyWeightedRangeFilter with the binary weights computed on `guide` (CV_8UC3: the saturated L1 colour distance of
// binalyWeightedRangeFilter.cpp:297-301; CV_8UC1: absolute difference) instead of on src itself.  Window, border
// (REPLICATE), (uchar)threshold, FP32 division and rounding are those of the reference's 8UC1 filter; with guide == src
// the result equals binalyWeightedRangeFilter(src, ...).  Only FULL_KERNEL is defined.
inline void jointBinalyWeightedRangeFilter(const Mat& src, const Mat& guide, Mat& dst, Size kernelSize, float threshold, int method = FULL_KERNEL)
{
	if (dst.empty()) dst.create(src.size(), src.type());
	dmc_image a = dmc_dropin::wrap(src), g = dmc_dropin::wrap(guide), b = dmc_dropin::wrap(dst);
	dmc_dropin::check(dmc_joint_bwrf(dmc_dropin::context(), &a, &g, &b, kernelSize.width, kernelSize.height, threshold, method), "jointBinalyWeightedRangeFilter");
}

// Fused min-max -> boundary reconstruction: blurRemoveMinMax(src, tmp, r) followed by boundaryReconstructionFilter(tmp,
// dest, ksize, frec, color, space) in one kernel (the intermediate image lives in shared memory only; src is read once).
// Bit-identical to the two reference calls (minmaxFilter.cpp:48-174, boundaryReconstructionFilter.cpp:12-131).
// Single channel CV_8U / CV_16U / CV_16S.
inline void minmaxBoundaryReconstructionFilter(const Mat& src, Mat& dest, const int r, Size ksize, const float frec, const float color, const float space)
{
	if (dest.empty()) dest.create(src.size(), src.type());
	dmc_image a = dmc_dropin::wrap(src), b = dmc_dropin::wrap(dest);
	dmc_dropin::check(dmc_minmax_boundary_reconstruction(dmc_dropin::context(), &a, &b, r, ksize.width, ksize.height, frec, color, space), "minmaxBoundaryReconstructionFilter");
}

namespace dmc_dropin {
inline void require_gray8(const Mat& m, const char* what) {
	if (m.type() == CV_8UC1 && !m.empty()) return;
#ifdef DMC_MINICV_HPP
	throw cv::Exception((std::string(what) + ": src must be a non-empty CV_8UC1 image").c_str(), __FILE__, __LINE__);
#else
	CV_Error(cv::Error::StsAssert, std::string(what) + ": src must be a non-empty CV_8UC1 image");
#endif
}
}  // namespace dmc_dropin

// Baseline JPEG encoding of a CV_8UC1 image on the GPU: `buf` receives the same bytes as
// cv::imencode(".jpg", src, buf, {IMWRITE_JPEG_QUALITY, quality}) with libjpeg-turbo.  quality in 0..100.
// optimize: optimised Huffman tables, the bytes of {IMWRITE_JPEG_QUALITY, quality, IMWRITE_JPEG_OPTIMIZE, 1}.
inline void jpegEncodeGray(const Mat& src, vector<uchar>& buf, int quality, bool optimize = false)
{
	dmc_dropin::require_gray8(src, "jpegEncodeGray");
	const Mat s = src.isContinuous() ? src : src.clone();
	const int flags = optimize ? DMC_JPEG_OPTIMIZE_HUFFMAN : 0;
	uint64_t cap = 0, off[2] = {0, 0};
	dmc_dropin::check(dmc_jpeg_encode_bound_ex(s.rows, s.cols, flags, &cap), "jpegEncodeGray");
	buf.resize((size_t)cap);
	dmc_dropin::check(dmc_jpeg_encode_gray_batch_ex(dmc_dropin::context(), s.data, DMC_MEM_HOST, 1, s.rows, s.cols, quality, flags, buf.data(), DMC_MEM_HOST, cap, off), "jpegEncodeGray");
	buf.resize((size_t)off[1]);
}

// JPEG round trip of a CV_8UC1 image on the GPU, the stream never leaving the device:
// dest = cv::imdecode(cv::imencode(".jpg", src, {IMWRITE_JPEG_QUALITY, quality}), 0).  Returns the stream's size in bytes
// (optimize: the size with optimised Huffman tables; dest is the same).
inline int degradeJPEGGray(const Mat& src, Mat& dest, int quality, bool optimize = false)
{
	dmc_dropin::require_gray8(src, "degradeJPEGGray");
	const Mat s = src.isContinuous() ? src : src.clone();
	Mat d;
	if (dest.data != src.data && dest.size() == src.size() && dest.type() == CV_8UC1 && dest.isContinuous()) d = dest;
	else d.create(src.size(), CV_8UC1);
	uint64_t bytes = 0;
	dmc_dropin::check(dmc_jpeg_degrade_gray_batch_ex(dmc_dropin::context(), s.data, d.data, 1, s.rows, s.cols, quality, optimize ? DMC_JPEG_OPTIMIZE_HUFFMAN : 0,
	                                                 DMC_MEM_HOST, &bytes), "degradeJPEGGray");
	if (d.data != dest.data) dest = d;
	return (int)bytes;
}

namespace dmc_dropin {
inline void require_color8(const Mat& m, const char* what) {
	if (m.type() == CV_8UC3 && !m.empty()) return;
#ifdef DMC_MINICV_HPP
	throw cv::Exception((std::string(what) + ": src must be a non-empty CV_8UC3 image").c_str(), __FILE__, __LINE__);
#else
	CV_Error(cv::Error::StsAssert, std::string(what) + ": src must be a non-empty CV_8UC3 image");
#endif
}
}  // namespace dmc_dropin

// Baseline colour JPEG encoding of a CV_8UC3 (BGR) image on the GPU: `buf` receives the same bytes as
// cv::imencode(".jpg", src, buf, {IMWRITE_JPEG_QUALITY, quality, IMWRITE_JPEG_SAMPLING_FACTOR, sampling}) with
// libjpeg-turbo.  quality in 0..100; sampling one of DMC_JPEG_SAMPLING_* (the values of cv::IMWRITE_JPEG_SAMPLING_FACTOR_*).
inline void jpegEncodeColor(const Mat& src, vector<uchar>& buf, int quality, int sampling = DMC_JPEG_SAMPLING_420)
{
	dmc_dropin::require_color8(src, "jpegEncodeColor");
	const Mat s = src.isContinuous() ? src : src.clone();
	uint64_t cap = 0, off[2] = {0, 0};
	dmc_dropin::check(dmc_jpeg_encode_color_bound(s.rows, s.cols, sampling, &cap), "jpegEncodeColor");
	buf.resize((size_t)cap);
	dmc_dropin::check(dmc_jpeg_encode_color_batch(dmc_dropin::context(), s.data, DMC_MEM_HOST, 1, s.rows, s.cols, quality, sampling, buf.data(), DMC_MEM_HOST, cap, off), "jpegEncodeColor");
	buf.resize((size_t)off[1]);
}

// Colour JPEG round trip of a CV_8UC3 image on the GPU, the stream never leaving the device:
// dest = cv::imdecode(cv::imencode(".jpg", src, {IMWRITE_JPEG_QUALITY, quality, IMWRITE_JPEG_SAMPLING_FACTOR, sampling}),
// IMREAD_COLOR).  Returns the stream's size in bytes.
inline int degradeJPEGColor(const Mat& src, Mat& dest, int quality, int sampling = DMC_JPEG_SAMPLING_420)
{
	dmc_dropin::require_color8(src, "degradeJPEGColor");
	const Mat s = src.isContinuous() ? src : src.clone();
	Mat d;
	if (dest.data != src.data && dest.size() == src.size() && dest.type() == CV_8UC3 && dest.isContinuous()) d = dest;
	else d.create(src.size(), CV_8UC3);
	uint64_t bytes = 0;
	dmc_dropin::check(dmc_jpeg_degrade_color_batch(dmc_dropin::context(), s.data, d.data, 1, s.rows, s.cols, quality, sampling, DMC_MEM_HOST, &bytes),
	                  "degradeJPEGColor");
	if (d.data != dest.data) dest = d;
	return (int)bytes;
}

// The JPEG rate-distortion sweep of one CV_8UC1 image on the GPU (the reference's simpleTest, main.cpp:516-526, for several
// qualities at once): for every qualities[k], bytes[k] = the size of cv::imencode(".jpg", src, {IMWRITE_JPEG_QUALITY, q}
// [, IMWRITE_JPEG_OPTIMIZE, 1]), psnr_coded[k] = cv::PSNR(src, the decoded image) and psnr_filtered[k] = cv::PSNR(src,
// PostFilterSet()(decoded, median_r, gaussian_r, minmax_r, brange_r, brange_th)).  Neither stream nor image leaves the device.
inline void jpegRateDistortionGray(const Mat& src, const vector<int>& qualities, vector<int>& bytes, vector<double>& psnr_coded,
                                   vector<double>& psnr_filtered, int median_r, int gaussian_r, int minmax_r, int brange_r, int brange_th,
                                   bool optimize = false)
{
	dmc_dropin::require_gray8(src, "jpegRateDistortionGray");
	const Mat s = src.isContinuous() ? src : src.clone();
	const size_t nq = qualities.size();
	vector<uint64_t> b(nq), sc(nq), sf(nq);
	dmc_chain_params p = {DMC_CHAIN_DISP8U, median_r, gaussian_r, minmax_r, brange_r, (float)brange_th, DMC_FULL_KERNEL, 0, 0, 0};
	dmc_dropin::check(dmc_jpeg_rd_sweep(dmc_dropin::context(), s.data, DMC_MEM_HOST, 1, s.rows, s.cols, qualities.data(), (int)nq,
	                                    optimize ? DMC_JPEG_OPTIMIZE_HUFFMAN : 0, &p, b.data(), sc.data(), sf.data()), "jpegRateDistortionGray");
	const uint64_t pixels = (uint64_t)s.rows * s.cols;
	bytes.resize(nq); psnr_coded.resize(nq); psnr_filtered.resize(nq);
	for (size_t k = 0; k < nq; k++) {
		bytes[k] = (int)b[k];
		psnr_coded[k] = dmc_psnr_from_sse(sc[k], pixels);
		psnr_filtered[k] = dmc_psnr_from_sse(sf[k], pixels);
	}
}

// The view-synthesis rate-distortion sweep of one frame on the GPU (pointcloudTest's view, main.cpp:276-373, for several
// qualities and cameras at once): `disp` (CV_8UC1 disparity) is coded at every qualities[k] (optimize: with optimised Huffman
// tables); bytes[k] is the stream's size.  For every camera v (R[v], t[v]: CV_64F 3x3 and 3x1; K shared), the reference view
// is fillSmallHole(projectImagefromXYZ(texture, reprojectXYZ(disp8U2depth32F(disp, focus*baseline, amp), f), R, t, K, isSub))
// in place, and psnr_coded[k][v] / psnr_filtered[k][v] = cv::PSNR of that view against the same view rendered from the
// decoded disparity (converted the same way) / from filterDisp8U2Depth32F(decoded, focus, baseline, amp, median_r,
// gaussian_r, minmax_r, brange_r, brange_th).  texture: CV_8UC3, the image that is splatted.  Nothing leaves the device.
inline void jpegViewRateDistortionGray(const Mat& disp, const Mat& texture, const vector<int>& qualities, double focus, double baseline, double amp,
                                       int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, double f,
                                       const vector<Mat>& R, const vector<Mat>& t, const Mat& K, bool isSub, vector<int>& bytes,
                                       vector<vector<double> >& psnr_coded, vector<vector<double> >& psnr_filtered, bool optimize = false)
{
	dmc_dropin::require_gray8(disp, "jpegViewRateDistortionGray");
	if (texture.type() != CV_8UC3 || texture.rows != disp.rows || texture.cols != disp.cols) {
#ifdef DMC_MINICV_HPP
		throw cv::Exception("jpegViewRateDistortionGray: texture must be CV_8UC3 of the size of disp", __FILE__, __LINE__);
#else
		CV_Error(cv::Error::StsAssert, "jpegViewRateDistortionGray: texture must be CV_8UC3 of the size of disp");
#endif
	}
	const Mat s = disp.isContinuous() ? disp : disp.clone();
	const Mat tex = texture.isContinuous() ? texture : texture.clone();
	const size_t nq = qualities.size(), nv = R.size() < t.size() ? R.size() : t.size();
	vector<double> r(9 * nv), tt(3 * nv), k(9);
	for (size_t v = 0; v < nv; v++) dmc_dropin::camera(R[v], t[v], K, &r[9 * v], &tt[3 * v], &k[0], "jpegViewRateDistortionGray");
	vector<uint64_t> b(nq), sc(nq * nv), sf(nq * nv);
	dmc_chain_params p = {DMC_CHAIN_DEPTH32F, median_r, gaussian_r, minmax_r, brange_r, brange_th, DMC_FULL_KERNEL, focus, baseline, amp};
	dmc_dropin::check(dmc_jpeg_view_rd_sweep(dmc_dropin::context(), s.data, tex.data, DMC_MEM_HOST, 1, s.rows, s.cols, qualities.data(), (int)nq,
	                                         optimize ? DMC_JPEG_OPTIMIZE_HUFFMAN : 0, &p, f, nv ? &r[0] : 0, nv ? &tt[0] : 0, (int)nv, &k[0], isSub ? 1 : 0, 0,
	                                         b.data(), sc.data(), sf.data()), "jpegViewRateDistortionGray");
	const uint64_t pixels = 3 * (uint64_t)s.rows * s.cols;
	bytes.resize(nq); psnr_coded.assign(nq, vector<double>(nv)); psnr_filtered.assign(nq, vector<double>(nv));
	for (size_t q = 0; q < nq; q++) {
		bytes[q] = (int)b[q];
		for (size_t v = 0; v < nv; v++) {
			psnr_coded[q][v] = dmc_psnr_from_sse(sc[q * nv + v], pixels);
			psnr_filtered[q][v] = dmc_psnr_from_sse(sf[q * nv + v], pixels);
		}
	}
}

// The two sweeps above with a third arm, the boundary reconstruction filter: psnr_brf[k] = cv::PSNR(src,
// boundaryReconstructionFilter(decoded, brf_ksize, frec, color, space)), the filter the reference keeps on the decoded
// disparity but comments out (main.cpp:306-311).  Scoring it there, next to the post filter set, is this library's definition.
inline void jpegRateDistortionGray(const Mat& src, const vector<int>& qualities, vector<int>& bytes, vector<double>& psnr_coded,
                                   vector<double>& psnr_filtered, int median_r, int gaussian_r, int minmax_r, int brange_r, int brange_th,
                                   Size brf_ksize, float frec, float color, float space, vector<double>& psnr_brf, bool optimize = false)
{
	dmc_dropin::require_gray8(src, "jpegRateDistortionGray");
	const Mat s = src.isContinuous() ? src : src.clone();
	const size_t nq = qualities.size();
	vector<uint64_t> b(nq), sc(nq), sf(nq), sb(nq);
	dmc_chain_params p = {DMC_CHAIN_DISP8U, median_r, gaussian_r, minmax_r, brange_r, (float)brange_th, DMC_FULL_KERNEL, 0, 0, 0};
	dmc_brf_params bp = {brf_ksize.width, brf_ksize.height, frec, color, space};
	dmc_dropin::check(dmc_jpeg_rd_sweep_ex(dmc_dropin::context(), s.data, DMC_MEM_HOST, 1, s.rows, s.cols, qualities.data(), (int)nq,
	                                       optimize ? DMC_JPEG_OPTIMIZE_HUFFMAN : 0, &p, &bp, b.data(), sc.data(), sf.data(), sb.data()), "jpegRateDistortionGray");
	const uint64_t pixels = (uint64_t)s.rows * s.cols;
	bytes.resize(nq); psnr_coded.resize(nq); psnr_filtered.resize(nq); psnr_brf.resize(nq);
	for (size_t k = 0; k < nq; k++) {
		bytes[k] = (int)b[k];
		psnr_coded[k] = dmc_psnr_from_sse(sc[k], pixels);
		psnr_filtered[k] = dmc_psnr_from_sse(sf[k], pixels);
		psnr_brf[k] = dmc_psnr_from_sse(sb[k], pixels);
	}
}

// psnr_brf[k][v] = cv::PSNR of the reference view against the view rendered from
// disp8U2depth32F(boundaryReconstructionFilter(decoded, brf_ksize, frec, color, space), focus*baseline, amp).
inline void jpegViewRateDistortionGray(const Mat& disp, const Mat& texture, const vector<int>& qualities, double focus, double baseline, double amp,
                                       int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, double f,
                                       const vector<Mat>& R, const vector<Mat>& t, const Mat& K, bool isSub, vector<int>& bytes,
                                       vector<vector<double> >& psnr_coded, vector<vector<double> >& psnr_filtered,
                                       Size brf_ksize, float frec, float color, float space, vector<vector<double> >& psnr_brf, bool optimize = false)
{
	dmc_dropin::require_gray8(disp, "jpegViewRateDistortionGray");
	if (texture.type() != CV_8UC3 || texture.rows != disp.rows || texture.cols != disp.cols) {
#ifdef DMC_MINICV_HPP
		throw cv::Exception("jpegViewRateDistortionGray: texture must be CV_8UC3 of the size of disp", __FILE__, __LINE__);
#else
		CV_Error(cv::Error::StsAssert, "jpegViewRateDistortionGray: texture must be CV_8UC3 of the size of disp");
#endif
	}
	const Mat s = disp.isContinuous() ? disp : disp.clone();
	const Mat tex = texture.isContinuous() ? texture : texture.clone();
	const size_t nq = qualities.size(), nv = R.size() < t.size() ? R.size() : t.size();
	vector<double> r(9 * nv), tt(3 * nv), k(9);
	for (size_t v = 0; v < nv; v++) dmc_dropin::camera(R[v], t[v], K, &r[9 * v], &tt[3 * v], &k[0], "jpegViewRateDistortionGray");
	vector<uint64_t> b(nq), sc(nq * nv), sf(nq * nv), sb(nq * nv);
	dmc_chain_params p = {DMC_CHAIN_DEPTH32F, median_r, gaussian_r, minmax_r, brange_r, brange_th, DMC_FULL_KERNEL, focus, baseline, amp};
	dmc_brf_params bp = {brf_ksize.width, brf_ksize.height, frec, color, space};
	dmc_dropin::check(dmc_jpeg_view_rd_sweep_ex(dmc_dropin::context(), s.data, tex.data, DMC_MEM_HOST, 1, s.rows, s.cols, qualities.data(), (int)nq,
	                                            optimize ? DMC_JPEG_OPTIMIZE_HUFFMAN : 0, &p, &bp, f, nv ? &r[0] : 0, nv ? &tt[0] : 0, (int)nv, &k[0], isSub ? 1 : 0, 0,
	                                            b.data(), sc.data(), sf.data(), sb.data()), "jpegViewRateDistortionGray");
	const uint64_t pixels = 3 * (uint64_t)s.rows * s.cols;
	bytes.resize(nq); psnr_coded.assign(nq, vector<double>(nv)); psnr_filtered.assign(nq, vector<double>(nv)); psnr_brf.assign(nq, vector<double>(nv));
	for (size_t q = 0; q < nq; q++) {
		bytes[q] = (int)b[q];
		for (size_t v = 0; v < nv; v++) {
			psnr_coded[q][v] = dmc_psnr_from_sse(sc[q * nv + v], pixels);
			psnr_filtered[q][v] = dmc_psnr_from_sse(sf[q * nv + v], pixels);
			psnr_brf[q][v] = dmc_psnr_from_sse(sb[q * nv + v], pixels);
		}
	}
}

namespace dmc_dropin {
inline void require(bool ok, const char* what) {
	if (ok) return;
#ifdef DMC_MINICV_HPP
	throw cv::Exception(what, __FILE__, __LINE__);
#else
	CV_Error(cv::Error::StsAssert, what);
#endif
}
// frames of one size and type, packed back to back (row by row: any row step)
inline vector<uchar> pack(const vector<Mat>& frames, int type, const char* what) {
	const Mat& f0 = frames[0];
	const size_t row = (size_t)f0.cols * f0.elemSize();
	vector<uchar> out(row * f0.rows * frames.size());
	for (size_t i = 0; i < frames.size(); i++) {
		require(frames[i].type() == type && frames[i].rows == f0.rows && frames[i].cols == f0.cols, what);
		for (int y = 0; y < f0.rows; y++) memcpy(&out[(i * f0.rows + y) * row], frames[i].ptr(y), row);
	}
	return out;
}
}  // namespace dmc_dropin

// pointcloudTest's preparation of sensor depth (main.cpp:254-260) on a batch: disp8[i] = fillOcclusion(depth16U2disp8U(
// depth16[i], focal_baseline, a, b), 0, FILL_DISPARITY), and with passes = 2 that filled again around a transpose (passes = 1
// is simpleTest's call, main.cpp:511-512).  depth16: CV_16UC1 frames of one size.  Bit-identical to those calls frame by frame.
inline void prepareDisparityBatch(const vector<Mat>& depth16, vector<Mat>& disp8, float focal_baseline, float a = 1.f, float b = 0.f, int passes = 2)
{
	disp8.clear();
	if (depth16.empty()) return;
	const int n = (int)depth16.size(), rows = depth16[0].rows, cols = depth16[0].cols;
	const vector<uchar> src = dmc_dropin::pack(depth16, CV_16UC1, "prepareDisparityBatch: depth16 must be CV_16UC1 frames of one size");
	vector<uchar> dst((size_t)n * rows * cols);
	dmc_dropin::check(dmc_prepare_disp_batch(dmc_dropin::context(), src.data(), dst.data(), n, rows, cols, focal_baseline, a, b, passes, DMC_MEM_HOST),
	                  "prepareDisparityBatch");
	disp8.resize(n);
	for (int i = 0; i < n; i++) {
		disp8[i].create(rows, cols, CV_8UC1);
		memcpy(disp8[i].data, &dst[(size_t)i * rows * cols], (size_t)rows * cols);
	}
}

// pointcloudTest's views (main.cpp:321-355) of a batch: views[v][i] = fillSmallHole(projectImagefromXYZ(texture[i],
// reprojectXYZ(depth[i], f), R[v], t[v], K, isSub)), the fill in place.  depth: frames of one size and one of the types
// reprojectXYZ takes (CV_8U, CV_16S, CV_16U, CV_32F: filterDisp8U2Depth32F's output as it is); texture: CV_8UC3 of that size.
inline void renderViewBatch(const vector<Mat>& depth, const vector<Mat>& texture, double f, const vector<Mat>& R, const vector<Mat>& t, const Mat& K,
                            bool isSub, vector<vector<Mat> >& views)
{
	views.clear();
	dmc_dropin::require(!R.empty() && R.size() == t.size(), "renderViewBatch: R and t must hold one camera each");
	dmc_dropin::require(depth.size() == texture.size(), "renderViewBatch: one texture per depth frame");
	const size_t nv = R.size();
	vector<double> r(9 * nv), tt(3 * nv), k(9);
	for (size_t v = 0; v < nv; v++) dmc_dropin::camera(R[v], t[v], K, &r[9 * v], &tt[3 * v], &k[0], "renderViewBatch");
	views.assign(nv, vector<Mat>());
	if (depth.empty()) return;
	const int n = (int)depth.size(), rows = depth[0].rows, cols = depth[0].cols, type = depth[0].type();
	const vector<uchar> d = dmc_dropin::pack(depth, type, "renderViewBatch: depth frames must share one size and type");
	const vector<uchar> tex = dmc_dropin::pack(texture, CV_8UC3, "renderViewBatch: texture must be CV_8UC3 frames of the depth's size");
	dmc_dropin::require(texture[0].rows == rows && texture[0].cols == cols, "renderViewBatch: texture must be CV_8UC3 frames of the depth's size");
	const size_t vb = (size_t)rows * cols * 3;
	vector<uchar> out(vb * n * nv);
	dmc_dropin::check(dmc_render_view_batch(dmc_dropin::context(), d.data(), type, tex.data(), DMC_MEM_HOST, n, rows, cols, f, &r[0], &tt[0], (int)nv, &k[0],
	                                        isSub ? 1 : 0, 0, out.data()), "renderViewBatch");
	for (size_t v = 0; v < nv; v++) {
		views[v].resize(n);
		for (int i = 0; i < n; i++) {
			views[v][i].create(rows, cols, CV_8UC3);
			memcpy(views[v][i].data, &out[(v * n + i) * vb], vb);
		}
	}
}

// Mean structural similarity (SSIM, Wang et al. 2004) of two CV_8UC1 or CV_8UC3 images of one size and type in host memory,
// on the GPU (dmc_ssim_batch): 11x11 Gaussian window with sigma 1.5, only window positions inside the image, C1 = (0.01*255)^2,
// C2 = (0.03*255)^2, FP64; for CV_8UC3 the mean of the three channels' values.  Both sides at least 11 x 11.
inline double structuralSimilarity(const Mat& a, const Mat& b)
{
	const int type = a.type();
	dmc_dropin::require((type == CV_8UC1 || type == CV_8UC3) && b.type() == type && a.rows == b.rows && a.cols == b.cols,
	                    "structuralSimilarity: a and b must be CV_8UC1 or CV_8UC3 images of one size and type");
	const Mat x = a.isContinuous() ? a : a.clone();
	const Mat y = b.isContinuous() ? b : b.clone();
	double mssim = 0;
	dmc_dropin::check(dmc_ssim_batch(dmc_dropin::context(), x.data, y.data, 1, x.rows, x.cols, type == CV_8UC3 ? 3 : 1, DMC_MEM_HOST, &mssim),
	                  "structuralSimilarity");
	return mssim;
}

// Baseline colour JPEG decoding on the GPU: dst = cv::imdecode(buf, IMREAD_COLOR), a CV_8UC3 BGR image, bit for bit
// (libjpeg-turbo's islow IDCT, fancy upsampling and colour conversion; one-component streams give B = G = R = Y).  Streams
// the decoder does not take (progressive, arithmetic, 12-bit, CMYK, RGB-coded, ...) throw with the reason.
inline void jpegDecodeColor(const vector<uchar>& buf, Mat& dst)
{
	int rows = 0, cols = 0, nc = 0;
	char why[256] = {0};
	if (dmc_jpeg_probe_color(buf.empty() ? 0 : buf.data(), buf.size(), &rows, &cols, &nc, why, sizeof why) != DMC_OK)
		dmc_dropin::require(false, (std::string("jpegDecodeColor: ") + why).c_str());
	dst.create(rows, cols, CV_8UC3);
	Mat out = dst.isContinuous() ? dst : Mat(rows, cols, CV_8UC3);
	const uint64_t off[2] = {0, (uint64_t)buf.size()};
	dmc_dropin::check(dmc_jpeg_decode_color_batch(dmc_dropin::context(), buf.data(), off, 1, rows, cols, out.data, DMC_MEM_HOST), "jpegDecodeColor");
	if (out.data != dst.data) out.copyTo(dst);
}
