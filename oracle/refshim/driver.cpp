// driver.cpp -- TEST INFRASTRUCTURE ONLY.
// extern "C" entry points around the UNMODIFIED reference translation units
// (/root/reference/PostFilterSetForDepthCoding/*.cpp, compiled against minicv.hpp by
// oracle/Makefile into oracle/_ref/libdmc_ref.so).  Every wrapper copies the caller's
// buffer into a 64-byte aligned, continuous Mat (the reference uses aligned SSE
// loads/stores on Mat data), calls the reference function, and copies the result out.
// Used only by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs.
// Built with -DDMC_SHIM_ONLY (oracle/libdmc_shim.so) it holds only the shim_* entry points, which need no
// reference source, so that the stand-ins can be pinned against cv2 without the reference tree.
#ifdef DMC_SHIM_ONLY
#include "minicv.hpp"
using namespace cv;
#else
#include "filter.h"
#include "util.h"

void binalyWeightedRangeFilter(const Mat& src, Mat& dst, int kernelSize, float threshold, int method, int borderType);
#endif

namespace {
Mat wrapCopy(const void* p, int rows, int cols, int type) {
    Mat m(rows, cols, type);
    memcpy(m.data, p, m.step * (size_t)rows);
    return m;
}
void copyOut(const Mat& m, void* p) { for (int y = 0; y < m.rows; y++) memcpy((uchar*)p + (size_t)y * m.cols * m.elemSize(), m.ptr(y), (size_t)m.cols * m.elemSize()); }
}  // namespace

#define DMC_TRY try {
#define DMC_CATCH } catch (const std::exception& e) { fprintf(stderr, "[dmc_ref] %s\n", e.what()); return -1; } return 0;

extern "C" {

#ifndef DMC_SHIM_ONLY
int ref_version() { return 1; }
void ref_set_num_threads(int n) {
#ifdef _OPENMP
    omp_set_num_threads(n > 0 ? n : omp_get_num_procs());
#endif
}
int ref_get_num_threads() { return cv::getNumThreads(); }

// PostFilterSet::operator()  (postFilterSet.cpp:57-63)
int ref_post_filter_set(const uchar* src, uchar* dst, int rows, int cols, int median_r, int gaussian_r, int minmax_r, int brange_r, int brange_th, int method) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_8U), d;
    PostFilterSet pfs; pfs(s, d, median_r, gaussian_r, minmax_r, brange_r, brange_th, method);
    if (d.empty()) return 1;
    copyOut(d, dst);
    DMC_CATCH
}
// PostFilterSet::filterDisp8U2Depth32F (postFilterSet.cpp:34-43)
int ref_filter_disp8u_depth32f(const uchar* src, float* dst, int rows, int cols, double focus, double baseline, double amp, int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, int method) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_8U), d;
    PostFilterSet pfs; pfs.filterDisp8U2Depth32F(s, d, focus, baseline, amp, median_r, gaussian_r, minmax_r, brange_r, brange_th, method);
    if (d.empty()) return 1;
    copyOut(d, dst);
    DMC_CATCH
}
// PostFilterSet::filterDisp8U2Depth16U (postFilterSet.cpp:21-32)
int ref_filter_disp8u_depth16u(const uchar* src, ushort* dst, int rows, int cols, double focus, double baseline, double amp, int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, int method) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_8U), d;
    PostFilterSet pfs; pfs.filterDisp8U2Depth16U(s, d, focus, baseline, amp, median_r, gaussian_r, minmax_r, brange_r, brange_th, method);
    if (d.empty()) return 1;
    copyOut(d, dst);
    DMC_CATCH
}
// PostFilterSet::filterDisp8U2Disp32F (postFilterSet.cpp:45-55) -- output is 16U despite the name
int ref_filter_disp8u_disp32f(const uchar* src, ushort* dst, int rows, int cols, int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, int method) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_8U), d;
    PostFilterSet pfs; pfs.filterDisp8U2Disp32F(s, d, median_r, gaussian_r, minmax_r, brange_r, brange_th, method);
    if (d.empty()) return 1;
    copyOut(d, dst);
    DMC_CATCH
}
// binalyWeightedRangeFilter (binalyWeightedRangeFilter.cpp:1106). dst is pre-filled with the caller's bytes so
// that the reference's silent no-op (type, method) pairs leave it untouched, as they would the caller's Mat.
int ref_bwrf(const void* src, void* dst, int rows, int cols, int cvtype, int kw, int kh, float th, int method, int inplace) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype);
    if (inplace) { binalyWeightedRangeFilter(s, s, Size(kw, kh), th, method); copyOut(s, dst); }
    else { Mat d = wrapCopy(dst, rows, cols, cvtype); binalyWeightedRangeFilter(s, d, Size(kw, kh), th, method); copyOut(d, dst); }
    DMC_CATCH
}
// blurRemoveMinMax (minmaxFilter.cpp:176)
int ref_blur_remove_minmax(const void* src, void* dst, int rows, int cols, int cvtype, int r, int inplace) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype);
    if (inplace) { blurRemoveMinMax(s, s, r); copyOut(s, dst); }
    else { Mat d; blurRemoveMinMax(s, d, r); copyOut(d, dst); }
    DMC_CATCH
}
int ref_blur_remove_minmax_base(const void* src, void* dst, int rows, int cols, int cvtype, int r) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype), d; blurRemoveMinMaxBase(s, d, r); copyOut(d, dst);
    DMC_CATCH
}
// maxFilter / minFilter (minmaxFilter.cpp:314, :394)
int ref_max_filter(const void* src, void* dst, int rows, int cols, int cvtype, int kw, int kh) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype), d; maxFilter(s, d, Size(kw, kh)); if (d.empty()) return 1; copyOut(d, dst);
    DMC_CATCH
}
int ref_min_filter(const void* src, void* dst, int rows, int cols, int cvtype, int kw, int kh) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype), d; minFilter(s, d, Size(kw, kh)); if (d.empty()) return 1; copyOut(d, dst);
    DMC_CATCH
}
// boundaryReconstructionFilter (boundaryReconstructionFilter.cpp:133)
int ref_brf(const void* src, void* dst, int rows, int cols, int cvtype, int kw, int kh, float frec, float color, float space, int inplace) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype);
    if (inplace) { boundaryReconstructionFilter(s, s, Size(kw, kh), frec, color, space); copyOut(s, dst); }
    else { Mat d; boundaryReconstructionFilter(s, d, Size(kw, kh), frec, color, space); if (d.empty()) return 1; copyOut(d, dst); }
    DMC_CATCH
}
// smallGaussianBlur (postFilterSet.cpp:4-16)
int ref_small_gaussian(const void* src, void* dst, int rows, int cols, int cvtype, int d, double sigma) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype), o; smallGaussianBlur(s, o, d, sigma); copyOut(o, dst);
    DMC_CATCH
}
// converters (depthmapUtil.cpp:685, :768, :840, :923)
int ref_disp16s2depth16u(const short* src, ushort* dst, int rows, int cols, float fb, float a, float b) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_16S), d; disp16S2depth16U(s, d, fb, a, b); copyOut(d, dst);
    DMC_CATCH
}
int ref_depth32f2disp8u(const float* src, uchar* dst, int rows, int cols, float fb, float a, float b) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_32F), d; depth32F2disp8U(s, d, fb, a, b); copyOut(d, dst);
    DMC_CATCH
}
int ref_depth16u2disp8u(const ushort* src, uchar* dst, int rows, int cols, float fb, float a, float b) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_16U), d; depth16U2disp8U(s, d, fb, a, b); copyOut(d, dst);
    DMC_CATCH
}
int ref_disp8u2depth32f(const uchar* src, float* dst, int rows, int cols, float fb, float a, float b) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_8U), d = wrapCopy(dst, rows, cols, CV_32F);   // b!=0 leaves part of dest untouched
    disp8U2depth32F(s, d, fb, a, b); copyOut(d, dst);
    DMC_CATCH
}
// fillOcclusion (depthmapUtil.cpp:643), in place
int ref_fill_occlusion(void* data, int rows, int cols, int cvtype, int invalid, int mode) {
    DMC_TRY
    Mat s = wrapCopy(data, rows, cols, cvtype); fillOcclusion(s, invalid, mode); copyOut(s, data);
    DMC_CATCH
}
// reprojectXYZ(depth, xyz, f) (depthmapUtil.cpp:483)
int ref_reproject_xyz(const void* depth, float* xyz, int rows, int cols, int cvtype, double f) {
    DMC_TRY
    Mat s = wrapCopy(depth, rows, cols, cvtype), d; reprojectXYZ(s, d, f); if (d.empty()) return 1;
    memcpy(xyz, d.data, (size_t)rows * cols * 3 * sizeof(float));
    DMC_CATCH
}

// point-cloud render: projectPointsSimple (depthmapUtil.cpp:148), projectImagefromXYZ (:285), fillSmallHole (:187)
int ref_project_points(const float* xyz, int n, const double* R9, const double* t3, const double* K9, float* pt) {
    DMC_TRY
    Mat x = wrapCopy(xyz, n, 1, CV_32FC3), R = wrapCopy(R9, 3, 3, CV_64F), t = wrapCopy(t3, 3, 1, CV_64F), K = wrapCopy(K9, 3, 3, CV_64F);
    std::vector<Point2f> dst(n + 4);
    projectPointsSimple(x, R, t, K, dst);
    memcpy(pt, dst.data(), sizeof(float) * 2 * (size_t)n);
    DMC_CATCH
}
int ref_project_image_from_xyz(const uchar* image, const float* xyz, int rows, int cols, const double* R9, const double* t3, const double* K9, int is_sub, uchar* dest, float* depth) {
    DMC_TRY
    Mat im = wrapCopy(image, rows, cols, CV_8UC3), x = wrapCopy(xyz, rows * cols, 1, CV_32FC3);
    Mat R = wrapCopy(R9, 3, 3, CV_64F), t = wrapCopy(t3, 3, 1, CV_64F), K = wrapCopy(K9, 3, 3, CV_64F), d, none1, none2;
    std::vector<Point2f> pt((size_t)rows * cols + 4);
    Mat z(rows, cols, CV_32F);
    projectImagefromXYZ(im, d, x, R, t, K, none1, none2, is_sub != 0, pt, z);
    copyOut(d, dest);
    if (depth) copyOut(z, depth);
    DMC_CATCH
}
int ref_fill_small_hole(const uchar* src, uchar* dst, int rows, int cols, int inplace) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_8UC3), d = inplace ? s : wrapCopy(dst, rows, cols, CV_8UC3);
    fillSmallHole(s, d);
    copyOut(d, dst);
    DMC_CATCH
}
#endif  // DMC_SHIM_ONLY

// ---- the shim's own stand-ins, exported so tests can pin them against cv2 4.13 ----
int shim_median_blur(const void* src, void* dst, int rows, int cols, int cvtype, int ksize) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype), d; cv::medianBlur(s, d, ksize); copyOut(d, dst);
    DMC_CATCH
}
int shim_gaussian_blur32f(const float* src, float* dst, int rows, int cols, int d, double sigma) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, CV_32F), o; cv::GaussianBlur(s, o, Size(d, d), sigma); copyOut(o, dst);
    DMC_CATCH
}
int shim_morph(const void* src, void* dst, int rows, int cols, int cvtype, int k, int is_max) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype), d, el = Mat::ones(k, k, CV_8U);
    if (is_max) cv::dilate(s, d, el); else cv::erode(s, d, el);
    copyOut(d, dst);
    DMC_CATCH
}
int shim_copy_make_border(const void* src, void* dst, int rows, int cols, int cvtype, int top, int bottom, int left, int right, int border) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, cvtype), d; cv::copyMakeBorder(s, d, top, bottom, left, right, border); copyOut(d, dst);
    DMC_CATCH
}
int shim_convert_to(const void* src, void* dst, int rows, int cols, int stype, int dtype) {
    DMC_TRY
    Mat s = wrapCopy(src, rows, cols, stype), d; s.convertTo(d, dtype); copyOut(d, dst);
    DMC_CATCH
}
int shim_gaussian_kernel32f(int n, double sigma, float* out) {
    std::vector<float> k = cv::getGaussianKernel32f(n, sigma); memcpy(out, k.data(), n * sizeof(float)); return 0;
}

}  // extern "C"
