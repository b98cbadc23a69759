"""The C++ drop-in (include/filter.h + include/util.h over the C ABI): the reference's own call sites
(main.cpp:303, :308, :485, :495, :526) compiled against our headers."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "tests", "cpp")


def _build(out_dir):
    """Builds the drop-in program into out_dir: the source tree may be read-only."""
    import __graft_entry__ as g
    g.build()
    exe = str(out_dir / "test_dropin")
    subprocess.check_call(["make", "-C", CPP, "OUT=" + exe], stdout=subprocess.DEVNULL)
    return exe


def test_dropin_headers_compile_and_link(tmp_path):
    """CPU-side: the reference's declarations compile against our headers and link against libdmc_b200.so."""
    exe = _build(tmp_path)
    assert os.path.exists(exe)
    hdr = open(os.path.join(ROOT, "include", "filter.h")).read()
    ref_decls = [   # PostFilterSetForDepthCoding/filter.h:12-45, verbatim
        "void splitBGRLineInterleave( const Mat& src, Mat& dest);",
        "void smallGaussianBlur(const Mat& src, Mat& dest, const int d, const double sigma);",
        "void maxFilter(const Mat& src, Mat& dest, Size ksize, int borderType=cv::BORDER_REPLICATE);",
        "void minFilter(const Mat& src, Mat& dest, Size ksize, int borderType=cv::BORDER_REPLICATE);",
        "void blurRemoveMinMax(Mat& src, Mat& dest, const int r);",
        "void blurRemoveMinMaxBase(Mat& src, Mat& dest, const int r);",
        "void binalyWeightedRangeFilter(const Mat& src, Mat& dst, Size kernelSize, float threshold, int method, int borderType=cv::BORDER_REPLICATE);",
        "void filterDisp8U2Depth32F(Mat& src, Mat& dest, double focus, double baseline, double amp, int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, int brange_method=FULL_KERNEL);",
        "void filterDisp8U2Depth16U(Mat& src, Mat& dest, double focus, double baseline, double amp, int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, int brange_method=FULL_KERNEL);",
        "void filterDisp8U2Disp32F(Mat& src, Mat& dest, int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, int brange_method=FULL_KERNEL);",
        "void operator()(Mat& src, Mat& dest, int median_r, int gaussian_r, int minmax_r, int brange_r, int brange_th, int brange_method=FULL_KERNEL);",
        "void boundaryReconstructionFilter(Mat& src, Mat& dest, Size ksize, const float frec, const float color, const float space);",
    ]
    for d in ref_decls:
        assert d in hdr, d
    util = open(os.path.join(ROOT, "include", "util.h")).read()
    util_decls = [  # PostFilterSetForDepthCoding/util.h:11-13, :24-28, :33, verbatim
        "void reprojectXYZ(const Mat& depth, Mat& xyz, double f);",
        "void projectImagefromXYZ(const Mat& image, Mat& destimage, const Mat& xyz, const Mat& R, const Mat& t, const Mat& K, const Mat& dist, Mat& mask, const bool isSub);",
        "void projectImagefromXYZ(const Mat& image, Mat& destimage, const Mat& xyz, const Mat& R, const Mat& t, const Mat& K, const Mat& dist, Mat& mask, const bool isSub, vector<Point2f>& pt, Mat& depth);",
        "void fillOcclusion(Mat& src, int invalidvalue, int disp_or_depth=FILL_DEPTH);",
        "void fillSmallHole(const Mat& src, Mat& dest);",
        "void depth32F2disp8U(Mat& src, Mat& dest, const float focal_baseline, float a=1.f, float b=0.f);",
        "void disp16S2depth16U(Mat& src, Mat& dest, const float focal_baseline, float a=1.f, float b=0.f);",
        "void depth16U2disp8U(Mat& src, Mat& dest, const float focal_baseline, float a=1.f, float b=0.f);",
        "void disp8U2depth32F(Mat& src, Mat& dest, const float focal_baseline, float a=1.f, float b=0.f);",
        "void projectPointsSimple(const Mat& xyz, const Mat& R, const Mat& t, const Mat& K, vector<Point2f>& dest);//multi points projection",
    ]
    for d in util_decls:
        assert d in util, d


@pytest.mark.gpu
def test_dropin_call_sites_bit_exact(tmp_path):
    exe = _build(tmp_path)
    res = subprocess.run([exe, os.path.join(ROOT, "oracle", "libdmc_oracle.so")], capture_output=True, text=True, cwd=ROOT, timeout=600)
    print(res.stdout[-3000:], res.stderr[-2000:])
    assert res.returncode == 0 and "ALL OK" in res.stdout
