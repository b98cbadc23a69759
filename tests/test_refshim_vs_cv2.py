"""Pins the third-party OpenCV stages.  The reference calls cv::medianBlur / GaussianBlur / dilate / erode /
copyMakeBorder / convertTo (no OpenCV version pinned, none vendored); both checkers restate them.  Here the
restatements (oracle/refshim/minicv.hpp and oracle/dmc_oracle.c) are compared with the real OpenCV in this
image (cv2 4.13.0), which SURVEY.md 8c names as the oracle of record for those calls."""
import numpy as np
import pytest

from _util import assert_bits_equal, make_image

cv2 = pytest.importorskip("cv2")
SHAPES = [(37, 53), (1, 7), (7, 1), (2, 2), (64, 48), (83, 131)]


@pytest.mark.parametrize("shape", SHAPES)
def test_median(port, shim, shape):
    rs = np.random.RandomState(11); H, W = shape
    for kind in ("pw", "noise"):
        a = make_image(rs, H, W, kind=kind)
        for k in (1, 3, 5, 7, 9, 13, 21):
            want = cv2.medianBlur(a, k) if k > 1 else a
            assert_bits_equal(port.median_blur(a, k), want, "port median k%d" % k)
            assert_bits_equal(shim.median_blur(a, k), want, "shim median k%d" % k)


@pytest.mark.parametrize("shape", SHAPES)
def test_morphology(port, shim, shape):
    rs = np.random.RandomState(12); H, W = shape
    for dt in (np.uint8, np.uint16, np.int16, np.float32):
        a = make_image(rs, H, W, dt)
        for k in (1, 3, 7, 11, 21):
            el = np.ones((k, k), np.uint8)
            for is_max, fn in ((True, cv2.dilate), (False, cv2.erode)):
                want = fn(a, el)
                assert_bits_equal(port.morph(a, k, is_max), want, "port morph")
                assert_bits_equal(shim.morph(a, k, is_max), want, "shim morph")


def test_gaussian_kernel_taps(port, shim):
    for gr in range(0, 11):
        n = 2 * gr + 1
        want = cv2.getGaussianKernel(n, gr + 0.5, cv2.CV_32F).ravel()
        assert_bits_equal(port.gaussian_kernel32f(n, gr + 0.5), want, "port taps gr%d" % gr)
        assert_bits_equal(shim.gaussian_kernel32f(n, gr + 0.5), want, "shim taps gr%d" % gr)
        for sigma in (0.0, -1.5):          # sigma <= 0: OpenCV's fixed small kernels (n <= 9), else the size-derived sigma
            want = cv2.getGaussianKernel(n, sigma, cv2.CV_32F).ravel()
            assert_bits_equal(port.gaussian_kernel32f(n, sigma), want, "port taps gr%d sigma %g" % (gr, sigma))
            assert_bits_equal(shim.gaussian_kernel32f(n, sigma), want, "shim taps gr%d sigma %g" % (gr, sigma))


def test_small_gaussian_nonpositive_sigma(port, ref):
    """smallGaussianBlur(src, dst, d, sigma <= 0): cv::GaussianBlur then uses getGaussianKernel's fixed taps (ADVICE r01)."""
    rs = np.random.RandomState(21)
    a = make_image(rs, 61, 83, kind="noise")
    for d in (1, 3, 5, 7, 9, 11, 13):
        cv2.setUseOptimized(False)
        try:
            f = cv2.GaussianBlur(a.astype(np.float32), (d, d), 0)
        finally:
            cv2.setUseOptimized(True)
        want8 = np.clip(np.rint(f), 0, 255).astype(np.uint8)
        assert_bits_equal(port.small_gaussian(a, d, 0.0), want8, "port smallGaussian d%d sigma 0" % d)
        assert_bits_equal(ref.small_gaussian(a, d, 0.0), want8, "shim smallGaussian d%d sigma 0" % d)


@pytest.mark.parametrize("shape", SHAPES)
def test_small_gaussian_8u_roundtrip(port, ref, shape):
    """smallGaussianBlur = 8U -> 32F -> GaussianBlur -> 8U (postFilterSet.cpp:4-16).  In FP32 the result is
    pinned to OpenCV's scalar op order (cv2.setUseOptimized(False)); cv2's default SIMD/FMA build may differ
    by <=1 ulp in float -- after the 8U rounding both must give the same bytes."""
    rs = np.random.RandomState(13); H, W = shape
    for kind in ("pw", "noise"):
        a = make_image(rs, H, W, kind=kind)
        for gr in (0, 1, 2, 3, 4, 5):
            d = 2 * gr + 1
            cv2.setUseOptimized(False)
            try:
                f = cv2.GaussianBlur(a.astype(np.float32), (d, d), gr + 0.5)
            finally:
                cv2.setUseOptimized(True)
            assert_bits_equal(port.gaussian_blur32f(a.astype(np.float32), d, gr + 0.5), f, "port gauss32f gr%d" % gr)
            assert_bits_equal(ref.gaussian_blur32f(a.astype(np.float32), d, gr + 0.5), f, "shim gauss32f gr%d" % gr)
            f_opt = cv2.GaussianBlur(a.astype(np.float32), (d, d), gr + 0.5)
            want8 = np.clip(np.rint(f_opt), 0, 255).astype(np.uint8)     # rint = round-half-even = cvRound
            assert_bits_equal(port.small_gaussian(a, d, gr + 0.5), want8, "port smallGaussian gr%d" % gr)
            assert_bits_equal(ref.small_gaussian(a, d, gr + 0.5), want8, "shim smallGaussian gr%d" % gr)


def test_copy_make_border(shim):
    rs = np.random.RandomState(14)
    for (H, W) in [(5, 7), (1, 3), (3, 1), (2, 2), (9, 4)]:
        for dt, cn in [(np.uint8, 1), (np.uint8, 3), (np.float32, 1), (np.uint16, 1)]:
            a = make_image(rs, H, W, dt, cn, kind="noise")
            for (t, b, l, r) in [(0, 0, 0, 0), (1, 1, 1, 1), (3, 2, 5, 21), (6, 6, 6, 6)]:
                for border in (cv2.BORDER_REPLICATE, cv2.BORDER_REFLECT_101):
                    assert_bits_equal(shim.copy_make_border(a, t, b, l, r, border), cv2.copyMakeBorder(a, t, b, l, r, border), "copyMakeBorder")


def test_convert_to(shim):
    f = np.array([[0.5, 1.5, 2.5, -0.5, -1.5, 254.5, 255.5, 256.0, 65535.4, 65535.5, 70000.0, -3.0,
                   np.inf, -np.inf, np.nan, 3e9, -3e9, 32767.5, -32768.5, 1e-3]], np.float32)
    for ddt, cvt in ((np.uint8, cv2.CV_8U), (np.uint16, cv2.CV_16U), (np.int16, cv2.CV_16S)):
        assert_bits_equal(shim.convert_to(f, ddt), _convert_cv2(f, cvt), "convertTo %s" % ddt.__name__)
    for sdt in (np.uint8, np.uint16, np.int16):
        a = np.arange(0, 4000, 7).reshape(1, -1).astype(sdt)
        assert_bits_equal(shim.convert_to(a, np.float32), a.astype(np.float32), "to float")


def _convert_cv2(f, cvt):
    # cv2 has no direct Mat::convertTo binding; cv2.add(src, 0, dtype=...) performs the same saturating cast path
    return cv2.add(f, np.zeros_like(f), dtype=cvt)
