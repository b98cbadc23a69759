"""Float dilate / erode on IEEE special values, without a GPU.

blurRemoveMinMax is cv::dilate and cv::erode followed by a select.  On ordered values any visiting order gives the same
bits, and there cv2, the shim (oracle/refshim/minicv.hpp) and the port (oracle/dmc_oracle.c) must agree.  With NaN, or
with +0 and -0 in one window, the result depends on the order; cv2 4.13 has no fixed rule there (it depends on where a
tap falls in a SIMD lane), so the shim's rule is the contract: each pass starts at the window's centre and folds the
in-image taps in order with std::max / std::min.  A numpy restatement of that rule pins the port to it here, and the GPU
tests of tests/test_gpu_type_matrix.py compare the kernels with the port on the same kind of images."""
import numpy as np
import pytest

from _util import assert_bits_equal, special_image

cv2 = pytest.importorskip("cv2")
SHAPES = [(37, 53), (1, 7), (7, 1), (2, 2), (64, 48), (83, 131)]
KS = list(range(1, 22, 2))


def shim_morph(a, k, is_max, centre_first=True):
    """minicv.hpp morph_: per pass m = centre value, then for every in-image tap i in increasing order
    m = std::max(m, v) = (m < v) ? v : m   (std::min(m, v) = (v < m) ? v : m); rows first, then columns.
    centre_first=False starts at the window's first in-image tap instead (the order the tests must tell apart)."""
    r = k // 2

    def fold(x, axis):
        n = x.shape[axis]
        lo = np.clip(np.arange(n) - r, 0, n - 1)
        m = x.copy() if centre_first else np.take(x, lo, axis=axis)
        for d in range(-r, r + 1):
            idx = np.arange(n) + d
            inside = ((idx >= 0) & (idx < n)).reshape([-1 if ax == axis else 1 for ax in range(x.ndim)])
            v = np.take(x, np.clip(idx, 0, n - 1), axis=axis)
            with np.errstate(invalid="ignore"):
                m = np.where(inside & ((m < v) if is_max else (v < m)), v, m)
        return m

    return fold(fold(a, 1), 0)


def shim_blur_remove_minmax(a, r, centre_first=True):
    """minmaxFilter.cpp blurRemoveMinMax_ through the shim, per channel: mx = dilate, mn = erode; mind = |a - mn|,
    maxd = |a - mx| (cv::absdiff), mask = cv::min(mind, maxd) = (maxd < mind) ? maxd : mind; out = mind == mask ? mn : mx."""
    if a.ndim == 3:
        return np.stack([shim_blur_remove_minmax(a[..., c], r, centre_first) for c in range(a.shape[2])], axis=2)
    mx = shim_morph(a, 2 * r + 1, True, centre_first); mn = shim_morph(a, 2 * r + 1, False, centre_first)
    with np.errstate(invalid="ignore", over="ignore"):
        mind = np.abs(a - mn); maxd = np.abs(a - mx)
        mask = np.where(maxd < mind, maxd, mind)
        return np.where(mind == mask, mn, mx)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("shape", SHAPES)
def test_ordered_specials_cv2_shim_port(port, shim, shape, dt):
    """±inf, ±max, values around ±FLT_MIN, subnormals and positive zeros: cv2 == shim == port, every odd k up to 21."""
    rs = np.random.RandomState(61); H, W = shape
    for trial in range(2):
        a = special_image(rs, H, W, dt, nan=False, negzero=False, p=0.3 if trial else 0.1)
        for k in KS:
            el = np.ones((k, k), np.uint8)
            for is_max, fn in ((True, cv2.dilate), (False, cv2.erode)):
                want = fn(a, el)
                assert_bits_equal(shim.morph(a, k, is_max), want, "shim k%d max%d %s" % (k, is_max, dt.__name__))
                assert_bits_equal(port.morph(a, k, is_max), want, "port k%d max%d %s" % (k, is_max, dt.__name__))
                assert_bits_equal(shim_morph(a, k, is_max), want, "restatement k%d max%d %s" % (k, is_max, dt.__name__))


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("shape", SHAPES)
def test_nan_and_signed_zero_follow_the_shim(port, shim, shape, dt):
    """NaN and zeros of both signs: shim == port == the centre-first restatement, for dilate / erode and for
    blurRemoveMinMax on one and three channels."""
    rs = np.random.RandomState(62); H, W = shape
    for kind in ("nan", "zeros", "all"):
        a = special_image(rs, H, W, dt, nan=kind != "zeros", negzero=True, p=0.05 if kind == "nan" else 0.2)
        if kind == "zeros":
            a[np.abs(a) < 1] = np.where(rs.rand(int((np.abs(a) < 1).sum())) < 0.5, -0.0, 0.0)
        else:
            a[rs.rand(H, W) < 0.05] = np.nan
        for k in KS:
            for is_max in (True, False):
                want = shim_morph(a, k, is_max)
                assert_bits_equal(shim.morph(a, k, is_max), want, "shim %s k%d max%d" % (kind, k, is_max))
                assert_bits_equal(port.morph(a, k, is_max), want, "port %s k%d max%d" % (kind, k, is_max))
        for r in (0, 1, 2, 5, 10):
            assert_bits_equal(port.blur_remove_minmax(a, r), shim_blur_remove_minmax(a, r), "blurRemoveMinMax %s r%d" % (kind, r))
        c3 = special_image(rs, H, W, dt, 3, nan=kind != "zeros", negzero=True, p=0.1)
        if kind != "zeros":
            c3[rs.rand(H, W, 3) < 0.05] = np.nan
        for r in (1, 2, 5):
            assert_bits_equal(port.blur_remove_minmax(c3, r), shim_blur_remove_minmax(c3, r), "blurRemoveMinMax C3 %s r%d" % (kind, r))


def test_the_images_tell_the_orders_apart(port):
    """The special-value images separate the centre-first order from a first-tap order: a kernel that starts its fold
    anywhere else fails the GPU tests built on them."""
    rs = np.random.RandomState(63)
    for dt in (np.float32, np.float64):
        for kind in ("nan", "zeros"):
            a = (rs.randint(-3, 4, size=(9, 11)) * 0.5).astype(dt)
            if kind == "nan":
                a[rs.rand(9, 11) < 0.1] = np.nan
            else:
                a[:] = np.where(rs.rand(9, 11) < 0.5, -0.0, 0.0)
                a[rs.rand(9, 11) < 0.3] = -1.0
            want = port.blur_remove_minmax(a, 1)
            assert_bits_equal(shim_blur_remove_minmax(a, 1), want, "centre first %s" % kind)
            first = shim_blur_remove_minmax(a, 1, centre_first=False)
            same = np.array_equal(np.isnan(first), np.isnan(want)) and np.array_equal(
                np.nan_to_num(first).view(np.uint8), np.nan_to_num(want).view(np.uint8))
            assert not same, "first-tap order gives the port's bits on the %s image" % kind


def test_single_special_in_a_flat_window(port):
    """One NaN or one -0 in a flat field, in the centre, on an edge and in a corner: where it survives is the rule."""
    for dt in (np.float32, np.float64):
        for (y, x) in ((2, 2), (0, 2), (4, 4), (2, 0)):
            a = np.ones((5, 5), dt); a[y, x] = np.nan
            got = port.morph(a, 3, True)
            want = np.ones((5, 5), dt); want[y, x] = np.nan                    # NaN only where it is the fold's seed
            assert_bits_equal(got, want, "NaN at %s" % ((y, x),))
            assert_bits_equal(shim_morph(a, 3, True), want, "restatement NaN at %s" % ((y, x),))
            z = np.zeros((5, 5), dt); z[y, x] = -0.0
            want = np.zeros((5, 5), dt); want[y, x] = -0.0                    # +0 > -0 is false: each pixel keeps its own sign
            for is_max in (True, False):
                assert_bits_equal(port.morph(z, 3, is_max).view(np.uint8), want.view(np.uint8), "-0 at %s" % ((y, x),))
