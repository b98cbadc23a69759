"""Bit-for-bit: the plain-C restatement (oracle/dmc_oracle.c) vs the UNMODIFIED reference sources
(oracle/_ref/libdmc_ref.so) on seeded random inputs, awkward shapes, every radius/threshold/type/method
of SURVEY.md 7.4.  Skipped where the reference build is absent."""
import numpy as np
import pytest

from _util import assert_bits_equal, make_image
from oracle.oracle_py import FULL_KERNEL, FULL_KERNEL_PAIR, SEPARABLE_KERNEL, FILL_DISPARITY, FILL_DEPTH

SHAPES = [(37, 53), (1, 5), (5, 1), (16, 16), (83, 131), (2, 150), (24, 641)]


@pytest.mark.parametrize("shape", SHAPES)
def test_median_gauss_minmax(port, ref, shape):
    rs = np.random.RandomState(1); H, W = shape
    for kind in ("pw", "noise", "const"):
        a = make_image(rs, H, W, kind=kind)
        for k in (1, 3, 5, 7, 9, 21):
            assert_bits_equal(port.median_blur(a, k), ref.median_blur(a, k), "median k%d" % k)
        for gr in (0, 1, 2, 3, 4, 5, 10):
            assert_bits_equal(port.small_gaussian(a, 2 * gr + 1, gr + 0.5), ref.small_gaussian(a, 2 * gr + 1, gr + 0.5), "gauss gr%d" % gr)
        assert_bits_equal(port.small_gaussian(a, 0, 0.5), ref.small_gaussian(a, 0, 0.5), "gauss d0")
    for r in (0, 1, 3, 5, 10):
        for dt in (np.uint8, np.uint16, np.int16, np.float32, np.float64):
            b = make_image(rs, H, W, dt)
            assert_bits_equal(port.blur_remove_minmax(b, r), ref.blur_remove_minmax(b, r), "brm r%d %s" % (r, dt.__name__))
            assert_bits_equal(ref.blur_remove_minmax(b, r, inplace=True), ref.blur_remove_minmax(b, r), "brm inplace")
            assert_bits_equal(ref.blur_remove_minmax_base(b, r), ref.blur_remove_minmax(b, r), "brm base twin")
    b = make_image(rs, H, W, np.uint8, 3)
    assert_bits_equal(port.blur_remove_minmax(b, 2), ref.blur_remove_minmax(b, 2), "brm C3")


def _mask_undefined(pa, ra, kw, kh, W, method, dtype):
    """32f path, rH%8==5, cols%4==0: rpad=-1 (binalyWeightedRangeFilter.cpp:993-997).  With a k x 1 kernel the
    last row's overflow read leaves the buffer (undefined); SEPARABLE then spreads it down the last column."""
    if dtype != np.uint8 and (kw >> 1) % 8 == 5 and W % 4 == 0:
        if method == SEPARABLE_KERNEL:
            pa[-(kh >> 1) - 1:, -1] = ra[-(kh >> 1) - 1:, -1]
        elif (kh >> 1) == 0:
            pa[-1, -1] = ra[-1, -1]


@pytest.mark.parametrize("shape", SHAPES)
def test_bwrf(port, ref, shape):
    rs = np.random.RandomState(2); H, W = shape
    for (kw, kh) in [(1, 1), (3, 3), (7, 7), (11, 11), (15, 15), (21, 21), (5, 1), (1, 5), (11, 1), (7, 3), (4, 4), (0, 3)]:
        for th in (0, 1, 10, 65, 254, 255, 10.9):
            for dt, cn in [(np.uint8, 1), (np.uint8, 3), (np.uint16, 1), (np.int16, 1), (np.float32, 1), (np.float32, 3)]:
                if kw > 11 and (th not in (10, 65) or cn == 3):
                    continue
                b = make_image(rs, H, W, dt, cn)
                init = make_image(rs, H, W, dt, cn, kind="noise")
                for m in (FULL_KERNEL, SEPARABLE_KERNEL):
                    pa = port.bwrf(b, kw, kh, th, m, dst_init=init); ra = ref.bwrf(b, kw, kh, th, m, dst_init=init)
                    _mask_undefined(pa, ra, kw, kh, W, m, dt)
                    assert_bits_equal(pa, ra, "bwrf %dx%d th%s %sC%d m%d" % (kw, kh, th, dt.__name__, cn, m))
    # 8U + FULL_KERNEL_PAIR is a silent no-op in the reference: dst keeps its previous contents
    b = make_image(rs, H, W); init = make_image(rs, H, W, kind="noise")
    assert_bits_equal(ref.bwrf(b, 5, 5, 10, FULL_KERNEL_PAIR, dst_init=init), init, "ref 8U PAIR no-op")
    assert_bits_equal(port.bwrf(b, 5, 5, 10, FULL_KERNEL_PAIR, dst_init=init), init, "port 8U PAIR no-op")
    # 16-bit + SEPARABLE: nothing happens either
    u = make_image(rs, H, W, np.uint16); iu = make_image(rs, H, W, np.uint16, kind="noise")
    assert_bits_equal(ref.bwrf(u, 5, 5, 10, SEPARABLE_KERNEL, dst_init=iu), iu, "ref 16U SEP no-op")
    assert_bits_equal(port.bwrf(u, 5, 5, 10, SEPARABLE_KERNEL, dst_init=iu), iu, "port 16U SEP no-op")
    # in-place is legal
    assert_bits_equal(ref.bwrf(b, 7, 7, 10, inplace=True), ref.bwrf(b, 7, 7, 10), "8u in-place")


def test_bwrf_inf_nan_propagation(port, ref):
    """0 * inf = NaN must propagate exactly as in the SSE kernel (binalyWeightedRangeFilter.cpp:525-526)."""
    rs = np.random.RandomState(3)
    a = make_image(rs, 40, 44, np.float32)
    a[10, 10] = np.inf; a[20, 30] = -np.inf; a[5, 40] = np.nan
    for k in (3, 5, 7):
        pa = port.bwrf(a, k, k, 30.0); ra = ref.bwrf(a, k, k, 30.0)
        assert_bits_equal(pa, ra, "inf/nan k%d" % k)
        assert np.isnan(pa).sum() >= 3
    d = np.zeros((33, 48), np.uint8); d[3:20, 5:30] = 90; d[8, 8] = 0    # disparity with a zero -> +inf depth
    assert_bits_equal(port.filter_disp8u_depth32f(d + 0, 75, 575, 2.6, 0, 0, 0, 2, 65.0), ref.filter_disp8u_depth32f(d + 0, 75, 575, 2.6, 0, 0, 0, 2, 65.0))
    assert_bits_equal(port.filter_disp8u_depth16u(d + 0, 75, 575, 2.6, 0, 0, 0, 2, 65.0), ref.filter_disp8u_depth16u(d + 0, 75, 575, 2.6, 0, 0, 0, 2, 65.0))


@pytest.mark.parametrize("shape", SHAPES[:5])
def test_brf_and_minmax_filters(port, ref, shape):
    rs = np.random.RandomState(4); H, W = shape
    for dt in (np.uint8, np.uint16, np.int16, np.float32, np.float64):
        for kind in ("pw", "const", "noise"):
            b = make_image(rs, H, W, dt, kind=kind)
            for (kw, kh, f, c, s) in [(1, 1, 1, 1, 1), (3, 3, 1, 1, 1), (7, 7, 1, 1, 1), (13, 13, 1, 1, 1), (5, 9, 0.5, 2, 1.5), (9, 5, 0, 0, 0)]:
                if kind == "noise" and kw > 7:
                    continue
                assert_bits_equal(port.brf(b, kw, kh, f, c, s), ref.brf(b, kw, kh, f, c, s), "brf %dx%d %s %s" % (kw, kh, dt.__name__, kind))
        b = make_image(rs, H, W, dt)
        assert_bits_equal(ref.brf(b, 7, 7, 1, 1, 1, inplace=True), ref.brf(b, 7, 7, 1, 1, 1), "brf in-place")
    for dt in (np.uint8, np.uint16, np.int16, np.float32):
        b = make_image(rs, H, W, dt)
        if dt == np.float32:
            b = b - 300     # negative data: the FLT_MIN seed of maxFilter leaks (minmaxFilter.cpp:332)
        for (kw, kh) in [(3, 3), (7, 5), (1, 3), (3, 1), (1, 1)]:
            assert_bits_equal(port.max_filter(b, kw, kh), ref.max_filter(b, kw, kh), "maxFilter %s" % dt.__name__)
            assert_bits_equal(port.min_filter(b, kw, kh), ref.min_filter(b, kw, kh), "minFilter %s" % dt.__name__)


def test_converters_fill_reproject(port, ref):
    rs = np.random.RandomState(5)
    for (H, W) in [(16, 16), (7, 9), (33, 21), (48, 64)]:
        d8 = make_image(rs, H, W, kind="noise")          # contains zeros -> inf
        d16 = (rs.randint(0, 65536, size=(H, W))).astype(np.uint16); d16[rs.rand(H, W) < 0.2] = 0
        s16 = (rs.randint(-3000, 3000, size=(H, W))).astype(np.int16)
        f32 = (rs.rand(H, W) * 5000).astype(np.float32); f32[rs.rand(H, W) < 0.1] = 0
        for (a, b) in [(2.6, 0.0), (1.0, 0.0), (2.6, 3.5)]:
            init = (rs.rand(H, W) * 9).astype(np.float32)
            assert_bits_equal(port.disp8u2depth32f(d8, 43125.0, a, b, dst=init), ref.disp8u2depth32f(d8, 43125.0, a, b, dst=init), "disp8U2depth32F")
            assert_bits_equal(port.depth32f2disp8u(f32, 43125.0, a, b), ref.depth32f2disp8u(f32, 43125.0, a, b), "depth32F2disp8U")
            assert_bits_equal(port.depth16u2disp8u(d16, 43125.0, a, b), ref.depth16u2disp8u(d16, 43125.0, a, b), "depth16U2disp8U")
            assert_bits_equal(port.disp16s2depth16u(s16, 43125.0, a, b), ref.disp16s2depth16u(s16, 43125.0, a, b), "disp16S2depth16U")
        for dt in (np.uint8, np.uint16, np.int16, np.float32):
            img = make_image(rs, H, W, dt); img[rs.rand(H, W) < 0.3] = 0; img[-1] = 9   # (a blanked LAST row makes the reference read past the buffer)
            if W > 2:
                assert_bits_equal(port.fill_occlusion(img, 0, FILL_DISPARITY), ref.fill_occlusion(img, 0, FILL_DISPARITY), "fill disp")
                img2 = img.copy(); img2[img2 == 0] = 1; img2[rs.rand(H, W) < 0.3] = 7; img2[-1] = 9
                assert_bits_equal(port.fill_occlusion(img2, 7, FILL_DEPTH), ref.fill_occlusion(img2, 7, FILL_DEPTH), "fill depth")
            assert_bits_equal(port.reproject_xyz(img, 510.0), ref.reproject_xyz(img, 510.0), "reprojectXYZ")


@pytest.mark.parametrize("shape", [(48, 64), (37, 53), (9, 150)])
def test_post_filter_set_entry_points(port, ref, shape):
    rs = np.random.RandomState(6); H, W = shape
    for trial in range(3):
        a = np.maximum(make_image(rs, H, W, kind=("pw", "noise", "pw")[trial]), 1)
        for (mr, gr, mmr, br, th) in [(2, 1, 3, 5, 10), (1, 0, 1, 3, 10), (0, 0, 0, 0, 0), (3, 2, 2, 4, 30), (1, 3, 0, 7, 255)]:
            for m in (FULL_KERNEL, SEPARABLE_KERNEL):
                assert_bits_equal(port.post_filter_set(a, mr, gr, mmr, br, th, m), ref.post_filter_set(a, mr, gr, mmr, br, th, m), "operator()")
            assert_bits_equal(port.filter_disp8u_depth32f(a, 75, 575, 2.6, mr, gr, mmr, br, th * 6.5), ref.filter_disp8u_depth32f(a, 75, 575, 2.6, mr, gr, mmr, br, th * 6.5), "Depth32F")
            assert_bits_equal(port.filter_disp8u_depth16u(a, 75, 575, 2.6, mr, gr, mmr, br, th * 6.5), ref.filter_disp8u_depth16u(a, 75, 575, 2.6, mr, gr, mmr, br, th * 6.5), "Depth16U")
            assert_bits_equal(port.filter_disp8u_disp32f(a, mr, gr, mmr, br, th + 0.5), ref.filter_disp8u_disp32f(a, mr, gr, mmr, br, th + 0.5), "Disp32F")


def test_reference_is_thread_count_invariant(ref_build):
    ref = ref_build
    rs = np.random.RandomState(7); a = make_image(rs, 96, 128)
    outs = []
    for n in (1, 3, 8):
        ref.set_num_threads(n)
        outs.append((ref.post_filter_set(a, 2, 1, 3, 5, 10), ref.brf(a, 7, 7, 1, 1, 1), ref.bwrf(a.astype(np.float32), 7, 7, 20.0)))
    ref.set_num_threads(0)
    for o in outs[1:]:
        for x, y in zip(o, outs[0]):
            assert_bits_equal(x, y, "thread-count invariance")


def test_max_min_filter_equal_dilate_erode_for_integers(port):
    rs = np.random.RandomState(8)
    for dt in (np.uint8, np.uint16, np.int16):
        b = make_image(rs, 31, 47, dt)
        for k in (3, 7):
            assert_bits_equal(port.max_filter(b, k, k), port.morph(b, k, True), "maxFilter == dilate")
            assert_bits_equal(port.min_filter(b, k, k), port.morph(b, k, False), "minFilter == erode")
