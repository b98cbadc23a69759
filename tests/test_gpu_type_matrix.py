"""The range filter and the min-max filters on every source type and channel count the C ABI accepts, bit for bit
against the CPU oracle (oracle/dmc_oracle.c):

  * binalyWeightedRangeFilter on 16UC3 / 16SC3: the three-channel tiled kernel (square windows) and the generic kernel
    (other windows) with 16-bit loads and saturating 16-bit stores, the padding quirk read through 16-bit loads, the
    FP32 sums that stop being exact at radius 10, FULL_KERNEL_PAIR, the no-op SEPARABLE_KERNEL, in place and strided;
    and the order of the three-channel L1 distance on 32FC3, where rounding makes it visible.
  * blurRemoveMinMax on {8U, 16U, 16S, 32F, 64F} x {C1, C3}: every radius, ties, saturated 16S distances, in place and
    pinned memory; NaN, signed zeros, infinities, subnormals and values around FLT_MIN for 32F / 64F, and for
    maxFilter / minFilter on 32F.  Where the visiting order of a float min / max shows (NaN, +0 against -0) the oracle
    follows the shim's centre-first order (tests/test_morph_special_values.py pins that rule on the CPU).
Run with `-m gpu` on a B200."""
import numpy as np
import pytest

from _util import assert_bits_equal, bits_equal, make_image, mask_undefined, special_image

pytestmark = pytest.mark.gpu

SHAPES = [(37, 53), (1, 5), (5, 1), (16, 16), (83, 131), (2, 150), (24, 641), (100, 1023)]
BIG = (520, 1100)
INT16 = [np.uint16, np.int16]
THS = (0, 10.9, 160, 65535, 1e9, -1, float("nan"))       # -1 and NaN: no tap passes, 0/0 -> cvRound(NaN) -> saturated store
MINMAX_TYPES = [np.uint8, np.uint16, np.int16, np.float32, np.float64]


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)          # raises loudly without a GPU / without the built library
    return m


def check_bwrf(dmc, port, b, kw, kh, th, method=None, init=None, msg=""):
    method = dmc.FULL_KERNEL if method is None else method
    want = port.bwrf(b, kw, kh, th, method, dst_init=init)
    got = dmc.binalyWeightedRangeFilter(b, None if init is None else init.copy(), (kw, kh), th, method)
    mask_undefined(got, want, kw, kh, b.shape[1], method, b.dtype.type, dmc)
    assert_bits_equal(got, want, "%s bwrf %dx%d th%s %s%s m%d" % (msg, kw, kh, th, b.dtype.name, b.shape[2:], method))
    return want


# ------------------------------------------------------------------------------------- range filter, 16-bit C3
@pytest.mark.parametrize("shape", SHAPES + [BIG])
def test_bwrf_16bit_c3_square(dmc, port, shape):
    """FULL_KERNEL, square windows r = 1..10: the three-channel tiled kernel with 16-bit loads and stores."""
    rs = np.random.RandomState(71); H, W = shape
    for dt in INT16:
        b = make_image(rs, H, W, dt, 3)
        for r in range(1, 11):
            for th in THS:
                check_bwrf(dmc, port, b, 2 * r + 1, 2 * r + 1, th)


@pytest.mark.parametrize("shape", SHAPES)
def test_bwrf_16bit_c3_windows(dmc, port, shape):
    """Non-square windows (the generic kernel), the degenerate ones, and SEPARABLE_KERNEL, which does nothing on 16-bit
    sources: a pre-filled dst comes back untouched."""
    rs = np.random.RandomState(72); H, W = shape
    for dt in INT16:
        b = make_image(rs, H, W, dt, 3)
        init = make_image(rs, H, W, dt, 3, kind="noise")
        for (kw, kh) in [(5, 1), (1, 5), (7, 3), (4, 4), (0, 3), (1, 1), (11, 1), (3, 21)]:
            for th in THS:
                check_bwrf(dmc, port, b, kw, kh, th, dmc.FULL_KERNEL, init)
            got = dmc.binalyWeightedRangeFilter(b, init.copy(), (kw, kh), 160, dmc.SEPARABLE_KERNEL)
            assert_bits_equal(got, init, "SEPARABLE_KERNEL on %sC3 is a no-op" % dt.__name__)


def test_bwrf_16bit_empty_window_copies(dmc, port):
    """A window of width or height 0 copies the image (binalyWeightedRangeFilter.cpp:980) at any threshold, negative and
    NaN included; a 1x1 window is a filter, whose one tap those thresholds reject."""
    rs = np.random.RandomState(70)
    for dt in INT16:
        for cn in (1, 3):
            b = make_image(rs, 29, 47, dt, cn)
            for (kw, kh) in [(0, 3), (5, 0), (0, 0)]:
                for th in THS:
                    want = check_bwrf(dmc, port, b, kw, kh, th)
                    assert_bits_equal(want, b, "empty window %dx%d th%s" % (kw, kh, th))
            for th in (-1, float("nan")):
                want = check_bwrf(dmc, port, b, 1, 1, th)
                assert not np.array_equal(want, b)


def test_bwrf_16bit_c3_padding_quirk(dmc, port):
    """r = 5 with cols % 4 == 0: the last column's tap (i, +5) reads the next colour plane (the next row for the last
    plane) through 16-bit loads.  Only the pixels mask_undefined names may differ, and the quirk must show in the
    oracle's output, or these images would not test it."""
    rs = np.random.RandomState(73)
    shown = {np.uint16: False, np.int16: False}
    for (H, W) in [(1, 4), (2, 8), (7, 12), (37, 16), (20, 128), (33, 132), (16, 256), (9, 640)]:
        for dt in INT16:
            b = make_image(rs, H, W, dt, 3)
            # the same image one column wider (a copy of the last one) has no quirk and the same replicated border
            wide = np.ascontiguousarray(np.concatenate([b, b[:, -1:]], axis=1))
            for (kw, kh) in [(11, 11), (11, 1), (11, 3), (11, 7)]:
                for th in (160, 1e9):
                    want = check_bwrf(dmc, port, b, kw, kh, th, msg="quirk %dx%d" % (H, W))
                    plain = port.bwrf(wide, kw, kh, th)[:, :W]
                    assert_bits_equal(want[:, :-1], plain[:, :-1], "the quirk touches the last column only")
                    shown[dt] |= not bits_equal(want[:, -1], plain[:, -1])
    assert all(shown.values()), shown


def test_bwrf_16bit_c3_extremes(dmc, port):
    """Values at the 16-bit limits: 16UC3 mostly 65535 and 16SC3 across -32768..32767, at r = 9 and r = 10.  At r = 10
    a disc has 317 taps and 317 * 65535 > 2^24, so the FP32 sums round and their order shows."""
    rs = np.random.RandomState(74); H, W = 70, 141
    hi = np.where(rs.rand(H, W, 3) < 0.9, 65535, rs.randint(0, 65536, size=(H, W, 3))).astype(np.uint16)
    sg = rs.randint(-32768, 32768, size=(H, W, 3)).astype(np.int16)
    sg[rs.rand(H, W) < 0.3] = (32767, -32768, 32767)
    for name, b in (("hi", hi), ("signed", sg)):
        for r in (9, 10):
            for th in (0, 17.5, 65535, 131070, 1e9, -1):
                check_bwrf(dmc, port, b, 2 * r + 1, 2 * r + 1, th, msg=name)
            check_bwrf(dmc, port, b, 2 * r + 1, 2 * r - 1, 1e9, msg=name)           # generic kernel, same sums


def test_bwrf_pair_equals_full_on_16bit(dmc, port):
    """FULL_KERNEL_PAIR on 16-bit sources is documented to return the FULL_KERNEL result."""
    rs = np.random.RandomState(75)
    for dt in INT16:
        for cn in (1, 3):
            for (H, W) in [(37, 53), (100, 1023)]:
                b = make_image(rs, H, W, dt, cn)
                for (kw, kh) in [(3, 3), (7, 7), (11, 11), (21, 21), (7, 3)]:
                    for th in (10.9, 160):
                        want = port.bwrf(b, kw, kh, th, dmc.FULL_KERNEL)
                        got = dmc.binalyWeightedRangeFilter(b, None, (kw, kh), th, dmc.FULL_KERNEL_PAIR)
                        mask_undefined(got, want, kw, kh, W, dmc.FULL_KERNEL, dt, dmc)
                        assert_bits_equal(got, want, "PAIR == FULL %sC%d %dx%d th%s" % (dt.__name__, cn, kw, kh, th))


def test_bwrf_16bit_c3_in_place_and_strided(dmc, port):
    rs = np.random.RandomState(76); H, W = 61, 97
    for dt in INT16:
        b = make_image(rs, H, W, dt, 3)
        for (kw, kh) in [(7, 7), (5, 1)]:
            c = b.copy(); dmc.binalyWeightedRangeFilter(c, c, (kw, kh), 160, dmc.FULL_KERNEL)
            assert_bits_equal(c, port.bwrf(b, kw, kh, 160), "in place %s %dx%d" % (dt.__name__, kw, kh))
        big = make_image(rs, H + 9, W + 23, dt, 3)
        view = big[4:4 + H, 7:7 + W]                                  # rows further apart than cols * 3 elements
        assert_bits_equal(dmc.binalyWeightedRangeFilter(view, None, (9, 9), 160, dmc.FULL_KERNEL),
                          port.bwrf(np.ascontiguousarray(view), 9, 9, 160), "strided src %s" % dt.__name__)


def test_bwrf_c3_distance_order(dmc, port):
    """The three-channel distance is (|d2| + |d1|) + |d0| in FP32.  With |d2| = 2^24 and |d1| = |d0| = 1 that is 2^24,
    while any other order gives 2^24 + 2, so a threshold of 2^24 keeps or drops the tap by the order alone.  Filtering
    the channel-reversed image (the reversed order) must give different bits, or this image would not test it."""
    rs = np.random.RandomState(77); H, W = 45, 140
    b = np.stack([rs.randint(0, 3, size=(H, W)), rs.randint(0, 3, size=(H, W)), rs.randint(0, 2, size=(H, W)) * 2 ** 24], axis=2)
    b = np.ascontiguousarray(b.astype(np.float32))
    th = float(2 ** 24)
    for (kw, kh) in [(3, 3), (5, 5), (11, 11), (21, 21), (7, 3)]:
        want = check_bwrf(dmc, port, b, kw, kh, th, msg="distance order")
        rev = port.bwrf(np.ascontiguousarray(b[..., ::-1]), kw, kh, th)[..., ::-1]
        assert not bits_equal(want, np.ascontiguousarray(rev)), "channel order does not show at %dx%d" % (kw, kh)


# ------------------------------------------------------------------------------------- blurRemoveMinMax
@pytest.mark.parametrize("shape", SHAPES)
def test_minmax_type_matrix(dmc, port, shape):
    """{8U, 16U, 16S, 32F, 64F} x {C1, C3}, r = 0..10 (multi-channel images run one plane per blockIdx.z)."""
    rs = np.random.RandomState(78); H, W = shape
    for dt in MINMAX_TYPES:
        for cn in (1, 3):
            for kind in ("pw", "noise"):
                b = make_image(rs, H, W, dt, cn, kind=kind)
                for r in range(0, 11):
                    assert_bits_equal(dmc.blurRemoveMinMax(b, None, r), port.blur_remove_minmax(b, r), "%sC%d %s r%d" % (dt.__name__, cn, kind, r))
            c = b.copy(); dmc.blurRemoveMinMax(c, c, 3)
            assert_bits_equal(c, port.blur_remove_minmax(b, 3), "in place %sC%d" % (dt.__name__, cn))


TIE = {np.uint8: (10, 20, 30), np.uint16: (1000, 30000, 59000), np.int16: (-30000, 0, 30000),
       np.float32: (-1.5, 0.25, 2.0), np.float64: (-1.5, 0.25, 2.0)}


def test_minmax_ties_go_to_min(dmc, port):
    """src - mn == mx - src selects mn: columns repeat (lo, mid, hi) with mid - lo == hi - mid, so at r = 1 every
    interior mid pixel ties."""
    H, W = 23, 61
    for dt in MINMAX_TYPES:
        lo, mid, hi = TIE[dt]
        row = np.array([lo, mid, hi] * (W // 3 + 1), dt)[:W]
        for cn in (1, 3):
            if cn == 1:
                a = np.ascontiguousarray(np.broadcast_to(row, (H, W)))
            else:
                a = np.ascontiguousarray(np.stack([np.roll(row, c)[None].repeat(H, 0) for c in range(3)], axis=2))
            got = dmc.blurRemoveMinMax(a, None, 1)
            assert_bits_equal(got, port.blur_remove_minmax(a, 1), "ties %sC%d" % (dt.__name__, cn))
            ties = (a[:, 1:-1] == mid) & (a[:, :-2] != a[:, 2:])
            assert ties.any() and np.all(got[:, 1:-1][ties] == lo), "ties %sC%d must take mn" % (dt.__name__, cn)


def test_minmax_16s_saturated_distances(dmc, port):
    """16S windows holding -32768 and 32767: |src - mn| and |mx - src| saturate at 32767 (cv::absdiff), so src in
    {-1, 0} ties and takes mn, and src = 5 is nearer mx by saturation only."""
    for v, want in ((0, -32768), (-1, -32768), (5, 32767), (-5, -32768)):
        a = np.array([[-32768, v, 32767]], np.int16)
        got = dmc.blurRemoveMinMax(a, None, 1)
        assert got[0, 1] == want, (v, got)
        assert_bits_equal(got, port.blur_remove_minmax(a, 1), "1x3 with %d" % v)
    rs = np.random.RandomState(79)
    for (H, W) in [(37, 53), (100, 1023)]:
        for cn in (1, 3):
            shape = (H, W) if cn == 1 else (H, W, cn)
            a = rs.randint(-200, 201, size=shape).astype(np.int16)
            sel = rs.rand(*shape)
            a[sel < 0.1] = -32768; a[(sel >= 0.1) & (sel < 0.2)] = 32767
            for r in (1, 2, 5):
                assert_bits_equal(dmc.blurRemoveMinMax(a, None, r), port.blur_remove_minmax(a, r), "16SC%d extremes r%d" % (cn, r))


def test_minmax_pinned_host(dmc, port):
    rs = np.random.RandomState(80); H, W = 57, 203
    b = make_image(rs, H, W, np.float32, 3)
    p = dmc.pinned_empty((H, W, 3), np.float32)
    p[:] = b
    dmc.blurRemoveMinMax(p, p, 2)
    assert_bits_equal(p, port.blur_remove_minmax(b, 2), "pinned 32FC3 in place")
    q = dmc.pinned_empty((H, W), np.uint16); o = dmc.pinned_empty((H, W), np.uint16)
    q[:] = make_image(rs, H, W, np.uint16)
    assert_bits_equal(dmc.blurRemoveMinMax(q, o, 4), port.blur_remove_minmax(np.array(q), 4), "pinned 16UC1")


# ------------------------------------------------------------------------------------- float special values
def specials(rs, H, W, dt, cn, kind):
    """kind "nan": NaN at 5 % of the pixels; "zeros": zeros of both signs; "all": every special value"""
    a = special_image(rs, H, W, dt, cn, nan=kind != "zeros", negzero=True, p=0.05 if kind == "nan" else 0.2)
    shape = a.shape
    if kind == "zeros":
        small = np.abs(a) < 1
        a[small] = np.where(rs.rand(int(small.sum())) < 0.5, -0.0, 0.0)
    else:
        a[rs.rand(*shape) < 0.05] = np.nan
    return a


@pytest.mark.parametrize("shape", SHAPES)
def test_minmax_float_specials(dmc, port, shape):
    """blurRemoveMinMax 32F / 64F, C1 and C3, on NaN, signed zeros, ±inf, ±max, subnormals and values around the
    smallest normal, at the border, in the middle of windows and as the first tap of windows."""
    rs = np.random.RandomState(81); H, W = shape
    for dt in (np.float32, np.float64):
        for cn in (1, 3):
            for kind in ("nan", "zeros", "all"):
                a = specials(rs, H, W, dt, cn, kind)
                for r in (1, 2, 5, 10):
                    assert_bits_equal(dmc.blurRemoveMinMax(a, None, r), port.blur_remove_minmax(a, r), "%s %sC%d r%d" % (kind, dt.__name__, cn, r))


def test_minmax_single_special(dmc, port):
    """One NaN or one -0 in a flat window, in the centre, on an edge, in a corner and at the first tap of its neighbours'
    windows."""
    for dt in (np.float32, np.float64):
        for (y, x) in ((3, 4), (0, 4), (6, 8), (3, 0), (0, 0), (1, 1)):
            for special, fill in ((np.nan, 1.0), (-0.0, 0.0), (0.0, -0.0)):
                a = np.full((7, 9), fill, dt); a[y, x] = special
                for r in (1, 2):
                    assert_bits_equal(dmc.blurRemoveMinMax(a, None, r), port.blur_remove_minmax(a, r), "%r at %s r%d" % (special, (y, x), r))


@pytest.mark.parametrize("shape", SHAPES)
def test_max_min_filter_f32_specials(dmc, port, shape):
    """maxFilter / minFilter 32F (FLT_MIN / FLT_MAX seeded sliding window) on the same special values."""
    rs = np.random.RandomState(82); H, W = shape
    for kind in ("nan", "zeros", "all"):
        a = specials(rs, H, W, np.float32, 1, kind)
        for (kw, kh) in [(3, 3), (5, 5), (11, 11), (21, 21), (7, 3), (1, 5)]:
            assert_bits_equal(dmc.maxFilter(a, None, (kw, kh)), port.max_filter(a, kw, kh), "maxFilter %s %dx%d" % (kind, kw, kh))
            assert_bits_equal(dmc.minFilter(a, None, (kw, kh)), port.min_filter(a, kw, kh), "minFilter %s %dx%d" % (kind, kw, kh))
