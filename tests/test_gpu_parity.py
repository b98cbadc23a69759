"""GPU parity tests proper: libdmc_b200.so (through the C ABI, via the Python mirror of filter.h) against the CPU
restatement (oracle/dmc_oracle.c) on the same seeded inputs and against the committed golden vectors produced by
the unmodified reference.  Bit-exact everywhere (NaN-aware for floats).  Run with `-m gpu` on a B200."""
import ctypes as C
import numpy as np
import pytest

from _util import assert_bits_equal, canon_crc, load_golden, load_png, make_image, mask_undefined

pytestmark = pytest.mark.gpu

FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6
SHAPES = [(37, 53), (1, 5), (5, 1), (16, 16), (83, 131), (2, 150), (24, 641), (100, 1023)]


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)          # raises loudly without a GPU / without the built library
    return m


# ---------------------------------------------------------------------------------------------- golden vectors
GOLD = load_golden()
CHAIN_INPUTS = [k for k in GOLD["inputs"] if "depth16" not in k]


def gpu_chain_op(m, key, img):
    fb = FOCUS * BASELINE
    pfs = m.PostFilterSet()
    if key == "pfs_2_1_3_5_10": return pfs(img, None, 2, 1, 3, 5, 10)
    if key == "pfs_1_0_1_3_10": return pfs(img, None, 1, 0, 1, 3, 10)
    if key == "pfs_2_1_3_5_10_sep": return pfs(img, None, 2, 1, 3, 5, 10, m.SEPARABLE_KERNEL)
    if key == "depth32f_1_0_1_3_65": return pfs.filterDisp8U2Depth32F(img, None, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0)
    if key == "depth16u_1_0_1_3_65": return pfs.filterDisp8U2Depth16U(img, None, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0)
    if key == "disp32f_1_0_1_3_10": return pfs.filterDisp8U2Disp32F(img, None, 1, 0, 1, 3, 10.0)
    if key == "depth32f2disp8u": return m.depth32F2disp8U(pfs.filterDisp8U2Depth32F(img, None, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0), None, fb, AMP, 0.0)
    if key == "reproject_xyz_510": return m.reprojectXYZ(pfs.filterDisp8U2Depth32F(img, None, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0), None, 510.0)
    if key == "brf_13_1_1_1": return m.boundaryReconstructionFilter(img, None, (13, 13), 1, 1, 1)
    if key == "brf_7_1_2_05": return m.boundaryReconstructionFilter(img, None, (7, 7), 1, 2, 0.5)
    if key.startswith("bwrf8u_r"): r = int(key[8]); return m.binalyWeightedRangeFilter(img, None, (2 * r + 1, 2 * r + 1), 10, m.FULL_KERNEL)
    if key == "bwrf8u_sep_11_th10": return m.binalyWeightedRangeFilter(img, None, (11, 11), 10, m.SEPARABLE_KERNEL)
    if key == "bwrf32f_r3_th65": return m.binalyWeightedRangeFilter(img.astype(np.float32) * 16.0, None, (7, 7), 65.0, m.FULL_KERNEL)
    if key == "bwrf32f_r5_th65": return m.binalyWeightedRangeFilter(img.astype(np.float32) * 16.0, None, (11, 11), 65.0, m.FULL_KERNEL)
    if key == "bwrf16u_r2_th160": return m.binalyWeightedRangeFilter(img.astype(np.uint16) * 16, None, (5, 5), 160.0, m.FULL_KERNEL)
    if key.startswith("minmax_r"): return m.blurRemoveMinMax(img, None, int(key[8:]))
    if key.startswith("median_k"): return m.medianBlur(img, None, int(key[8:]))
    if key.startswith("gauss_gr"): gr = int(key[8:]); return m.smallGaussianBlur(img, None, 2 * gr + 1, gr + 0.5)
    if key == "disp8u2depth32f": return m.disp8U2depth32F(img, None, fb, AMP, 0.0)
    raise KeyError(key)


@pytest.mark.parametrize("name", CHAIN_INPUTS)
def test_golden_chain(dmc, name):
    """Kinect (JPEG q50/q80) and x264 fixtures of the reference: every operator must hash to the reference's CRC."""
    img = load_png(name)
    for key, want in GOLD["inputs"][name]["golden"].items():
        assert canon_crc(gpu_chain_op(dmc, key, img)) == want, (name, key)


def test_golden_depth16(dmc):
    name = "kinect_meeting_depth16_crop.png"; d16 = load_png(name); g = GOLD["inputs"][name]["golden"]
    fb = FOCUS * BASELINE
    disp = dmc.depth16U2disp8U(d16, None, fb, AMP, 0.0)
    assert canon_crc(disp) == g["depth16u2disp8u"]
    f1 = dmc.fillOcclusion(disp.copy(), 0, dmc.FILL_DISPARITY)
    assert canon_crc(f1) == g["fill_disparity_1pass"]
    # pointcloudTest's two-pass fill (main.cpp:257-260): fill, transpose, fill, transpose -- all four through the library
    t = dmc.fillOcclusion(dmc.transpose(f1), 0, dmc.FILL_DISPARITY)
    assert canon_crc(dmc.transpose(t)) == g["fill_disparity_2pass"]
    for dt in (np.uint8, np.uint16, np.float32, np.float64):
        a = (np.arange(37 * 91).reshape(37, 91) % 251).astype(dt)
        assert_bits_equal(dmc.transpose(a), np.ascontiguousarray(a.T), "transpose %s" % dt.__name__)
    assert canon_crc(dmc.reprojectXYZ(d16, None, 510.0)) == g["reproject_xyz_16u_510"]


# ---------------------------------------------------------------------------------------------- seeded random vs oracle
@pytest.mark.parametrize("shape", SHAPES)
def test_median_gauss_minmax(dmc, port, shape):
    rs = np.random.RandomState(21); H, W = shape
    for kind in ("pw", "noise", "const"):
        a = make_image(rs, H, W, kind=kind)
        for k in (1, 3, 5, 7, 9, 21):
            assert_bits_equal(dmc.medianBlur(a, None, k), port.median_blur(a, k), "median k%d" % k)
        for gr in (0, 1, 2, 3, 4, 5, 10):
            assert_bits_equal(dmc.smallGaussianBlur(a, None, 2 * gr + 1, gr + 0.5), port.small_gaussian(a, 2 * gr + 1, gr + 0.5), "gauss gr%d" % gr)
        assert_bits_equal(dmc.smallGaussianBlur(a, None, 0, 0.5), a, "gauss d=0")
        for d in (3, 5, 7, 9, 11):          # sigma <= 0: OpenCV's fixed small kernels
            assert_bits_equal(dmc.smallGaussianBlur(a, None, d, 0.0), port.small_gaussian(a, d, 0.0), "gauss d%d sigma 0" % d)
    for r in (0, 1, 3, 5, 10):
        for dt in (np.uint8, np.uint16, np.int16, np.float32, np.float64):
            b = make_image(rs, H, W, dt)
            want = port.blur_remove_minmax(b, r)
            assert_bits_equal(dmc.blurRemoveMinMax(b, None, r), want, "blurRemoveMinMax r%d %s" % (r, dt.__name__))
            assert_bits_equal(dmc.blurRemoveMinMaxBase(b, None, r), want, "blurRemoveMinMaxBase")
            c = b.copy(); dmc.blurRemoveMinMax(c, c, r)
            assert_bits_equal(c, want, "blurRemoveMinMax in-place")
    b = make_image(rs, H, W, np.uint8, 3)
    assert_bits_equal(dmc.blurRemoveMinMax(b, None, 2), port.blur_remove_minmax(b, 2), "blurRemoveMinMax C3")


@pytest.mark.parametrize("shape", [(83, 131), (100, 1023), (64, 256)])
def test_bwrf_radius_sweep(dmc, port, shape):
    """Every radius of the packed fast paths (8UC1 r<=6, 8UC3 r<=7, float r<=7), the thresholds either side of the
    exact-fp16 limits (ntaps*th and (2r+1)*th around 2048) and the BASELINE config-3 values (th 160 / 30)."""
    rs = np.random.RandomState(31); H, W = shape
    for r in range(1, 11):
        k = 2 * r + 1
        for dt, cn, ths in [(np.uint8, 1, (10, 25, 30, 140, 255)), (np.uint8, 3, (10, 30, 140, 255)), (np.uint16, 1, (160,)), (np.float32, 1, (30.5,))]:
            b = make_image(rs, H, W, dt, cn)
            for th in ths:
                want = port.bwrf(b, k, k, th, dmc.FULL_KERNEL)
                got = dmc.binalyWeightedRangeFilter(b, None, (k, k), th, dmc.FULL_KERNEL)
                mask_undefined(got, want, k, k, W, dmc.FULL_KERNEL, dt, dmc)
                assert_bits_equal(got, want, "bwrf sweep r%d th%s %sC%d" % (r, th, dt.__name__, cn))


def test_bwrf_integer_mode_limits(dmc, port):
    """16-bit sources run the 32-bit range filter in packed integers (csrc/dmc_bwrf32f_tiled.cu): the largest sums (253 taps
    of 65535 at radius 9), radius 10 (float path again), thresholds that pass everything / nothing / are not integers,
    negative values, and negative thresholds (no tap passes: 0/0 in the reference)."""
    rs = np.random.RandomState(41); H, W = 70, 141
    hi = np.where(rs.rand(H, W) < 0.9, 65535, rs.randint(0, 65536, size=(H, W))).astype(np.uint16)
    mix = rs.randint(0, 65536, size=(H, W)).astype(np.uint16)
    sg = rs.randint(-32768, 32768, size=(H, W)).astype(np.int16)
    near = (30000 + rs.randint(-40, 41, size=(H, W))).astype(np.uint16)
    for r in (1, 4, 7, 8, 9, 10):
        k = 2 * r + 1
        for name, b in (("hi", hi), ("mix", mix), ("signed", sg), ("near", near)):
            for th in (0, 0.99, 17.5, 40, 65535, 1e9, -1):
                want = port.bwrf(b, k, k, th, dmc.FULL_KERNEL)
                got = dmc.binalyWeightedRangeFilter(b, None, (k, k), th, dmc.FULL_KERNEL)
                mask_undefined(got, want, k, k, W, dmc.FULL_KERNEL, b.dtype.type, dmc)
                assert_bits_equal(got, want, "bwrf integer mode %s r%d th%s" % (name, r, th))


@pytest.mark.parametrize("shape", SHAPES)
def test_bwrf(dmc, port, shape):
    rs = np.random.RandomState(22); H, W = shape
    for (kw, kh) in [(1, 1), (3, 3), (7, 7), (11, 11), (15, 15), (21, 21), (5, 1), (1, 5), (11, 1), (7, 3), (4, 4), (0, 3)]:
        for th in (0, 1, 10, 65, 254, 255, 10.9):
            for dt, cn in [(np.uint8, 1), (np.uint8, 3), (np.uint16, 1), (np.int16, 1), (np.float32, 1), (np.float32, 3)]:
                if kw > 11 and (th not in (10, 65) or cn == 3):
                    continue
                b = make_image(rs, H, W, dt, cn)
                init = make_image(rs, H, W, dt, cn, kind="noise")
                for meth in (dmc.FULL_KERNEL, dmc.SEPARABLE_KERNEL):
                    want = port.bwrf(b, kw, kh, th, meth, dst_init=init)
                    got = dmc.binalyWeightedRangeFilter(b, init.copy(), (kw, kh), th, meth)
                    mask_undefined(got, want, kw, kh, W, meth, dt, dmc)
                    assert_bits_equal(got, want, "bwrf %dx%d th%s %sC%d m%d" % (kw, kh, th, dt.__name__, cn, meth))
    # silent no-ops leave dst untouched
    b = make_image(rs, H, W); init = make_image(rs, H, W, kind="noise")
    assert_bits_equal(dmc.binalyWeightedRangeFilter(b, init.copy(), (5, 5), 10, dmc.FULL_KERNEL_PAIR), init, "8U PAIR no-op")
    u = make_image(rs, H, W, np.uint16); iu = make_image(rs, H, W, np.uint16, kind="noise")
    assert_bits_equal(dmc.binalyWeightedRangeFilter(u, iu.copy(), (5, 5), 10, dmc.SEPARABLE_KERNEL), iu, "16U SEP no-op")
    d64 = make_image(rs, H, W, np.float64); i64 = d64 * 0 + 5
    assert_bits_equal(dmc.binalyWeightedRangeFilter(d64, i64.copy(), (5, 5), 10, dmc.FULL_KERNEL), i64, "64F no-op")
    # in place
    c = b.copy(); dmc.binalyWeightedRangeFilter(c, c, (7, 7), 10, dmc.FULL_KERNEL)
    assert_bits_equal(c, port.bwrf(b, 7, 7, 10), "8u in-place")
    f = make_image(rs, H, W, np.float32); c = f.copy(); dmc.binalyWeightedRangeFilter(c, c, (7, 7), 30.0, dmc.FULL_KERNEL)
    assert_bits_equal(c, port.bwrf(f, 7, 7, 30.0), "32f in-place")
    # FULL_KERNEL_PAIR on 16-bit/float: documented to return the FULL_KERNEL result (no parity claim vs the racy reference)
    assert_bits_equal(dmc.binalyWeightedRangeFilter(f, None, (5, 5), 8.0, dmc.FULL_KERNEL_PAIR), port.bwrf(f, 5, 5, 8.0), "PAIR == FULL")


def test_bwrf_type_assert(dmc):
    a = np.zeros((8, 8, 2), np.uint8)
    with pytest.raises(dmc.DmcError):      # CV_Assert(type == 8UC1 || 8UC3)
        dmc.binalyWeightedRangeFilter(a, None, (3, 3), 10, dmc.FULL_KERNEL)
    with pytest.raises(dmc.DmcError):      # CV_Assert(src.size() == dst.size()) -- via the C ABI directly
        from depthmapcompression_b200.filters import _img, lib
        ctx = dmc.default_context(); s = _img(np.zeros((8, 8), np.uint8)); d = _img(np.zeros((8, 9), np.uint8))
        ctx.check(lib.dmc_bwrf(ctx.h, C.byref(s), C.byref(d), 3, 3, 10.0, 0, 1))


def test_bwrf_inf_nan_propagation(dmc, port):
    rs = np.random.RandomState(23)
    a = make_image(rs, 40, 44, np.float32)
    a[10, 10] = np.inf; a[20, 30] = -np.inf; a[5, 40] = np.nan
    for k in (3, 5, 7):
        got = dmc.binalyWeightedRangeFilter(a, None, (k, k), 30.0, dmc.FULL_KERNEL)
        assert_bits_equal(got, port.bwrf(a, k, k, 30.0), "inf/nan k%d" % k)
    d = np.zeros((33, 48), np.uint8); d[3:20, 5:30] = 90; d[8, 8] = 0
    pfs = dmc.PostFilterSet()
    assert_bits_equal(pfs.filterDisp8U2Depth32F(d, None, 75, 575, 2.6, 0, 0, 0, 2, 65.0), port.filter_disp8u_depth32f(d, 75, 575, 2.6, 0, 0, 0, 2, 65.0), "inf depth32F")
    assert_bits_equal(pfs.filterDisp8U2Depth16U(d, None, 75, 575, 2.6, 0, 0, 0, 2, 65.0), port.filter_disp8u_depth16u(d, 75, 575, 2.6, 0, 0, 0, 2, 65.0), "inf depth16U")


@pytest.mark.parametrize("shape", SHAPES[:6])
def test_brf_and_minmax_filters(dmc, port, shape):
    rs = np.random.RandomState(24); H, W = shape
    for dt in (np.uint8, np.uint16, np.int16, np.float32, np.float64):
        for kind in ("pw", "const", "noise"):
            b = make_image(rs, H, W, dt, kind=kind)
            for (kw, kh, f, c, s) in [(1, 1, 1, 1, 1), (3, 3, 1, 1, 1), (7, 7, 1, 1, 1), (13, 13, 1, 1, 1), (5, 9, 0.5, 2, 1.5), (9, 5, 0, 0, 0), (21, 21, 1, 1, 1)]:
                if kind == "noise" and kw > 7:
                    continue
                assert_bits_equal(dmc.boundaryReconstructionFilter(b, None, (kw, kh), f, c, s), port.brf(b, kw, kh, f, c, s), "brf %dx%d %s %s" % (kw, kh, dt.__name__, kind))
        b = make_image(rs, H, W, dt); c = b.copy(); dmc.boundaryReconstructionFilter(c, c, (7, 7), 1, 1, 1)
        assert_bits_equal(c, port.brf(b, 7, 7, 1, 1, 1), "brf in-place")
    for dt in (np.uint8, np.uint16, np.int16, np.float32):
        b = make_image(rs, H, W, dt)
        for neg in ((False, True) if dt == np.float32 else (False,)):
            bb = b - 300 if neg else b      # negative floats: the FLT_MIN seed of maxFilter leaks (minmaxFilter.cpp:332)
            for (kw, kh) in [(3, 3), (7, 5), (1, 3), (3, 1), (1, 1)]:
                assert_bits_equal(dmc.maxFilter(bb, None, (kw, kh)), port.max_filter(bb, kw, kh), "maxFilter %s" % dt.__name__)
                assert_bits_equal(dmc.minFilter(bb, None, (kw, kh)), port.min_filter(bb, kw, kh), "minFilter %s" % dt.__name__)


def test_converters_fill_reproject(dmc, port):
    rs = np.random.RandomState(25)
    for (H, W) in [(16, 16), (7, 9), (33, 21), (48, 64), (480, 640)]:
        d8 = make_image(rs, H, W, kind="noise")
        d16 = (rs.randint(0, 65536, size=(H, W))).astype(np.uint16); d16[rs.rand(H, W) < 0.2] = 0
        s16 = (rs.randint(-3000, 3000, size=(H, W))).astype(np.int16)
        f32 = (rs.rand(H, W) * 5000).astype(np.float32); f32[rs.rand(H, W) < 0.1] = 0
        for (a, b) in [(2.6, 0.0), (1.0, 0.0), (2.6, 3.5)]:
            init = (rs.rand(H, W) * 9).astype(np.float32)
            assert_bits_equal(dmc.disp8U2depth32F(d8, init.copy(), 43125.0, a, b), port.disp8u2depth32f(d8, 43125.0, a, b, dst=init), "disp8U2depth32F")
            assert_bits_equal(dmc.depth32F2disp8U(f32, None, 43125.0, a, b), port.depth32f2disp8u(f32, 43125.0, a, b), "depth32F2disp8U")
            assert_bits_equal(dmc.depth16U2disp8U(d16, None, 43125.0, a, b), port.depth16u2disp8u(d16, 43125.0, a, b), "depth16U2disp8U")
            assert_bits_equal(dmc.disp16S2depth16U(s16, None, 43125.0, a, b), port.disp16s2depth16u(s16, 43125.0, a, b), "disp16S2depth16U")
        for dt in (np.uint8, np.uint16, np.int16, np.float32):
            img = make_image(rs, H, W, dt); img[rs.rand(H, W) < 0.3] = 0; img[-1] = 9
            if W > 2:
                assert_bits_equal(dmc.fillOcclusion(img.copy(), 0, dmc.FILL_DISPARITY), port.fill_occlusion(img, 0, 0), "fill disparity")
                img2 = img.copy(); img2[img2 == 0] = 1; img2[rs.rand(H, W) < 0.3] = 7; img2[-1] = 9
                assert_bits_equal(dmc.fillOcclusion(img2.copy(), 7, dmc.FILL_DEPTH), port.fill_occlusion(img2, 7, 1), "fill depth")
            assert_bits_equal(dmc.reprojectXYZ(img, None, 510.0).reshape(-1, 3), port.reproject_xyz(img, 510.0), "reprojectXYZ")


@pytest.mark.parametrize("shape", [(48, 64), (37, 53), (9, 150), (480, 640)])
def test_post_filter_set_entry_points(dmc, port, shape):
    rs = np.random.RandomState(26); H, W = shape
    pfs = dmc.PostFilterSet()
    for trial in range(3):
        a = np.maximum(make_image(rs, H, W, kind=("pw", "noise", "pw")[trial]), 1)
        for (mr, gr, mmr, br, th) in [(2, 1, 3, 5, 10), (1, 0, 1, 3, 10), (0, 0, 0, 0, 0), (3, 2, 2, 4, 30), (1, 3, 0, 7, 255), (10, 10, 10, 10, 20)]:
            if (mr == 10 and (H > 100 or trial)):
                continue
            for meth in (dmc.FULL_KERNEL, dmc.SEPARABLE_KERNEL):
                assert_bits_equal(pfs(a, None, mr, gr, mmr, br, th, meth), port.post_filter_set(a, mr, gr, mmr, br, th, meth), "operator() %s m%d" % ((mr, gr, mmr, br, th), meth))
                assert_bits_equal(pfs.filterDisp8U2Depth32F(a, None, 75, 575, 2.6, mr, gr, mmr, br, th * 6.5, meth),
                                  port.filter_disp8u_depth32f(a, 75, 575, 2.6, mr, gr, mmr, br, th * 6.5, meth), "Depth32F %s m%d" % ((mr, gr, mmr, br, th), meth))
            assert_bits_equal(pfs.filterDisp8U2Depth16U(a, None, 75, 575, 2.6, mr, gr, mmr, br, th * 6.5), port.filter_disp8u_depth16u(a, 75, 575, 2.6, mr, gr, mmr, br, th * 6.5), "Depth16U")
            assert_bits_equal(pfs.filterDisp8U2Disp32F(a, None, mr, gr, mmr, br, th + 0.5), port.filter_disp8u_disp32f(a, mr, gr, mmr, br, th + 0.5), "Disp32F")
    # repeated calls on one PostFilterSet with a changing image size (scratch reallocation) and a strided source view
    big = np.maximum(make_image(rs, 120, 200), 1)
    view = big[10:90, 20:150]                     # non-dense rows: step > cols
    assert_bits_equal(pfs(view, None, 2, 1, 3, 5, 10), port.post_filter_set(np.ascontiguousarray(view), 2, 1, 3, 5, 10), "strided src")
    c = np.ascontiguousarray(view).copy(); pfs(c, c, 2, 1, 3, 5, 10)
    assert_bits_equal(c, port.post_filter_set(np.ascontiguousarray(view), 2, 1, 3, 5, 10), "operator() in-place")
    out = pfs(a, None, 1, 0, 1, 3, 10, dmc.FULL_KERNEL_PAIR) if False else None     # 8U + PAIR leaves dest unspecified in the reference
    assert out is None


def test_full_size_1080p_and_batch(dmc, port):
    """BASELINE.json sizes: 1080p frames through the batched entry point (device-resident and host-streamed) equal
    the oracle frame by frame; sharding covers every frame exactly once."""
    import torch
    from oracle.oracle_py import synth_disp, degrade_blocks
    from depthmapcompression_b200.filters import chain_params
    from depthmapcompression_b200 import capi
    H, W, N = 1080, 1920, 6
    frames = np.stack([degrade_blocks(synth_disp(H, W, 1000 + f, shift=(2 * f, f)), f) for f in range(N)])
    ctx = dmc.default_context()
    for chain, params, odt in [(capi.CHAIN_DISP8U, (2, 1, 3, 5, 10), np.uint8), (capi.CHAIN_DISP8U, (1, 0, 1, 3, 10), np.uint8),
                               (capi.CHAIN_DEPTH32F, (1, 0, 1, 3, 65), np.float32)]:
        p = chain_params(chain, *params, focus=FOCUS, baseline=BASELINE, amp=AMP)
        if chain == capi.CHAIN_DISP8U:
            want = np.stack([port.post_filter_set(f, *params) for f in frames[:3]])
        else:
            want = np.stack([port.filter_disp8u_depth32f(f, FOCUS, BASELINE, AMP, *params) for f in frames[:3]])
        # host-streamed (pageable numpy memory)
        out_h = np.zeros((N, H, W), odt)
        ctx.chain_batch(frames, out_h, N, H, W, p, device=False)
        assert_bits_equal(out_h[:3], want, "host batch")
        # device-resident
        d_in = torch.from_numpy(frames).cuda()
        d_out = torch.zeros((N, H, W), dtype={np.uint8: torch.uint8, np.float32: torch.float32}[odt], device="cuda")
        torch.cuda.synchronize()
        ctx.chain_batch(d_in.data_ptr(), d_out.data_ptr(), N, H, W, p, device=True)
        ctx.synchronize()
        assert_bits_equal(d_out.cpu().numpy(), out_h, "device batch == host batch")
    # the same chain on arrays of image descriptors: separately allocated frames, some with a row stride, some device-resident
    p8 = chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10)
    want8 = np.zeros((N, H, W), np.uint8); ctx.chain_batch(frames, want8, N, H, W, p8, device=False)
    wide = np.zeros((H, W + 40), np.uint8); wide[:, :W] = frames[1]
    srcs = [frames[0].copy(), wide[:, :W]] + [frames[i].copy() for i in range(2, N)]
    owide = np.zeros((H, W + 24), np.uint8)
    dsts = [np.zeros((H, W), np.uint8), owide[:, :W]] + [np.zeros((H, W), np.uint8) for _ in range(2, N)]
    ctx.chain_batch_images(srcs, dsts, p8)
    for i in range(N):
        assert_bits_equal(np.ascontiguousarray(dsts[i]), want8[i], "descriptor batch, frame %d" % i)
    assert not owide[:, W:].any()                                   # the padding of a strided dst is not touched
    pd = chain_params(capi.CHAIN_DEPTH32F, 1, 0, 1, 3, 65, focus=FOCUS, baseline=BASELINE, amp=AMP)
    d32 = [np.zeros((H, W), np.float32) for _ in range(3)]
    ctx.chain_batch_images(srcs[:3], d32, pd)
    for i in range(3):
        assert_bits_equal(d32[i], port.filter_disp8u_depth32f(frames[i], FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65), "descriptor batch depth32f %d" % i)
    with pytest.raises(dmc.DmcError):
        ctx.chain_batch_images(srcs[:2], [np.zeros((H, W), np.uint8), np.zeros((H, W - 1), np.uint8)], p8)
    # many tiny frames in one call (more frames than one launch can take in gridDim.z)
    tiny = np.random.RandomState(5).randint(1, 256, size=(70000, 8, 12)).astype(np.uint8)
    out_t = np.zeros_like(tiny)
    ctx.chain_batch(tiny, out_t, tiny.shape[0], 8, 12, chain_params(capi.CHAIN_DISP8U, 1, 0, 1, 1, 10), device=False)
    for i in (0, 1, 65534, 65535, 65536, 69999):
        assert_bits_equal(out_t[i], port.post_filter_set(tiny[i], 1, 0, 1, 1, 10), "tiny frame %d" % i)
    # the in-process multi-GPU frame-batch scheduler (here: every visible device, plus two contexts on device 0)
    import torch as _t
    p8 = chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10)
    want8 = np.zeros((N, H, W), np.uint8); ctx.chain_batch(frames, want8, N, H, W, p8, device=False)
    for devs in ([0, 0], list(range(_t.cuda.device_count())), [0, 0, 0, 0, 0, 0, 0]):      # 7 shards over 6 frames: one is empty
        got8 = np.zeros((N, H, W), np.uint8)
        dmc.multi_chain_batch(devs, frames, got8, p8)
        assert_bits_equal(got8, want8, "multi_chain_batch %s" % devs)
        sched = dmc.FrameBatchScheduler(devs)
        for rep in range(2):
            got8[:] = 0; sched.chain_batch(frames, got8, N, H, W, p8)
            assert_bits_equal(got8, want8, "FrameBatchScheduler %s" % devs)
        sched.close()
    # frame sharding: contiguous, disjoint, complete
    for n in (0, 1, 7, 1000):
        for world in (1, 2, 4, 8):
            seen = []
            for r in range(world):
                b, c = dmc.shard_frames(n, r, world); seen += list(range(b, b + c))
            assert seen == list(range(n))


def test_batched_depth16u_and_disp32f_chains(dmc, port):
    """dmc_chain_batch with CHAIN_DEPTH16U / CHAIN_DISP32F at batch sizes > 1 (VERDICT r01: only single frames were tested):
    host-streamed and device-resident, a batch larger than one 256 MiB frame group, ragged frame sizes, through the
    descriptor entry point and through the scheduler."""
    import torch
    from depthmapcompression_b200.filters import chain_params
    from depthmapcompression_b200 import capi
    rs = np.random.RandomState(77)
    ctx = dmc.default_context()
    for (H, W, N) in [(37, 53, 9), (480, 640, 5), (96, 200, 300)]:
        frames = np.stack([np.maximum(make_image(rs, H, W), 1) for _ in range(min(N, 9))])
        frames = np.ascontiguousarray(np.concatenate([frames] * ((N + len(frames) - 1) // len(frames)))[:N])
        for chain, odt, ref in [(capi.CHAIN_DEPTH16U, np.uint16, lambda f: port.filter_disp8u_depth16u(f, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0)),
                                (capi.CHAIN_DISP32F, np.uint16, lambda f: port.filter_disp8u_disp32f(f, 2, 1, 2, 4, 12.5))]:      # (CV_16U out, postFilterSet.cpp:54)
            p = chain_params(chain, *((1, 0, 1, 3, 65.0) if chain == capi.CHAIN_DEPTH16U else (2, 1, 2, 4, 12.5)), focus=FOCUS, baseline=BASELINE, amp=AMP)
            out_h = np.zeros((N, H, W), odt)
            ctx.chain_batch(frames, out_h, N, H, W, p, device=False)
            for i in sorted(set([0, 1, N // 2, N - 1])):
                assert_bits_equal(out_h[i], ref(frames[i]), "chain %d batch %d frame %d host" % (chain, N, i))
            d_in = torch.from_numpy(frames).cuda()
            d_out = torch.zeros((N, H, W), dtype=torch.int16, device="cuda")
            ctx.chain_batch(d_in.data_ptr(), d_out.data_ptr(), N, H, W, p, device=True); ctx.synchronize()
            assert_bits_equal(d_out.cpu().numpy().view(odt), out_h, "chain %d batch %d device == host" % (chain, N))
            if N <= 9:
                dsts = [np.zeros((H, W), odt) for _ in range(N)]
                ctx.chain_batch_images([f.copy() for f in frames], dsts, p)
                assert_bits_equal(np.stack(dsts), out_h, "chain %d descriptor batch" % chain)
    # a batch of 1080p frames that spans more than one frame group (group = 256 MiB of input = 129 frames) with a float output
    H, W, N = 1080, 1920, 140
    base = np.maximum(make_image(rs, H, W), 1)
    d_in = torch.from_numpy(base).cuda()[None].repeat(N, 1, 1).contiguous(); d_in[N - 1] = torch.flip(d_in[0], dims=(1,)); d_in[129] = torch.flip(d_in[0], dims=(0,))
    d_out = torch.zeros((N, H, W), dtype=torch.int16, device="cuda")
    p = chain_params(capi.CHAIN_DEPTH16U, 1, 0, 1, 3, 65.0, focus=FOCUS, baseline=BASELINE, amp=AMP)
    ctx.chain_batch(d_in.data_ptr(), d_out.data_ptr(), N, H, W, p, device=True); ctx.synchronize()
    for i, f in ((0, base), (128, base), (129, base[::-1]), (N - 1, base[:, ::-1])):
        assert_bits_equal(d_out[i].cpu().numpy().view(np.uint16), port.filter_disp8u_depth16u(np.ascontiguousarray(f), FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0), "1080p depth16U batch frame %d" % i)


def test_full_size_4k_multiview_config(dmc, port):
    """BASELINE.json configs[3]: 3840x2160 16-bit depth + RGB, binary weighted range filter radius sweep.  Full-size
    frames against the oracle for r = 1, 5 (the r = 5 float path exercises the reference's padding quirk: cols % 4 == 0)."""
    from oracle.oracle_py import synth_disp
    H, W = 2160, 3840
    rs = np.random.RandomState(41)
    base = synth_disp(H, W, 3)
    d16 = base.astype(np.uint16) * 16 + rs.randint(0, 16, size=(H, W)).astype(np.uint16)
    for r in (1, 5):
        k = 2 * r + 1
        assert_bits_equal(dmc.binalyWeightedRangeFilter(d16, None, (k, k), 160.0, dmc.FULL_KERNEL), port.bwrf(d16, k, k, 160.0), "4K 16U r%d" % r)
    rgb = np.stack([base, np.roll(base, 7, 1), np.roll(base, 11, 0)], axis=2)
    rgb = np.clip(rgb.astype(np.int16) + rs.randint(-4, 5, size=rgb.shape), 0, 255).astype(np.uint8)
    assert_bits_equal(dmc.binalyWeightedRangeFilter(rgb, None, (7, 7), 30.0, dmc.FULL_KERNEL), port.bwrf(rgb, 7, 7, 30.0), "4K 8UC3 r3")
    # config 5 at full size: 1080p chain -> reprojectXYZ
    img = np.maximum(make_image(rs, 1080, 1920), 1)
    pfs = dmc.PostFilterSet()
    d32 = pfs.filterDisp8U2Depth32F(img, None, 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0)
    assert_bits_equal(d32, port.filter_disp8u_depth32f(img, 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0), "1080p Depth32F")
    assert_bits_equal(dmc.reprojectXYZ(d32, None, 510.0).reshape(-1, 3), port.reproject_xyz(d32, 510.0), "1080p reprojectXYZ")


def test_single_frame_graph_replay(dmc, port):
    """Repeated identical device-resident single-frame calls are replayed from a CUDA graph (SURVEY 7.1-6): the result
    must follow the buffers' CONTENTS, parameter changes, and survive scratch reallocation by a larger frame."""
    import ctypes as C
    import torch
    from depthmapcompression_b200 import capi
    from depthmapcompression_b200.capi import DmcImage, lib
    ctx = dmc.default_context()
    rs = np.random.RandomState(41)

    def run(d_in, d_out, H, W, args):
        si, so = DmcImage(d_in.data_ptr(), H, W, capi.CV_8U, 0, capi.MEM_DEVICE), DmcImage(d_out.data_ptr(), H, W, capi.CV_8U, 0, capi.MEM_DEVICE)
        ctx.check(lib.dmc_post_filter_set(ctx.h, C.byref(si), C.byref(so), *args, 0)); ctx.synchronize()
        return d_out.cpu().numpy()

    H, W = 120, 200
    a = np.maximum(make_image(rs, H, W), 1)
    d_in = torch.from_numpy(a).cuda(); d_out = torch.zeros((H, W), dtype=torch.uint8, device="cuda")
    n0 = ctx.kernel_launches
    for i in range(5):
        assert_bits_equal(run(d_in, d_out, H, W, (2, 1, 3, 5, 10)), port.post_filter_set(a, 2, 1, 3, 5, 10), "repeat %d" % i)
    assert ctx.kernel_launches - n0 == 5 * 4                  # four kernels per call, replayed or not
    b = np.maximum(make_image(rs, H, W, kind="noise"), 1)
    d_in.copy_(torch.from_numpy(b).cuda())                      # same pointers, new contents
    assert_bits_equal(run(d_in, d_out, H, W, (2, 1, 3, 5, 10)), port.post_filter_set(b, 2, 1, 3, 5, 10), "new contents")
    for i in range(3):                                          # new parameters: new graph
        assert_bits_equal(run(d_in, d_out, H, W, (1, 0, 1, 3, 7)), port.post_filter_set(b, 1, 0, 1, 3, 7), "new parameters %d" % i)
    H2, W2 = 400, 700                                           # larger frame: scratch buffers are reallocated
    c = np.maximum(make_image(rs, H2, W2), 1)
    e_in = torch.from_numpy(c).cuda(); e_out = torch.zeros((H2, W2), dtype=torch.uint8, device="cuda")
    for i in range(3):
        assert_bits_equal(run(e_in, e_out, H2, W2, (2, 1, 3, 5, 10)), port.post_filter_set(c, 2, 1, 3, 5, 10), "larger frame %d" % i)
    for i in range(3):
        assert_bits_equal(run(d_in, d_out, H, W, (1, 0, 1, 3, 7)), port.post_filter_set(b, 1, 0, 1, 3, 7), "back to the small frame %d" % i)


def test_pinned_host_images_zero_copy(dmc, port):
    """Host images in pinned memory (dmc_host_alloc / dmc_host_register) are filtered in place over the host link and the
    repeated call is replayed from a CUDA graph: results follow the contents, in-place calls and strided views still
    work, every single-image operator accepts them, and unregistered memory goes back to the copying path."""
    rs = np.random.RandomState(43)
    ctx = dmc.default_context()
    H, W = 120, 200
    a = np.maximum(make_image(rs, H, W), 1)
    p_in = dmc.pinned_empty((H, W), np.uint8); p_out = dmc.pinned_empty((H, W), np.uint8); p_f = dmc.pinned_empty((H, W), np.float32)
    pfs = dmc.PostFilterSet()
    replays0 = ctx.kernel_launches
    for i in range(5):
        p_in[:] = np.roll(a, i, axis=1)                         # same pointers, new contents
        got = pfs(p_in, p_out, 2, 1, 3, 5, 10)
        assert got is p_out
        assert_bits_equal(p_out, port.post_filter_set(np.roll(a, i, axis=1), 2, 1, 3, 5, 10), "pinned repeat %d" % i)
        pfs.filterDisp8U2Depth32F(p_in, p_f, 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0)
        assert_bits_equal(p_f, port.filter_disp8u_depth32f(np.roll(a, i, axis=1), 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0), "pinned depth32F %d" % i)
    assert ctx.kernel_launches - replays0 == 5 * (4 + 3)
    p_in[:] = a
    pfs(p_in, p_in, 2, 1, 3, 5, 10)                             # in place on pinned memory
    assert_bits_equal(p_in, port.post_filter_set(a, 2, 1, 3, 5, 10), "pinned in place")
    p_in[:] = a
    v = p_in[3:-5, 8:-2]                                        # strided view: copied, not mapped
    assert_bits_equal(pfs(v, None, 1, 0, 1, 3, 7), port.post_filter_set(np.ascontiguousarray(a[3:-5, 8:-2]), 1, 0, 1, 3, 7), "pinned strided view")
    assert_bits_equal(dmc.boundaryReconstructionFilter(p_in, p_out, (7, 7), 1, 1, 1), port.brf(a, 7, 7, 1, 1, 1), "pinned brf")
    assert_bits_equal(dmc.binalyWeightedRangeFilter(p_in, p_out, (7, 7), 10, dmc.FULL_KERNEL), port.bwrf(a, 7, 7, 10), "pinned bwrf")
    assert_bits_equal(dmc.blurRemoveMinMax(p_in, p_in, 2), port.blur_remove_minmax(a, 2), "pinned minmax in place")
    r_in = a.copy(); r_out = np.zeros((H, W), np.uint8)
    dmc.host_register(r_in); dmc.host_register(r_out)
    try:
        for i in range(3):
            assert_bits_equal(pfs(r_in, r_out, 2, 1, 3, 5, 10), port.post_filter_set(a, 2, 1, 3, 5, 10), "registered %d" % i)
    finally:
        dmc.host_unregister(r_in); dmc.host_unregister(r_out)
    assert_bits_equal(pfs(r_in, r_out, 2, 1, 3, 5, 10), port.post_filter_set(a, 2, 1, 3, 5, 10), "after unregister")
    big = dmc.pinned_empty((1080, 1920), np.uint8); big[:] = np.maximum(make_image(rs, 1080, 1920), 1)    # above the in-place limit: copied
    assert_bits_equal(pfs(big, None, 1, 0, 1, 3, 7)[:64], port.post_filter_set(big, 1, 0, 1, 3, 7)[:64], "pinned large")


def test_overlapping_device_views(dmc, port):
    """src and dst that overlap PARTIALLY in device memory (offset views of one buffer) must behave like separate buffers
    (ADVICE r01: aliasing used to be detected by pointer equality only)."""
    import ctypes as C
    import torch
    from depthmapcompression_b200 import capi
    from depthmapcompression_b200.capi import DmcImage, lib
    ctx = dmc.default_context()
    rs = np.random.RandomState(43)
    H, W = 96, 160
    a = np.maximum(make_image(rs, H, W), 1)
    want = port.post_filter_set(a, 2, 1, 3, 5, 10)
    want_bwrf = port.bwrf(a, 11, 11, 10.0, 0)
    for shift in (W * 5, W * 40 + 16, -W * 7):          # dst starts `shift` bytes after (before) src inside one allocation
        buf = torch.zeros(H * W * 3, dtype=torch.uint8, device="cuda")
        s0 = H * W; d0 = s0 + shift
        buf[s0:s0 + H * W] = torch.from_numpy(a.ravel()).cuda()
        si = DmcImage(buf.data_ptr() + s0, H, W, capi.CV_8U, 0, capi.MEM_DEVICE); so = DmcImage(buf.data_ptr() + d0, H, W, capi.CV_8U, 0, capi.MEM_DEVICE)
        ctx.check(lib.dmc_post_filter_set(ctx.h, C.byref(si), C.byref(so), 2, 1, 3, 5, 10, 0)); ctx.synchronize()
        assert_bits_equal(buf[d0:d0 + H * W].cpu().numpy().reshape(H, W), want, "chain, overlapping views shift %d" % shift)
        buf[s0:s0 + H * W] = torch.from_numpy(a.ravel()).cuda()
        ctx.check(lib.dmc_bwrf(ctx.h, C.byref(si), C.byref(so), 11, 11, C.c_float(10.0), 0, capi.BORDER_REPLICATE)); ctx.synchronize()
        assert_bits_equal(buf[d0:d0 + H * W].cpu().numpy().reshape(H, W), want_bwrf, "bwrf, overlapping views shift %d" % shift)
    # frame batches: dst batch shifted by half a frame against src
    N = 3
    frames = np.stack([np.maximum(make_image(rs, H, W), 1) for _ in range(N)])
    wantb = np.stack([port.post_filter_set(f, 1, 0, 1, 3, 10) for f in frames])
    buf = torch.zeros(H * W * (N + 2), dtype=torch.uint8, device="cuda")
    s0 = H * W; d0 = s0 + H * W // 2
    buf[s0:s0 + N * H * W] = torch.from_numpy(frames.ravel()).cuda()
    p = dmc.filters.chain_params(capi.CHAIN_DISP8U, 1, 0, 1, 3, 10)
    ctx.chain_batch(buf.data_ptr() + s0, buf.data_ptr() + d0, N, H, W, p, device=True); ctx.synchronize()
    assert_bits_equal(buf[d0:d0 + N * H * W].cpu().numpy().reshape(N, H, W), wantb, "chain batch, overlapping views")


def test_gateway_routing(dmc, port):
    """dmc_set_gateway: the host traffic of a batch runs over another device's link, the kernels read / write that
    device's HBM over NVLink.  Results must not change.  Needs two GPUs with peer access (skipped on a one-GPU box)."""
    from depthmapcompression_b200 import capi
    if capi.lib.dmc_device_count() < 2:
        pytest.skip("needs two GPUs")
    rs = np.random.RandomState(47)
    H, W, N = 270, 480, 37
    frames = np.stack([np.maximum(make_image(rs, H, W), 1) for _ in range(N)])
    p = dmc.filters.chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10)
    ctx = dmc.Context(0)
    plain = np.zeros_like(frames); ctx.chain_batch(frames, plain, N, H, W, p, device=False)
    for i in (0, N // 2, N - 1):
        assert_bits_equal(plain[i], port.post_filter_set(frames[i], 2, 1, 3, 5, 10), "own link, frame %d" % i)
    ctx.set_gateway(1)
    assert ctx.gateway == 1
    for rep in range(3):                       # repeated: buffers and events are reused across calls
        routed = np.zeros_like(frames); ctx.chain_batch(frames, routed, N, H, W, p, device=False)
        assert_bits_equal(routed, plain, "through the gateway, repetition %d" % rep)
    p32 = dmc.filters.chain_params(capi.CHAIN_DEPTH32F, 1, 0, 1, 3, 65.0, focus=75.0, baseline=575.0, amp=2.6)
    r32 = np.zeros((N, H, W), np.float32); ctx.chain_batch(frames, r32, N, H, W, p32, device=False)
    ctx.set_gateway(-1)
    assert ctx.gateway == -1
    o32 = np.zeros((N, H, W), np.float32); ctx.chain_batch(frames, o32, N, H, W, p32, device=False)
    assert_bits_equal(r32, o32, "Depth32F through the gateway")
    info = dmc.hostlink_probe([0, 1])
    assert info["all_gbs"] > 1 and len(info["gateway"]) == 2
    sched = dmc.FrameBatchScheduler([0, 1])
    out = np.zeros_like(frames); sched.chain_batch(frames, out, N, H, W, p)
    assert_bits_equal(out, plain, "scheduler over two devices")
    ctx.close()
