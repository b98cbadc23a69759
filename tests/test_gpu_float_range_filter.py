"""The 32-bit range filter, the float chains and the disparity <-> depth converters on IEEE edge values, bit for bit
against the CPU oracle (which tests/test_float_range_filter_reference.py pins on the same inputs with a numpy
restatement).

The frames of tests/_float_edge_cases.py put distances exactly on the threshold (and on its float neighbours), sums
whose low bits depend on the tap order, signed zeros, subnormals, infinities, NaN and overflowing sums at the corners,
the 128-pixel tile columns, the rows where 2R-row tiles meet, the partial right and bottom tiles, the padding quirk's
last column and column 0 of the next row.  They run through every tiled variant (radius 1..10, C1 and C3, short and
full tiles), the generic kernel (non-square windows, SEPARABLE_KERNEL), in place, the 16-bit sources' integer mode with
thresholds it must read like the float compare, the three float chains single-frame and batched, and the converters.
Only the coverage test runs without a GPU; run the rest with `-m gpu` on a B200."""
import numpy as np
import pytest

import _float_edge_cases as E
from _util import assert_bits_equal, make_image, mask_undefined
from test_gpu_tile_variants import (CHAIN_DEPTH16U, CHAIN_DEPTH32F, CHAIN_DISP32F, MARK, TABLE, run_chain_device,
                                    variant_bwrf32f)
from test_float_range_filter_reference import _port_convert, conv_init

F = np.float32
FULL_KERNEL, SEPARABLE_KERNEL = 0, 2
SMALL = (45, 260)           # 3 x 3 tiles of 128 x 16: the short variants; 260 % 4 == 0: the padding quirk at r = 5
SMALL_ODD = (45, 261)       # a last tile one column wide, no quirk
BIG = (520, 1100)           # 9 x 33 tiles at R = 8: >= 2 x 148, the full variants (and the quirk at r = 5)


def square_runs(r, cn):
    """(case, shape, thresholds) of the square window of radius r: every case and threshold on the small frames; on the
    big frame, where the C1 float kernel has a full variant of its own (r <= 5), each case's own thresholds"""
    out = []
    for case in (E.CASES_C1 if cn == 1 else E.CASES_C3):
        out.append((case, SMALL, E.all_thresholds(case)))
        if r == 5:
            out.append((case, SMALL_ODD, E.all_thresholds(case)))
        if cn == 1 and r <= 5:
            out.append((case, BIG, list(case.thresholds)))
    return out


def test_cases_reach_every_float_variant():
    """the square-window runs reach every MODE-0 entry of the single-channel tiled kernel and every entry of the
    three-channel one (test_gpu_tile_variants.TABLE)"""
    reached = set()
    for r in range(1, 11):
        for cn in (1, 3):
            for case, (H, W), ths in square_runs(r, cn):
                reached |= {variant_bwrf32f(r, float(th), "f32", 1, H, W, cn) for th in ths}
    want = {v for v in TABLE if (v[0] == "bwrf32f_tiled" and v[3] == 0) or v[0] == "bwrf32f_c3_tiled"}
    assert want and not want - reached, "not reached: %s" % sorted(want - reached)


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)          # raises loudly without a GPU / without the built library
    return m


def check(dmc, port, img, kw, kh, th, method=FULL_KERNEL, in_place=False, msg=""):
    want = port.bwrf(img, kw, kh, th, method)
    if in_place:
        got = img.copy()
        dmc.binalyWeightedRangeFilter(got, got, (kw, kh), th, method)
    else:
        got = dmc.binalyWeightedRangeFilter(img, None, (kw, kh), th, method)
    mask_undefined(got, want, kw, kh, img.shape[1], method, img.dtype.type, dmc)
    assert_bits_equal(got, want, "%s %s %dx%d m%d th %r%s" % (msg, img.shape, kw, kh, method, th, " in place" if in_place else ""))


@pytest.mark.gpu
@pytest.mark.parametrize("cn", [1, 3])
@pytest.mark.parametrize("r", range(1, 11))
def test_square_window(dmc, port, r, cn):
    k = 2 * r + 1
    for case, (H, W), ths in square_runs(r, cn):
        img = case.image(H, W)
        for th in ths:
            check(dmc, port, img, k, k, th, msg=case.name)


@pytest.mark.gpu
@pytest.mark.parametrize("cn", [1, 3])
@pytest.mark.parametrize("window", [(7, 3, FULL_KERNEL), (11, 1, FULL_KERNEL), (1, 5, FULL_KERNEL), (4, 4, FULL_KERNEL),
                                    (11, 11, SEPARABLE_KERNEL), (7, 3, SEPARABLE_KERNEL), (5, 0, SEPARABLE_KERNEL)],
                         ids=lambda w: "%dx%d-m%d" % w)
def test_generic_kernel(dmc, port, window, cn):
    """windows the tiled kernels do not take; (11, 1) and the row pass of (11, 11) carry the padding quirk on W = 260"""
    kw, kh, method = window
    for case in (E.CASES_C1 if cn == 1 else E.CASES_C3):
        for shape in (SMALL, SMALL_ODD):
            img = case.image(*shape)
            for th in E.all_thresholds(case):
                check(dmc, port, img, kw, kh, th, method, msg=case.name)


@pytest.mark.gpu
@pytest.mark.parametrize("cn", [1, 3])
def test_in_place(dmc, port, cn):
    for case in (E.CASES_C1 if cn == 1 else E.CASES_C3):
        img = case.image(*SMALL)
        for kw, kh, method in [(3, 3, FULL_KERNEL), (11, 11, FULL_KERNEL), (21, 21, FULL_KERNEL), (7, 3, FULL_KERNEL),
                               (5, 5, SEPARABLE_KERNEL)]:
            for th in case.thresholds:
                check(dmc, port, img, kw, kh, th, method, in_place=True, msg=case.name)


# ------------------------------------------------------------------------------------------------ 16-bit sources
def int_thresholds():
    """+-inf, -0.0, the smallest subnormal, k and its float neighbours around integer distances, 65535.99: the integer
    accumulation (th >= 0, r <= 9) reads |c - v| <= th as |c - v| <= floor(th), which must agree with the float compare"""
    ths = [E.INF, -E.INF, F(-0.0), E.SUB, F(65535.99), F(65535.0), F(1e9)]
    for k in (0.0, 1.0, 50.0, 200.0, 4000.0):
        ths += E.around(k)
    return ths


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.uint16, np.int16], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("r", range(1, 11))
def test_16bit_thresholds(dmc, port, r, dt):
    rs = np.random.RandomState(100 + r)
    k = 2 * r + 1
    for shape in (SMALL, SMALL_ODD):
        img = make_image(rs, shape[0], shape[1], dt)
        for th in int_thresholds():
            check(dmc, port, img, k, k, th, msg=np.dtype(dt).name)


# ------------------------------------------------------------------------------------------------ chains
FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6     # the constants of run_chain_device
MAF = F(F(AMP) * F(FOCUS * BASELINE))       # a * focal_baseline in float32 (depthmapUtil.cpp:935)
DISPS = (60, 61, 90, 91, 200, 201)


def disparity_frame(seed, H, W):
    """8 x 8 blocks of the disparities DISPS (adjacent values side by side), so that depth distances fl(maf/d1) - fl(maf/d2)
    of neighbouring blocks are known"""
    rs = np.random.RandomState(seed)
    blk = np.array(DISPS, np.uint8)[rs.randint(0, len(DISPS), size=((H + 7) // 8, (W + 7) // 8))]
    return np.ascontiguousarray(np.kron(blk, np.ones((8, 8), np.uint8))[:H, :W])


def depth_thresholds():
    """th = |fl(maf/d1) - fl(maf/d2)| for adjacent disparities, and its float neighbours"""
    ths = []
    for d1, d2 in ((60, 61), (90, 91), (200, 201)):
        ths += E.around(abs(F(MAF / F(d1)) - F(MAF / F(d2))))
    return ths


def chain_oracle(port, chain, f, br, th):
    if chain == CHAIN_DEPTH32F:
        return port.filter_disp8u_depth32f(f, FOCUS, BASELINE, AMP, 0, 0, 0, br, th)
    if chain == CHAIN_DEPTH16U:
        return port.filter_disp8u_depth16u(f, FOCUS, BASELINE, AMP, 0, 0, 0, br, th)
    return port.filter_disp8u_disp32f(f, 0, 0, 0, br, th)


def chain_single(dmc, chain, f, br, th):
    pfs = dmc.PostFilterSet()
    if chain == CHAIN_DEPTH32F:
        return pfs.filterDisp8U2Depth32F(f, None, FOCUS, BASELINE, AMP, 0, 0, 0, br, th)
    if chain == CHAIN_DEPTH16U:
        return pfs.filterDisp8U2Depth16U(f, None, FOCUS, BASELINE, AMP, 0, 0, 0, br, th)
    return pfs.filterDisp8U2Disp32F(f, None, 0, 0, 0, br, th)


def chain_runs(chain):
    """(radius, thresholds): depth chains at every radius with the depth distances; Disp32F with thresholds at and
    around integer distances, at r = 10 (the float accumulation) and with th < 0 (the float accumulation at any r)"""
    if chain == CHAIN_DISP32F:
        ints = [t for k in (0.0, 1.0, 30.0, 31.0) for t in E.around(k)]
        return [(r, ints) for r in (1, 5, 9, 10)] + [(r, [F(-1.0), -E.INF, E.NAN]) for r in (1, 5, 10)]
    return [(r, depth_thresholds() + [E.INF, F(-0.0)]) for r in range(1, 11)]


@pytest.mark.gpu
@pytest.mark.parametrize("chain", [CHAIN_DEPTH32F, CHAIN_DEPTH16U, CHAIN_DISP32F], ids=["depth32F", "depth16U", "disp32F"])
def test_chains(dmc, port, chain):
    """PostFilterSet's float chains on one frame and dmc_chain_batch on three, against the oracle's chains"""
    H, W = SMALL
    frames = np.stack([disparity_frame(7 + i, H, W) for i in range(3)])
    ctx = dmc.default_context()
    for r, ths in chain_runs(chain):
        for th in ths:
            params = (0, 0, 0, r, float(th))
            want = [chain_oracle(port, chain, f, r, th) for f in frames]
            assert_bits_equal(chain_single(dmc, chain, frames[0], r, th), want[0], "chain %d r%d th %r single" % (chain, r, th))
            got, rest = run_chain_device(dmc, ctx, frames, chain, params)
            assert (rest == MARK).all(), "chain %d r%d th %r: bytes outside the batch were written" % (chain, r, th)
            for i in range(len(frames)):
                assert_bits_equal(got[i], want[i], "chain %d r%d th %r batch frame %d" % (chain, r, th, i))


# ------------------------------------------------------------------------------------------------ converters
@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(E.CONV_SOURCES))
def test_converters(dmc, port, kind):
    fn = {"disp8u2depth32f": dmc.disp8U2depth32F, "depth32f2disp8u": dmc.depth32F2disp8U,
          "depth16u2disp8u": dmc.depth16U2disp8U, "disp16s2depth16u": dmc.disp16S2depth16U}[kind]
    for src in E.converter_arrays(kind):
        for fb, a, b in E.CONV_PARAMS:
            init = conv_init(src.shape) if kind == "disp8u2depth32f" else None
            want = _port_convert(port, kind, src, fb, a, b, init)
            got = fn(src, None if init is None else init.copy(), fb, a, b)
            assert_bits_equal(got, want, "%s n=%d fb=%r a=%r b=%r" % (kind, src.size, fb, a, b))
