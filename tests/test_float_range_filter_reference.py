"""The 32-bit range filter and the disparity <-> depth converters of the CPU oracle, pinned on IEEE edge values by a plain
numpy restatement (no GPU).

The reference build cannot be run on new inputs here, so the oracle (oracle/dmc_oracle.c) is what the GPU tests compare
with; this file checks that the oracle computes what its rules say on the adversarial inputs of tests/_float_edge_cases.py:
  * bwrf32 below restates the filter in float32, vectorised over pixels and thresholds, taps in raster order,
    BORDER_REPLICATE, C1 and C3, any window, FULL_KERNEL and SEPARABLE_KERNEL, and the padding quirk of the last column;
    it equals port.bwrf bit for bit on every case.
  * Mutants of bwrf32 (`<` for `<=`, the distance in double, c - th <= v <= c + th, another C3 order of additions, taps
    in reverse, t starting at -0.0, flush to zero, `if (w) t += v`) each differ from the oracle on some case, so the
    inputs tell those rules apart: a kernel that broke one of them would fail the GPU tests that use the same inputs.
  * convert restates the converters' SIMD body (saturating packs) and scalar tail (truncating casts) and equals the
    oracle on arrays that put NaN, infinities, signed zeros, subnormals, ties and out-of-range quotients in both parts."""
import math

import numpy as np
import pytest

import _float_edge_cases as E
from _util import assert_bits_equal, bits_equal

F = np.float32
FULL_KERNEL, SEPARABLE_KERNEL = 0, 2
MUTANTS = ["lt", "dist_f64", "interval", "c3_order", "reverse", "t_negzero", "ftz", "if_w"]


# --------------------------------------------------------------------------------------------------- the restatement
def taps(kw, kh):
    """raster order over the window, kept iff sqrt(i^2 + j^2) <= max(rV, rH) in double"""
    rH, rV = kw >> 1, kh >> 1
    rmax = max(rH, rV)
    return [(i, j) for i in range(-rV, rV + 1) for j in range(-rH, rH + 1) if math.sqrt(i * i + j * j) <= rmax]


def _flush(a):
    """flush-to-zero of subnormals, sign kept"""
    a = np.asarray(a, F)
    return np.where(np.abs(a) < E.TINY, np.copysign(F(0), a), a).astype(F)


def _pass(x, kw, kh, ths, mutant):
    """one filter pass on x: (H, W, cn) float32 -> (T, H, W, cn), for the T thresholds ths"""
    H, W, cn = x.shape
    rH, rV = kw >> 1, kh >> 1
    p = np.pad(x, ((rV, rV), (rH, rH), (0, 0)), mode="edge")
    if rH % 8 == 5 and W % 4 == 0:
        # the reference's right padding is one column short: tap (i, +rH) of the last column reads the first element
        # of the next line of its buffer (oracle/dmc_oracle.c, bwrf_32f).  C1: column 0 of the next padded row; C3
        # (planes split line by line): planes 1 and 2 of the same row, plane 0 of the next row.  No next line: the
        # replicated value stays (the reference reads past its buffer there).
        for q in range(H + 2 * rV):
            y, nxt = min(max(q - rV, 0), H - 1), min(max(q - rV + 1, 0), H - 1)
            has_next = q + 1 < H + 2 * rV
            if cn == 1:
                if has_next:
                    p[q, -1, 0] = x[nxt, 0, 0]
            else:
                p[q, -1, 0], p[q, -1, 1] = x[y, 0, 1], x[y, 0, 2]
                if has_next:
                    p[q, -1, 2] = x[nxt, 0, 0]
    th = np.asarray(ths, F).reshape(-1, 1, 1)
    if mutant == "ftz":
        x, p, th = _flush(x), _flush(p), _flush(th)
    t = np.full((len(ths), H, W, cn), F(-0.0) if mutant == "t_negzero" else F(0.0), F)
    wsum = np.zeros((len(ths), H, W), F)
    order = taps(kw, kh)
    for i, j in (order[::-1] if mutant == "reverse" else order):
        v = p[rV + i:rV + i + H, rH + j:rH + j + W]
        if mutant == "dist_f64":
            ad = np.abs(x.astype(np.float64) - v.astype(np.float64))
            d = ad[..., 0] if cn == 1 else (ad[..., 2] + ad[..., 1]) + ad[..., 0]
            w = (d <= th.astype(np.float64)).astype(F)
        elif mutant == "interval" and cn == 1:
            c, vv = x[..., 0], v[..., 0]
            w = ((c - th <= vv) & (vv <= c + th)).astype(F)
        else:
            ad = np.abs(x - v)
            if mutant == "ftz":
                ad = _flush(ad)
            if cn == 1:
                d = ad[..., 0]
            elif mutant == "c3_order":
                d = (ad[..., 0] + ad[..., 1]) + ad[..., 2]
            else:
                d = (ad[..., 2] + ad[..., 1]) + ad[..., 0]
            if mutant == "ftz":
                d = _flush(d)
            w = (d < th if mutant == "lt" else d <= th).astype(F)
        if mutant == "if_w":
            t = np.where(w[..., None] != 0, t + v, t)
        else:
            t = t + w[..., None] * v
        if mutant == "ftz":
            t = _flush(t)
        wsum = wsum + w
    out = t / wsum[..., None]
    return _flush(out) if mutant == "ftz" else out


def bwrf32(src, kw, kh, ths, method=FULL_KERNEL, mutant=None):
    """binalyWeightedRangeFilter on a 32FC1 / 32FC3 image for each threshold of ths -> (T,) + src.shape"""
    x = np.asarray(src, F)
    x3 = x.reshape(x.shape[0], x.shape[1], -1)
    T = len(ths)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        if method == SEPARABLE_KERNEL:
            if kw <= 1:
                out = np.broadcast_to(x3, (T,) + x3.shape).copy()
            else:
                h = _pass(x3, kw, 1, ths, mutant)
                out = h if kh == 0 else np.stack([_pass(h[k], 1, kh, ths[k:k + 1], mutant)[0] for k in range(T)])
        elif kw == 0 or kh == 0:
            out = np.broadcast_to(x3, (T,) + x3.shape).copy()
        else:
            out = _pass(x3, kw, kh, ths, mutant)
    return out.reshape((T,) + x.shape)


# --------------------------------------------------------------------------------------------------- filter cases
SHAPES = [(21, 36), (20, 37)]           # 36 % 4 == 0: the padding quirk at rH = 5
SQUARE = [(2 * r + 1, 2 * r + 1, FULL_KERNEL) for r in range(1, 11)]
WINDOWS = [(7, 3, FULL_KERNEL), (11, 1, FULL_KERNEL), (1, 5, FULL_KERNEL), (4, 4, FULL_KERNEL), (0, 3, FULL_KERNEL),
           (1, 1, FULL_KERNEL), (11, 11, SEPARABLE_KERNEL), (7, 3, SEPARABLE_KERNEL), (5, 0, SEPARABLE_KERNEL),
           (1, 5, SEPARABLE_KERNEL)]


def _runs(cn, windows, shapes=SHAPES):
    for case in (E.CASES_C1 if cn == 1 else E.CASES_C3):
        for H, W in shapes:
            img = case.image(H, W)
            for kw, kh, method in windows:
                yield case, img, kw, kh, method


@pytest.mark.parametrize("cn", [1, 3])
@pytest.mark.parametrize("windows", ["square", "other"])
def test_restatement_equals_oracle(port, cn, windows):
    for case, img, kw, kh, method in _runs(cn, SQUARE if windows == "square" else WINDOWS):
        ths = E.all_thresholds(case)
        want = bwrf32(img, kw, kh, ths, method)
        for k, th in enumerate(ths):
            assert_bits_equal(want[k], port.bwrf(img, kw, kh, th, method),
                              "%s %s %dx%d m%d th %r" % (case.name, img.shape, kw, kh, method, th))


def _differs(port, mutant):
    """the first (case, window, threshold) where the mutant and the oracle disagree, or None"""
    for cn in ((1,) if mutant == "interval" else (3,) if mutant == "c3_order" else (1, 3)):
        for case, img, kw, kh, method in _runs(cn, SQUARE[:3] + WINDOWS[:2] + [WINDOWS[6]], SHAPES[:1]):
            ths = E.all_thresholds(case)
            got = bwrf32(img, kw, kh, ths, method, mutant)
            for k, th in enumerate(ths):
                if not bits_equal(got[k], port.bwrf(img, kw, kh, th, method)):
                    return case.name, kw, kh, method, th
    return None


@pytest.mark.parametrize("mutant", MUTANTS)
def test_mutant_differs_from_oracle(port, mutant):
    """the inputs are adversarial: a restatement with one rule changed disagrees with the oracle somewhere"""
    assert _differs(port, mutant) is not None, "no case tells the mutant %r from the oracle" % mutant


def test_mutants_are_told_apart_by_the_case_made_for_them(port):
    """each rule is decided by the family built for it, not only by accident of another family"""
    want = {"lt": "round", "dist_f64": "round", "interval": "round", "c3_order": "c3_order", "reverse": "sum_order",
            "t_negzero": "signed_zeros", "ftz": "subnormal", "if_w": "nan_inf"}
    for mutant, family in want.items():
        for cn in ((3,) if mutant == "c3_order" else (1,)):
            case = next(c for c in (E.CASES_C1 if cn == 1 else E.CASES_C3) if c.name.startswith(family))
            img = case.image(*SHAPES[0])
            ths = E.all_thresholds(case)
            got, ok = bwrf32(img, 3, 3, ths, FULL_KERNEL, mutant), bwrf32(img, 3, 3, ths)
            assert any(not bits_equal(got[k], ok[k]) for k in range(len(ths))), (mutant, case.name)


def test_in_place_and_prefilled_dst(port):
    """the oracle's result does not depend on what dst held"""
    case = E.CASES_C1[0]
    img = case.image(*SHAPES[0])
    for th in case.thresholds:
        want = bwrf32(img, 5, 5, [th])[0]
        assert_bits_equal(port.bwrf(img, 5, 5, th, FULL_KERNEL, dst_init=img), want, "dst = src contents")


# --------------------------------------------------------------------------------------------------- converters
INT_MIN = -2 ** 31


def cvround(v):
    """cvRound / cvtps2dq: round half to even; NaN or outside [-2^31, 2^31) -> INT_MIN"""
    v = np.asarray(v, F)
    ok = (v >= F(-2.0 ** 31)) & (v < F(2.0 ** 31))
    return np.where(ok, np.rint(np.where(ok, v, F(0))).astype(np.int64), INT_MIN)


def convert(kind, src, fb, a, b, dst=None):
    """the converters of depthmapUtil.cpp: elements [0, 16 (n / 16)) follow the SIMD body, the rest the scalar tail"""
    s = np.asarray(src).reshape(-1)
    n = s.size
    sse = n // 16 * 16
    fb, a, b = F(fb), F(a), F(b)
    maf = F(a * fb)
    body, tail = slice(0, sse), slice(sse, n)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        if kind == "disp8u2depth32f":
            out = np.zeros(n, F) if dst is None else np.array(dst, F).reshape(-1).copy()
            sf = s.astype(F)
            if b == 0:
                out[body] = maf / sf[body]
                out[tail] = maf / sf[tail] + b
            else:       # SIMD body commented out in the reference: the tail loop converts the FIRST n % 16 elements
                out[:n - sse] = maf / sf[:n - sse] + b
            return out.reshape(np.shape(src))
        if kind == "depth16u2disp8u":
            sf = np.concatenate([s[body].view(np.int16).astype(F), s[tail].astype(F)])      # sign-extending SIMD load
        else:
            sf = s.astype(F)
        v = maf / sf
        vb = v + b
        ib = cvround(vb[body] if b != 0 else v[body])
        it = cvround(vb[tail])
        if kind == "disp16s2depth16u":
            out = np.concatenate([np.clip(ib, -32768, 32767) & 0xFFFF, it & 0xFFFF]).astype(np.uint16)
        else:
            out = np.concatenate([np.clip(np.clip(ib, -32768, 32767), 0, 255), it & 0xFF]).astype(np.uint8)
    return out.reshape(np.shape(src))


def _port_convert(port, kind, src, fb, a, b, dst=None):
    if kind == "disp8u2depth32f":
        return port.disp8u2depth32f(src, fb, a, b, dst=dst)
    return getattr(port, kind)(src, fb, a, b)


def conv_init(shape):
    return (np.arange(int(np.prod(shape)), dtype=F).reshape(shape) * F(0.25) - F(3))


@pytest.mark.parametrize("kind", sorted(E.CONV_SOURCES))
def test_converter_restatement_equals_oracle(port, kind):
    arrays = E.converter_arrays(kind)
    assert {a.size % 16 for a in arrays} == {0, 1, 15}
    tails = set()
    for src in arrays:
        tails |= set(src.reshape(-1)[src.size // 16 * 16:].view(np.uint8 if src.dtype == np.uint8 else "u%d" % src.itemsize).tolist())
        for fb, a, b in E.CONV_PARAMS:
            init = conv_init(src.shape) if kind == "disp8u2depth32f" else None
            want = _port_convert(port, kind, src, fb, a, b, init)
            assert_bits_equal(convert(kind, src, fb, a, b, init), want, "%s n=%d fb=%r a=%r b=%r" % (kind, src.size, fb, a, b))
    vals = E.CONV_SOURCES[kind]
    assert tails == set(vals.view(np.uint8 if vals.dtype == np.uint8 else "u%d" % vals.itemsize).tolist()), "a value never reaches the tail"


def test_converter_quotients_reach_the_edges():
    """the parameter sets put the quotients where the body and tail rules differ: on +-0.5 ties, around 255 / 256 /
    32767 / 65535 and around +-2^31"""
    s = E.CONV_SOURCES["depth32f2disp8u"]
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        qs = {float(F(F(a) * F(fb)) / x + F(b)) for fb, a, b in E.CONV_PARAMS for x in s}
    for want in (0.5, -0.5, 1.5, -1.5, 2.5, 255.5, 256.5, -255.5, 32767.5, 65535.5, 255.0, 256.0, 65535.0,
                 2.0 ** 31, -2.0 ** 31, 2147483520.0, float("inf"), float("-inf")):
        assert want in qs, want


def test_assert_bits_equal_reports_signed_zero_mismatches():
    a = np.zeros(5, F)
    b = a.copy()
    b[3] = -0.0
    with pytest.raises(AssertionError, match=r"1 of 5 elements differ; first at \(3,\)"):
        assert_bits_equal(a, b, "zeros")
    n = np.array([np.nan, 1.0], F)
    assert_bits_equal(n, np.array([-np.nan, 1.0], F))          # any NaN matches any NaN
