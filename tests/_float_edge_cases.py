"""Inputs on which the 32-bit range filter and the disparity <-> depth converters can go wrong bit by bit, shared by
tests/test_float_range_filter_reference.py (CPU), tests/test_gpu_float_range_filter.py and tools/fuzz_parity.py.

The range filter's rules (oracle/dmc_oracle.c, bwrf_32f): taps in raster order, w = |fl(c - v)| <= th (C3: the
distance is (|d2| + |d1|) + |d0|), t = t + w*v with 0*inf = NaN, W = W + w, out = t / W, no flush to zero.  Each case
below is a frame family built so that one of those rules decides some output pixel, with the thresholds that make it
decide: distances that land exactly on th, sums whose value depends on the tap order, signed zeros, subnormals,
infinities, NaN and sums that overflow.  The special pixels are stamped where the kernels change schedule
(`stamp_points`)."""
from typing import Callable, List, NamedTuple

import numpy as np

F = np.float32
INF = F(np.inf)
NAN = F(np.nan)
FMAX = F(np.finfo(F).max)
TINY = F(np.finfo(F).tiny)                      # smallest normal
SUB = F(np.finfo(F).smallest_subnormal)

# thresholds every case also runs with: NaN, +-inf, +-0, the smallest subnormal, FLT_MAX and a negative value
SPECIAL_TH = [NAN, INF, -INF, F(0.0), F(-0.0), SUB, FMAX, F(-1.0)]


def around(th):
    """th and its two float32 neighbours"""
    th = F(th)
    return [np.nextafter(th, -INF), th, np.nextafter(th, INF)]


def stamp_points(H, W):
    """Pixels where a kernel changes schedule: the corners, the 128-pixel tile columns (x = 127 / 128, 255 / 256), the
    rows where tiles of 2R rows meet (R = 1, 2, 4, 8), the last row and column (partial tiles; the padding quirk reads
    column 0 of the next row for the last column), and one interior pixel with no other stamp within 10 pixels, so
    that centres at every offset of the disc's rim see it alone."""
    xs = {0, 1, W - 2, W - 1} | {x for k in range(128, W, 128) for x in (k - 1, k)}
    ys = {0, 3, 4, 7, 8, 15, 16, 31, 32, H - 2, H - 1}
    pts = {(y, x) for y in ys for x in xs if 0 <= y < H and 0 <= x < W}
    if H >= 3 and W >= 3:
        pts.add((H // 2, W // 3))
    return sorted(pts)


class Case(NamedTuple):
    name: str
    cn: int
    image: Callable            # (H, W) -> float32 image, (H, W) or (H, W, 3)
    thresholds: List           # the thresholds that decide its special pixels (SPECIAL_TH come on top)


def _stamped(H, W, cn, background, motif):
    """background: (H, W, cn) float32; motif: list of (dx, value-per-channel) written right of every stamp point"""
    a = np.array(background, F).reshape(H, W, cn)
    for y, x in stamp_points(H, W):
        for dx, val in motif:
            if x + dx < W:
                a[y, x + dx] = val
    return np.ascontiguousarray(a[:, :, 0] if cn == 1 else a)


def _fill(H, W, cn, v):
    return np.full((H, W, cn), v, F)


# (c, v) pairs whose float difference rounds: down in magnitude (the exact distance is above th = |fl(c - v)|, so a
# distance in double precision or the test c - th <= v <= c + th rejects a tap the filter takes), up, and to even
ROUND_PAIRS = [(1e8, -0.3), (1.0, 3e-8), (16777216.0, -1.0), (1e8, 0.3), (0.1, -0.2), (-3e7, 1.1)]


def _round_case(c, v, cn):
    c, v = F(c), F(v)
    th = abs(F(c - v))
    if cn == 1:
        img = lambda H, W: _stamped(H, W, 1, _fill(H, W, 1, c), [(0, v)])
    else:   # the pair in channel 0, equal channels 1 and 2: the C3 distance is (0 + 0) + |fl(c - v)|
        img = lambda H, W: _stamped(H, W, 3, _fill(H, W, 3, (c, 5.0, 7.0)), [(0, (v, 5.0, 7.0))])
    return Case("round_%g_%g_c%d" % (c, v, cn), cn, img, around(th))


def _sum_order_case(cn):
    """1e8, -1e8, 1 in a row on zeros, all within th: raster order sums them to 1, reversed order to 0"""
    motif = [(0, F(1e8)), (1, F(-1e8)), (2, F(1.0))]
    return Case("sum_order_c%d" % cn, cn, lambda H, W: _stamped(H, W, cn, _fill(H, W, cn, 0.0), motif), [F(1e9), FMAX, INF])


def _c3_order_case():
    """|d| = (1, e, e) with e = 2^-24 in the three channel orders on zeros: (|d2| + |d1|) + |d0| is 1 + 2^-23 when the 1
    is in channel 0 and 1 (ties to even) otherwise; any other order of additions swaps those results.  th = 1."""
    e = F(2.0 ** -24)
    motif = [(0, (1.0, e, e)), (1, (e, 1.0, e)), (3, (e, e, 1.0))]
    return Case("c3_order", 3, lambda H, W: _stamped(H, W, 3, _fill(H, W, 3, 0.0), motif), around(1.0))


def _zeros_case(cn):
    """a plateau of -0.0 with +0.0 stamps: the sums start at +0.0, so every output is +0.0"""
    return Case("signed_zeros_c%d" % cn, cn, lambda H, W: _stamped(H, W, cn, _fill(H, W, cn, -0.0), [(0, F(0.0))]),
                [F(1.0)])


def _subnormal_case(cn):
    """subnormal values, distances and thresholds; the smallest normal value and its neighbours stamped"""
    def img(H, W):
        rs = np.random.RandomState(H * 7 + W + cn)
        bg = (rs.randint(-8, 9, size=(H, W, cn)) * SUB).astype(F)
        return _stamped(H, W, cn, bg, [(0, TINY), (1, np.nextafter(TINY, F(0))), (2, -TINY)])
    return Case("subnormal_c%d" % cn, cn, img, [F(2 * SUB), F(4 * SUB), F(TINY / 2), TINY])


def _specials_case(cn):
    """NaN and the infinities as centre and tap among half-integers; th = +inf takes every finite distance and rejects
    inf - inf = NaN"""
    def img(H, W):
        rs = np.random.RandomState(H * 5 + W + cn)
        bg = (rs.randint(-3, 4, size=(H, W, cn)) * 0.5).astype(F)
        a = bg.copy()
        for k, (y, x) in enumerate(stamp_points(H, W)):
            a[y, x, k % cn] = (NAN, INF, -INF)[k % 3]
        return np.ascontiguousarray(a[:, :, 0] if cn == 1 else a)
    return Case("nan_inf_c%d" % cn, cn, img, [F(1.0), F(30.0)])


def _overflow_case(cn):
    """values near +-FLT_MAX: sums overflow to inf, distances between opposite signs to inf"""
    motif = [(0, FMAX), (1, -FMAX), (2, F(0.75) * FMAX)]
    return Case("overflow_c%d" % cn, cn, lambda H, W: _stamped(H, W, cn, _fill(H, W, cn, F(0.75) * FMAX), motif),
                [F(0.5) * FMAX, FMAX])


def cases(cn):
    out = [_round_case(c, v, cn) for c, v in ROUND_PAIRS]
    out += [_sum_order_case(cn), _zeros_case(cn), _subnormal_case(cn), _specials_case(cn), _overflow_case(cn)]
    if cn == 3:
        out.append(_c3_order_case())
    return out


CASES_C1 = cases(1)
CASES_C3 = cases(3)


def all_thresholds(case):
    return list(case.thresholds) + SPECIAL_TH


# ---------------------------------------------------------------------------------------------------------- converters
# Source values, and (focal_baseline, a, b) such that v = a*fb / s + b lands on +-0.5 ties (5/2, 511/2, 513/2, 1/1 - 0.5),
# around 255 / 256 / 32767 / 65535 (255, 511, 512, 513, 65535, 131071 over 1 and 2) and around +-2^31 (2^32 and 2^32 - 256 over
# +-2), besides the quotients by 0, negative and subnormal sources.
CONV_SOURCES = {
    "disp8u2depth32f": np.array([0, 1, 2, 3, 4, 7, 128, 255], np.uint8),
    "depth32f2disp8u": np.array([NAN, INF, -INF, 0.0, -0.0, 1.0, 2.0, -1.0, -2.0, 3.0, 0.5, 4.0, SUB, -SUB, TINY / 4,
                                 1e-30, 1e30, FMAX, -FMAX, 1e-3, 65535.0], F),
    "depth16u2disp8u": np.array([0, 1, 2, 3, 4, 255, 256, 32767, 32768, 40000, 65534, 65535], np.uint16),
    "disp16s2depth16u": np.array([0, 1, -1, 2, -2, 3, -3, 4, 255, -256, 32767, -32768], np.int16),
}
CONV_PARAMS = [(1.0, 1.0, 0.0), (5.0, 1.0, 0.0), (511.0, 1.0, 0.0), (513.0, 1.0, 0.0), (65535.0, 1.0, 0.0),
               (131071.0, 1.0, 0.0), (2.0 ** 32, 1.0, 0.0), (4294967040.0, 1.0, 0.0), (-511.0, 1.0, 0.0),
               (1.0, 1.0, 0.5), (1.0, 1.0, -0.5), (255.0, 1.0, 0.0), (512.0, 1.0, 0.0), (43125.0, 2.6, 0.0),
               (1.0, -0.0, 0.0), (1.0, 1.0, -0.0)]


def converter_arrays(kind):
    """Arrays of n = 16 m + t elements, t in {0, 1, 15}: the first 16 m (the reference's SIMD body) hold every source
    value, the last t (its scalar tail) a rotation of them, so every value goes through both parts."""
    vals = CONV_SOURCES[kind]
    m = -(-len(vals) // 16)
    body = np.resize(vals, 16 * m)
    out = [body.reshape(1, -1)]
    for t in (1, 15):
        for o in range(0, len(vals), t):
            tail = np.resize(np.roll(vals, -o), t)
            out.append(np.concatenate([body, tail]).reshape(1, -1))
    out.append(np.concatenate([np.resize(vals, 48), np.resize(np.roll(vals, 3), 15)]).reshape(3, 21))   # 2-D, n % 16 = 15
    return out
