"""Shared helpers for the parity tests (bit-exact, NaN-aware comparison; golden fixture loading)."""
import json
import os
import zlib

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def crc(a):
    return "%08x" % (zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF)


def bits_equal(a, b):
    """Bit-exact equality; for floats 'both NaN' counts as equal (x86 emits 0xFFC00000, CUDA 0x7FFFFFFF)."""
    a = np.asarray(a); b = np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if a.dtype.kind == "f":
        na, nb = np.isnan(a), np.isnan(b)
        if not np.array_equal(na, nb):
            return False
        iv = np.uint32 if a.dtype == np.float32 else np.uint64
        return np.array_equal(a[~na].view(iv), b[~nb].view(iv))
    return np.array_equal(a, b)


def assert_bits_equal(a, b, msg=""):
    if not bits_equal(a, b):
        a = np.asarray(a); b = np.asarray(b)
        if a.shape == b.shape and a.dtype == b.dtype:
            if a.dtype.kind == "f":     # the rule of bits_equal: bits differ (-0.0 vs +0.0 too), unless both are NaN
                na, nb = np.isnan(a), np.isnan(b)
                iv = np.dtype("u%d" % a.dtype.itemsize)
                bad = (na != nb) | (~na & ~nb & (a.view(iv) != b.view(iv)))
            else:
                bad = a != b
            idx = np.argwhere(bad)
            first = tuple(int(i) for i in idx[0]) if len(idx) else None
            raise AssertionError("%s: %d of %d elements differ; first at %s: got %r expected %r"
                                 % (msg, int(bad.sum()), a.size, first, a[first] if first is not None else None,
                                    b[first] if first is not None else None))
        raise AssertionError("%s: shape/dtype mismatch %s %s vs %s %s" % (msg, a.shape, a.dtype, b.shape, b.dtype))


def ntaps(r):
    """taps of the range filter's circular window of radius r (circle_halfwidth per row)"""
    n = 0
    for dy in range(-r, r + 1):
        lim, j = r * r - dy * dy, 0
        while (j + 1) * (j + 1) <= lim:
            j += 1
        n += 2 * j + 1
    return n


def mask_undefined(got, want, kw, kh, W, method, dtype, m):
    """Copies into `got` the range-filter outputs the reference leaves undefined: it reads past its padded buffer there
    (see oracle/dmc_oracle.c, bwrf_32f).  `m` is the package, for its method constants."""
    if dtype != np.uint8 and (kw >> 1) % 8 == 5 and W % 4 == 0:
        if method == m.SEPARABLE_KERNEL:
            got[-(kh >> 1) - 1:, -1] = want[-(kh >> 1) - 1:, -1]
        elif (kh >> 1) == 0:
            got[-1, -1] = want[-1, -1]


def canon_crc(a):
    """CRC with NaNs canonicalised to the x86 default NaN (0xFFC00000) so GPU outputs hash like the reference's."""
    a = np.ascontiguousarray(a)
    if a.dtype == np.float32:
        a = a.copy(); v = a.view(np.uint32); v[np.isnan(a)] = 0xFFC00000
    return crc(a)


def load_golden():
    with open(os.path.join(GOLDEN_DIR, "golden.json")) as f:
        return json.load(f)


def load_png(name):
    import cv2
    img = cv2.imread(os.path.join(GOLDEN_DIR, name), cv2.IMREAD_UNCHANGED)
    assert img is not None, name
    return img


def make_image(rs, H, W, dtype=np.uint8, cn=1, kind="pw"):
    """Piecewise-constant + noise (exercises both weight outcomes) or pure noise."""
    shape = (H, W) if cn == 1 else (H, W, cn)
    if kind == "noise":
        a = rs.randint(0, 256, size=shape)
    elif kind == "const":
        a = np.full(shape, 77)
    else:
        blk = rs.randint(0, 256, size=((H + 7) // 8, (W + 7) // 8) + (() if cn == 1 else (cn,)))
        a = np.kron(blk, np.ones((8, 8) + (() if cn == 1 else (1,))))[:H, :W] + rs.randint(-6, 7, size=shape)
        a = np.clip(a, 0, 255)
    if dtype == np.uint16:
        a = a * 200 + rs.randint(0, 50, size=shape)
    elif dtype == np.int16:
        a = a * 200 - 20000
    elif dtype in (np.float32, np.float64):
        a = a * 3.7 + 0.25 * rs.randint(0, 4, size=shape)
    return np.ascontiguousarray(a.astype(dtype))


def special_floats(dtype, nan=True, negzero=True):
    """IEEE values a float min / max can get wrong: infinities, the largest finite values, the smallest normal value
    and its neighbours (FLT_MIN seeds maxFilter), subnormals, zeros and NaN."""
    f = np.finfo(dtype); t = dtype(f.tiny); z = dtype(0)
    v = [z, np.inf, -np.inf, f.max, -f.max, t, -t, np.nextafter(t, z), np.nextafter(t, dtype(1)), -np.nextafter(t, z),
         t / dtype(4), -t / dtype(4), f.smallest_subnormal, -f.smallest_subnormal]
    if negzero:
        v.append(-z)
    if nan:
        v.append(np.nan)
    return np.array(v, dtype)


def special_image(rs, H, W, dtype, cn=1, nan=True, negzero=True, p=0.2):
    """Half-integers in -1.5..1.5 (many ties and zeros) with a fraction `p` of the pixels, and every corner, replaced by
    special_floats.  With `negzero` the zeros take random signs."""
    shape = (H, W) if cn == 1 else (H, W, cn)
    a = (rs.randint(-3, 4, size=shape) * 0.5).astype(dtype)
    if negzero:
        a[(a == 0) & (rs.rand(*shape) < 0.5)] = -0.0
    sp = special_floats(dtype, nan, negzero)
    pick = rs.rand(*shape) < p
    a[pick] = sp[rs.randint(0, len(sp), size=int(pick.sum()))]
    for y, x in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)):
        a[y, x] = sp[rs.randint(0, len(sp), size=a[y, x].shape)]
    return np.ascontiguousarray(a)
