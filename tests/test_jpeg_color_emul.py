"""CPU checks of the colour JPEG decoder (csrc/dmc_jpeg_color.cu) that need no GPU:

  * the lane-parallel decode of interleaved MCUs, the one-lane restart-interval decode and the upsampling / colour
    conversion, emulated from the kernels' own primitives (tests/cpp/jpeg_color_emul.cpp over csrc/dmc_jpeg_color_core.h),
    must reproduce cv2.imdecode(buf, IMREAD_COLOR) bit for bit over sizes, contents, the five samplings cv2 writes,
    qualities, table kinds, restart intervals and lane counts;
  * a Python restatement of libjpeg-turbo's upsampling and colour conversion, applied to decoded component planes, must
    equal both cv2 and the host restatement of the kernels;
  * the colour parser must refuse every stream kind it does not decode with its reason, and never crash.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from _util import assert_bits_equal

cv2 = pytest.importorskip("cv2")
import _jpeg_color_cases as cases  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "cpp", "jpeg_color_emul.cpp")
LIB = os.path.join(HERE, "cpp", "libjpeg_color_emul.so")
CSRC = os.path.join(os.path.dirname(HERE), "depthmapcompression_b200", "csrc")
LANES = 768                   # kJCT of dmc_jpeg_color.cu


@pytest.fixture(scope="module")
def emul():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("dmc_jpeg_core.h", "dmc_jpeg_color_core.h", "dmc_jpeg_parse.h")]
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        tmp = LIB + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fwrapv", "-fsanitize=undefined", "-fno-sanitize-recover=undefined", "-o", tmp, SRC])
        os.replace(tmp, LIB)
    lib = C.CDLL(LIB)
    lib.jpeg_color_emul_decode.restype = C.c_int
    lib.jpeg_color_emul_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_char_p, C.c_size_t]
    lib.jpeg_color_emul_planes.restype = C.c_long
    lib.jpeg_color_emul_planes.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.c_char_p, C.c_size_t]
    lib.jpeg_color_emul_convert.restype = None
    lib.jpeg_color_emul_convert.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_void_p]
    lib.jpeg_color_emul_probe.restype = C.c_int
    lib.jpeg_color_emul_probe.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_size_t]
    lib.jpeg_color_emul_ycc_tables.restype = None
    lib.jpeg_color_emul_ycc_tables.argtypes = [C.c_void_p]
    return lib


def _buf(stream):
    a = np.frombuffer(bytes(stream), np.uint8).copy() if len(stream) else np.zeros(1, np.uint8)
    return a, len(stream)


def decode(lib, stream, H, W, lanes):
    a, n = _buf(stream)
    out = np.full((H, W, 3), 0xAB, np.uint8); rounds = C.c_int(); err = C.create_string_buffer(256)
    rc = lib.jpeg_color_emul_decode(a.ctypes.data, n, H, W, out.ctypes.data, lanes, C.byref(rounds), err, 256)
    assert rc == 0, err.value
    return out, rounds.value


def probe(lib, stream):
    a, n = _buf(stream)
    err = C.create_string_buffer(256); r, c, k = C.c_int(), C.c_int(), C.c_int()
    rc = lib.jpeg_color_emul_probe(a.ctypes.data if n else None, n, C.byref(r), C.byref(c), C.byref(k), err, 256)
    return rc, err.value.decode(), (r.value, c.value, k.value)


def check(lib, stream, H, W, lanes, what):
    got, rounds = decode(lib, stream, H, W, lanes)
    assert_bits_equal(got, cases.reference(stream), what)
    return rounds


@pytest.mark.parametrize("sampling", list(cases.SAMPLINGS))
def test_small_frames_match_cv2(emul, sampling):
    """Every small size x content x quality x table kind (standard, optimised, restart intervals) x lane count."""
    worst = 0
    for H, W in cases.SIZES:
        for kind in cases.KINDS:
            img = cases.image(kind, H, W)
            for q in cases.QUALITIES:
                for tables in cases.TABLES:
                    s = cases.encode(img, q, sampling, tables)
                    for lanes in (1, 7, LANES):
                        worst = max(worst, check(emul, s, H, W, lanes, "%dx%d %s %s q%d %s lanes %d" % (H, W, kind, sampling, q, tables, lanes)))
    assert worst >= 1            # the synchronisation rounds were exercised
    print("%s: at most %d synchronisation rounds" % (sampling, worst))


@pytest.mark.parametrize("sampling", list(cases.SAMPLINGS))
def test_vga_frames_match_cv2(emul, sampling):
    H, W = 480, 640
    rounds = {}
    for kind in cases.KINDS + ("textured",):
        img = cases.textured(H, W) if kind == "textured" else cases.image(kind, H, W)
        for q in cases.QUALITIES:
            for tables in cases.TABLES:
                if tables == "restart" and q not in (50, 90):
                    continue
                s = cases.encode(img, q, sampling, tables, rst=7)
                rounds[(kind, q, tables)] = check(emul, s, H, W, LANES, "480x640 %s %s q%d %s" % (kind, sampling, q, tables))
    s = cases.encode(cases.textured(H, W, 1), 80, sampling)
    check(emul, s, H, W, 7, "480x640 textured %s q80 lanes 7" % sampling)
    print(sampling, "rounds on textured content:", {k[1:]: v for k, v in rounds.items() if k[0] == "textured"})


def test_1080p_frames_match_cv2_and_report_rounds(emul):
    H, W = 1080, 1920
    report = []
    for sampling in cases.SAMPLINGS:
        img = cases.textured(H, W, 3)
        for q in (50, 80):
            s = cases.encode(img, q, sampling)
            r = check(emul, s, H, W, LANES, "1080p textured %s q%d" % (sampling, q))
            report.append((sampling, q, len(s), r))
            # content with entropy synchronises within a few rounds; flat content may take up to one round per lane
            # (the result is exact either way), so only textured content is bounded here
            assert r <= 16, "synchronisation took %d rounds" % r
    check(emul, cases.encode(cases.textured(H, W, 4), 80, "420", "restart", rst=16), H, W, LANES, "1080p restart")
    print("1080p (sampling, quality, bytes, rounds):", report)


def test_every_quality_matches_cv2(emul):
    img = cases.image("noise", 17, 23, 5)
    for q in range(0, 101):
        for tables in ("standard", "optimised"):
            s = cases.encode(img, q, "420", tables)
            check(emul, s, 17, 23, 7, "17x23 4:2:0 q%d %s" % (q, tables))


def test_one_component_streams_decode_to_gray_bgr(emul):
    for H, W in ((1, 1), (15, 17), (61, 83), (480, 640)):
        g = cases.image("noise", H, W)[:, :, 0].copy()
        for q in (5, 50, 100):
            for tables in cases.TABLES:
                s = cases.encode(g, q, tables=tables)
                assert probe(emul, s)[2] == (H, W, 1)
                got, _ = decode(emul, s, H, W, LANES)
                assert_bits_equal(got, cases.reference(s), "gray %dx%d q%d %s" % (H, W, q, tables))
                assert_bits_equal(got[:, :, 0], cv2.imdecode(s, 0), "gray plane")


def test_refusals_carry_their_reason(emul):
    img = cases.image("noise", 24, 40)
    rc, why, size = probe(emul, bytes(cases.encode(img, 75)))
    assert rc == 0 and size == (24, 40, 3), why
    for stream, words in cases.refused_streams(img):
        rc, why, _ = probe(emul, stream)
        assert rc != 0 and words in why, (words, why)
    # the same markers that libjpeg reads as YCbCr are decoded as such
    for stream in cases.accepted_variants(img):
        rc, why, _ = probe(emul, stream)
        assert rc == 0, why
        got, _ = decode(emul, stream, 24, 40, LANES)
        assert_bits_equal(got, cases.reference(stream), "accepted variant")


def test_truncated_and_malformed_streams_never_crash(emul):
    """Every truncation of a colour stream is refused or decoded without a fault (the library is built with UBSAN)."""
    img = cases.image("noise", 20, 36)
    for sampling in ("420", "411"):
        for tables in ("standard", "restart"):
            good = bytes(cases.encode(img, 60, sampling, tables))
            for n in range(0, len(good), 3):
                rc, _, size = probe(emul, good[:n])
                if rc == 0:
                    decode(emul, good[:n], 20, 36, 5)
    assert probe(emul, b"")[0] != 0 and probe(emul, b"not a jpeg")[0] != 0


def test_garbage_scans_do_not_depend_on_the_lane_count(emul):
    rs = np.random.RandomState(11)
    for sampling in cases.SAMPLINGS:
        good = bytes(cases.encode(cases.image("noise", 48, 80), 90, sampling))
        j = good.index(b"\xff\xda")
        head = good[:j + 2 + int.from_bytes(good[j + 2:j + 4], "big")]
        for trial in range(6):
            body = bytes(rs.randint(0, 256, int(rs.randint(0, 4000))).astype(np.uint8)).replace(b"\xff", b"\xfe")
            s = head + body + b"\xff\xd9"
            a, _ = decode(emul, s, 48, 80, LANES)
            b, _ = decode(emul, s, 48, 80, 5)
            c, _ = decode(emul, s, 48, 80, 1)
            assert_bits_equal(a, b, "garbage scan %s %d: 768 vs 5 lanes" % (sampling, trial))
            assert_bits_equal(a, c, "garbage scan %s %d: 768 vs 1 lane" % (sampling, trial))


# ---- upsampling and colour conversion, restated in numpy from libjpeg-turbo's jdsample.c / jdcolor.c ------------------
def _fix(x):
    return int(x * 65536 + 0.5)


def np_upsample(c, dw, dh, hy, vy, H, W):
    c = c.astype(np.int64)[:dh, :dw]
    if hy == 1 and vy == 1:
        return c[:H, :W]
    if hy == 1 and vy == 2:
        up = np.vstack([c[:1], c[:-1]]); dn = np.vstack([c[1:], c[-1:]])
        out = np.empty((2 * dh, dw), np.int64)
        out[0::2] = (3 * c + up + 1) >> 2
        out[1::2] = (3 * c + dn + 2) >> 2
        return out[:H, :W]
    if hy == 2 and vy == 1 and dw > 2:
        lf = np.hstack([c[:, :1], c[:, :-1]]); rt = np.hstack([c[:, 1:], c[:, -1:]])
        out = np.empty((dh, 2 * dw), np.int64)
        out[:, 0::2] = (3 * c + lf + 1) >> 2
        out[:, 1::2] = (3 * c + rt + 2) >> 2
        out[:, 0] = c[:, 0]; out[:, -1] = c[:, -1]
        return out[:H, :W]
    if hy == 2 and vy == 2 and dw > 2:
        up = np.vstack([c[:1], c[:-1]]); dn = np.vstack([c[1:], c[-1:]])
        out = np.empty((2 * dh, 2 * dw), np.int64)
        for v, nb in ((0, up), (1, dn)):
            s = 3 * c + nb
            lf = np.hstack([s[:, :1], s[:, :-1]]); rt = np.hstack([s[:, 1:], s[:, -1:]])
            even = (3 * s + lf + 8) >> 4; odd = (3 * s + rt + 7) >> 4
            even[:, 0] = (4 * s[:, 0] + 8) >> 4; odd[:, -1] = (4 * s[:, -1] + 7) >> 4
            out[v::2, 0::2] = even; out[v::2, 1::2] = odd
        return out[:H, :W]
    return np.repeat(np.repeat(c, vy, 0), hy, 1)[:H, :W]


def np_convert(y, cb, cr):
    x = np.arange(256) - 128
    cr_r = (_fix(1.402) * x + (1 << 15)) >> 16
    cb_b = (_fix(1.772) * x + (1 << 15)) >> 16
    cr_g = -_fix(0.71414) * x
    cb_g = -_fix(0.34414) * x + (1 << 15)
    y = y.astype(np.int64)
    bgr = np.dstack([y + cb_b[cb], y + ((cb_g[cb] + cr_g[cr]) >> 16), y + cr_r[cr]])
    return np.clip(bgr, 0, 255).astype(np.uint8)


def planes_of(lib, stream, H, W):
    geom = (C.c_int * 7)(); err = C.create_string_buffer(256)
    a, n = _buf(stream)
    size = lib.jpeg_color_emul_planes(a.ctypes.data, n, H, W, None, 0, geom, err, 256)
    assert size > 0, err.value
    p = np.zeros(size, np.uint8)
    assert lib.jpeg_color_emul_planes(a.ctypes.data, n, H, W, p.ctypes.data, p.size, geom, err, 256) == size
    nc, hy, vy, yw, yh, cw, ch = list(geom)
    Y = p[:yw * yh].reshape(yh, yw)
    cb = p[yw * yh:yw * yh + cw * ch].reshape(ch, cw)
    cr = p[yw * yh + cw * ch:].reshape(ch, cw)
    return p, geom, (hy, vy), Y, cb, cr


def ycc_image(H, W, luma, chroma, seed):
    """A BGR image whose YCbCr has the given luma (a constant or 'ramp') and chroma pattern ('noise' or 'ramp')."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    Y = np.full((H, W), float(luma)) if luma != "ramp" else 40 + 170.0 * xx / max(W - 1, 1)
    if chroma == "noise":
        cb, cr = rs.randint(0, 256, (H, W)).astype(float), rs.randint(0, 256, (H, W)).astype(float)
    else:
        cb, cr = 255.0 * xx / max(W - 1, 1), 255.0 * yy / max(H - 1, 1)
    b = Y + 1.772 * (cb - 128); g = Y - 0.34414 * (cb - 128) - 0.71414 * (cr - 128); r = Y + 1.402 * (cr - 128)
    return np.clip(np.rint(np.dstack([b, g, r])), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("sampling", list(cases.SAMPLINGS))
def test_upsampling_and_conversion_restatement(emul, sampling):
    """From the decoded planes: numpy restatement == the kernels' host restatement == cv2, on flat luma with varying
    chroma (where upsampling alone shapes the picture), chroma ramps and saturated content."""
    t = np.zeros(1024, np.int32)
    emul.jpeg_color_emul_ycc_tables(t.ctypes.data)
    x = np.arange(256) - 128
    assert np.array_equal(t[:256], (_fix(1.402) * x + (1 << 15)) >> 16)
    assert np.array_equal(t[768:], -_fix(0.34414) * x + (1 << 15))
    n = 0
    for H, W in ((1, 1), (2, 3), (3, 3), (8, 8), (15, 17), (17, 23), (61, 83), (64, 96)):
        for luma, chroma in ((128, "noise"), (128, "ramp"), (30, "noise"), ("ramp", "ramp")):
            for img in (ycc_image(H, W, luma, chroma, H * W), cases.image("saturated", H, W)):
                s = cases.encode(img, 100, sampling)
                p, geom, (hy, vy), Y, cb, cr = planes_of(emul, s, H, W)
                dw, dh = -(-W // hy), -(-H // vy)
                want = cases.reference(s)
                mine = np_convert(Y[:H, :W], np_upsample(cb, dw, dh, hy, vy, H, W), np_upsample(cr, dw, dh, hy, vy, H, W))
                assert_bits_equal(mine, want, "numpy restatement %dx%d %s %s/%s" % (H, W, sampling, luma, chroma))
                host = np.zeros((H, W, 3), np.uint8)
                emul.jpeg_color_emul_convert(p.ctypes.data, geom, H, W, host.ctypes.data)
                assert_bits_equal(host, want, "host restatement %dx%d %s" % (H, W, sampling))
                n += 1
    assert n == 64
