"""CPU checks of the colour JPEG encoder (csrc/dmc_jpeg_color_enc.cu) that need no GPU.

tests/cpp/jpeg_color_enc_emul.cpp runs the encoder's kernels lane by lane on the CPU from the very same primitives
(csrc/dmc_jpeg_color_enc_core.h over csrc/dmc_jpeg_enc_core.h): colour conversion, chroma downsampling with libjpeg's
edge rules, dummy blocks, interleaved MCUs with two table sets, the lanes' MCU runs, word packing and byte stuffing.  Its
streams must equal cv2.imencode(img, [IMWRITE_JPEG_QUALITY, q, IMWRITE_JPEG_SAMPLING_FACTOR, s]) byte for byte for every
sampling cv2 writes and any number of lanes.  The header and the worst-case size bound are checked too.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
import _jpeg_color_cases as cases  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "cpp", "jpeg_color_enc_emul.cpp")
LIB = os.path.join(HERE, "cpp", "libjpeg_color_enc_emul.so")
CSRC = os.path.join(os.path.dirname(HERE), "depthmapcompression_b200", "csrc")

SIZES = cases.SIZES + [(1080, 1920), (1081, 1919), (3, 10000)]
KINDS = cases.KINDS + ("textured",)
QUALITIES = (0, 1, 5, 25, 50, 75, 90, 100)
HEADER_BYTES = 623


@pytest.fixture(scope="module")
def emul():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("dmc_jpeg_core.h", "dmc_jpeg_enc_core.h", "dmc_jpeg_color_enc_core.h")]
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        tmp = LIB + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fsanitize=undefined", "-fno-sanitize-recover=undefined", "-o", tmp, SRC])
        os.replace(tmp, LIB)
    lib = C.CDLL(LIB)
    lib.jpeg_color_enc_emul.restype = C.c_longlong
    lib.jpeg_color_enc_emul.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_ulonglong]
    lib.jpeg_color_enc_bound.restype = C.c_ulonglong
    lib.jpeg_color_enc_bound.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.jpeg_color_enc_header.restype = C.c_int
    lib.jpeg_color_enc_header.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    return lib


def image(kind, H, W):
    return cases.textured(H, W, seed=H + W) if kind == "textured" else cases.image(kind, H, W)


def cv2_encode(img, q, sampling):
    return bytes(cases.encode(img, q, sampling))


def emul_encode(lib, img, q, sampling, lanes):
    img = np.ascontiguousarray(img, np.uint8)
    H, W, _ = img.shape
    cap = lib.jpeg_color_enc_bound(H, W, cases.SAMPLINGS[sampling])
    out = np.empty(cap, np.uint8)
    n = lib.jpeg_color_enc_emul(img.ctypes.data, H, W, q, cases.SAMPLINGS[sampling], lanes, out.ctypes.data, cap)
    assert n > 0, "emulation failed with %d" % n
    return bytes(out[:n])


@pytest.mark.parametrize("shape", SIZES)
@pytest.mark.parametrize("sampling", list(cases.SAMPLINGS))
def test_emulation_matches_cv2_imencode(emul, shape, sampling):
    """Every size x content x quality, lane counts 1, 7 and 1024 (the large frames: the kernel's 1024 lanes and 7)."""
    H, W = shape
    large = H * W >= 1 << 20
    for kind in KINDS:
        if large and kind != "textured" and kind != "noise":
            qualities = (50,)
        else:
            qualities = QUALITIES if not large else (0, 50, 90, 100)
        img = image(kind, H, W)
        for q in qualities:
            want = cv2_encode(img, q, sampling)
            for lanes in ((7, 1024) if large else (1, 7, 1024)):
                got = emul_encode(emul, img, q, sampling, lanes)
                assert got == want, "%dx%d %s %s q%d lanes %d: %d vs %d bytes" % (H, W, kind, sampling, q, lanes, len(got), len(want))


def test_emulation_every_quality(emul):
    img = cases.textured(37, 53, seed=12)
    for sampling in cases.SAMPLINGS:
        for q in range(0, 101):
            assert emul_encode(emul, img, q, sampling, 5) == cv2_encode(img, q, sampling), "%s q%d" % (sampling, q)


def test_chroma_below_an_even_last_row_pair(emul):
    """Rule 3 of dmc_jpeg_color_enc_core.h: below the image, libjpeg copies the last DOWNSAMPLED chroma row rather than
    downsampling replicated input rows.  A frame whose two last rows differ tells the two apart at 4:2:0 and 4:4:0."""
    img = np.zeros((6, 16, 3), np.uint8)
    img[4] = (0, 0, 255)
    img[5] = (255, 0, 0)
    for sampling in ("420", "440"):
        for q in (50, 100):
            assert emul_encode(emul, img, q, sampling, 3) == cv2_encode(img, q, sampling), "%s q%d" % (sampling, q)


def test_header_matches_cv2(emul):
    """The 623-byte header depends only on size, quality and sampling, and equals cv2's for every sampling x quality."""
    img = cases.image("gradient", 17, 23)
    out = np.empty(HEADER_BYTES, np.uint8)
    for sampling, s in cases.SAMPLINGS.items():
        for q in range(0, 101):
            assert emul.jpeg_color_enc_header(q, 17, 23, s, out.ctypes.data) == HEADER_BYTES
            assert bytes(out) == cv2_encode(img, q, sampling)[:HEADER_BYTES], "%s q%d" % (sampling, q)
    assert emul.jpeg_color_enc_header(50, 17, 23, 0x222222, out.ctypes.data) < 0
    assert emul.jpeg_color_enc_bound(17, 23, 0x222222) == 0


def test_worst_case_bound(emul):
    """Real stream sizes never exceed the bound: noise at q100 for every sampling, and the numbers behind it."""
    rs = np.random.RandomState(1)
    for H, W in ((1, 1), (15, 17), (1080, 1920)):
        img = rs.randint(0, 256, (H, W, 3)).astype(np.uint8)
        for sampling, s in cases.SAMPLINGS.items():
            n = len(cv2_encode(img, 100, sampling))
            bound = emul.jpeg_color_enc_bound(H, W, s)
            assert n <= bound, "%dx%d %s: %d > bound %d" % (H, W, sampling, n, bound)
    # 623 header bytes + EOI + (22 + 63 * 26 bits per block) * 2 for stuffing; 1080p 4:2:0 has 68 x 120 MCUs of 6 blocks
    assert emul.jpeg_color_enc_bound(8, 8, cases.SAMPLINGS["444"]) == 625 + 2 * ((3 * 1660 + 7) // 8)
    assert emul.jpeg_color_enc_bound(1080, 1920, cases.SAMPLINGS["420"]) == 625 + 2 * ((68 * 120 * 6 * 1660 + 7) // 8)
