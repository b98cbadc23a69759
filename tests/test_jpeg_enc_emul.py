"""CPU checks of the GPU JPEG encoder (csrc/dmc_jpeg_enc.cu) that need no GPU.

tests/cpp/jpeg_enc_emul.cpp runs the encoder's kernels lane by lane on the CPU, from the very same primitives
(csrc/dmc_jpeg_enc_core.h): transform, per-lane bit offsets, word packing with shared boundary words, byte stuffing.  Its
streams must equal cv2.imencode(img, [IMWRITE_JPEG_QUALITY, q]) byte for byte for any number of lanes.  The file also
proves the multiply-high quantiser exhaustively and checks the worst-case size bound.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "cpp", "jpeg_enc_emul.cpp")
LIB = os.path.join(HERE, "cpp", "libjpeg_enc_emul.so")
CSRC = os.path.join(os.path.dirname(HERE), "depthmapcompression_b200", "csrc")

SIZES = [(1, 1), (7, 9), (8, 8), (131, 150), (64, 641), (480, 640), (1080, 1920), (3, 10000)]
QUALITIES = (1, 5, 25, 50, 75, 80, 95, 100)


@pytest.fixture(scope="module")
def emul():
    deps = [SRC, os.path.join(CSRC, "dmc_jpeg_enc_core.h"), os.path.join(CSRC, "dmc_jpeg_core.h")]
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fsanitize=undefined", "-fno-sanitize-recover=undefined", "-o", LIB, SRC])
    lib = C.CDLL(LIB)
    lib.jpeg_enc_emul.restype = C.c_longlong
    lib.jpeg_enc_emul.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_ulonglong]
    lib.jpeg_enc_bound.restype = C.c_ulonglong
    lib.jpeg_enc_bound.argtypes = [C.c_int, C.c_int]
    lib.jpeg_enc_check_quant.restype = C.c_longlong
    return lib


def cv2_encode(img, q):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return bytes(buf)


def emul_encode(lib, img, q, lanes):
    img = np.ascontiguousarray(img, np.uint8)
    H, W = img.shape
    cap = lib.jpeg_enc_bound(H, W)
    out = np.empty(cap, np.uint8)
    n = lib.jpeg_enc_emul(img.ctypes.data, H, W, q, lanes, out.ctypes.data, cap)
    assert n > 0, "emulation failed with %d" % n
    return bytes(out[:n])


def images(H, W, seed=3):
    from oracle.oracle_py import synth_disp, degrade_blocks
    rs = np.random.RandomState(seed)
    out = {"noise": rs.randint(0, 256, (H, W)).astype(np.uint8), "zeros": np.zeros((H, W), np.uint8),
           "full": np.full((H, W), 255, np.uint8)}
    if H > 16 and W > 16:
        out["degraded"] = degrade_blocks(synth_disp(H, W, seed), seed)
    return out


def test_quantiser_multiply_high_is_exact(emul):
    assert emul.jpeg_enc_check_quant() == 0


@pytest.mark.parametrize("shape", SIZES)
def test_emulation_matches_cv2_imencode(emul, shape):
    H, W = shape
    for kind, img in images(H, W).items():
        for q in QUALITIES:
            want = cv2_encode(img, q)
            lane_counts = (1024,) if H * W >= 1 << 20 else (1, 7, 1024)
            for lanes in lane_counts:
                got = emul_encode(emul, img, q, lanes)
                assert got == want, "%dx%d %s q%d lanes %d: %d vs %d bytes" % (H, W, kind, q, lanes, len(got), len(want))


def test_emulation_every_quality(emul):
    rs = np.random.RandomState(12)
    img = np.clip(rs.normal(120, 40, (37, 53)), 0, 255).astype(np.uint8)
    for q in range(0, 101):
        assert emul_encode(emul, img, q, 5) == cv2_encode(img, q), "q%d" % q


def test_worst_case_bound(emul):
    rs = np.random.RandomState(1)
    for H, W in ((8, 8), (64, 64), (480, 640), (1080, 1920)):
        yy, xx = np.mgrid[:H, :W]
        cases = {"noise": rs.randint(0, 256, (H, W)).astype(np.uint8),
                 "checker1": np.where((yy + xx) % 2 == 0, 0, 255).astype(np.uint8),
                 "checker2": np.where(((yy // 2) + (xx // 2)) % 2 == 0, 255, 0).astype(np.uint8)}
        bound = emul.jpeg_enc_bound(H, W)
        for kind, img in cases.items():
            for q in (95, 100):
                n = len(cv2_encode(img, q))
                assert n <= bound, "%dx%d %s q%d: %d > bound %d" % (H, W, kind, q, n, bound)
    # the numbers behind the bound: 328 header bytes + EOI + (20 + 63 * 26 bits per block) * 2 for stuffing
    assert emul.jpeg_enc_bound(8, 8) == 330 + 2 * ((1658 + 7) // 8)
    assert emul.jpeg_enc_bound(1080, 1920) == 330 + 2 * ((32400 * 1658 + 7) // 8)
