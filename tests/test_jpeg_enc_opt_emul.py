"""CPU checks of the GPU JPEG encoder's optimised-table mode (csrc/dmc_jpeg_enc.cu with DMC_JPEG_OPTIMIZE_HUFFMAN) that
need no GPU.

tests/cpp/jpeg_enc_opt_emul.cpp runs the mode's kernels on the CPU from the very same primitives (csrc/dmc_jpeg_enc_core.h):
the AC symbol counts, the DC category counts, the warp-parallel table builder with its 32 lanes emulated, the frame's
header and the entropy stage with the frame's tables.  Its streams must equal cv2.imencode(img, [IMWRITE_JPEG_QUALITY, q,
IMWRITE_JPEG_OPTIMIZE, 1]) byte for byte.  The table builder alone must equal a serial restatement of libjpeg's
jpeg_gen_optimal_table on histograms no image needs to produce, the optimised bound must hold, and the parser's hashed
table de-duplication must give the pools and indices of a linear scan.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "cpp", "jpeg_enc_opt_emul.cpp")

SIZES = [(1, 1), (7, 9), (8, 8), (131, 150), (64, 641), (480, 640), (1080, 1920), (3, 10000)]
QUALITIES = (1, 5, 25, 50, 75, 80, 95, 100)


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    lib_path = str(tmp_path_factory.mktemp("opt_emul") / "libjpeg_enc_opt_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fsanitize=undefined", "-fno-sanitize-recover=undefined", "-o", lib_path, SRC])
    lib = C.CDLL(lib_path)
    lib.jpeg_enc_opt_emul.restype = C.c_longlong
    lib.jpeg_enc_opt_emul.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_ulonglong, C.POINTER(C.c_int)]
    lib.jpeg_enc_opt_bound.restype = C.c_ulonglong
    lib.jpeg_enc_opt_bound.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.jpeg_opt_table_check.restype = C.c_int
    lib.jpeg_opt_table_check.argtypes = [C.c_void_p, C.c_int]
    lib.jpeg_dedup_check.restype = C.c_int
    lib.jpeg_dedup_check.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    return lib


def cv2_encode(img, q, optimize=True):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize)])
    assert ok
    return bytes(buf)


def emul_encode(lib, img, q, lanes, folded=None):
    img = np.ascontiguousarray(img, np.uint8)
    H, W = img.shape
    cap = lib.jpeg_enc_opt_bound(H, W, 1)
    out = np.empty(cap, np.uint8)
    f = C.c_int(0)
    n = lib.jpeg_enc_opt_emul(img.ctypes.data, H, W, q, lanes, out.ctypes.data, cap, C.byref(f))
    assert n > 0, "emulation failed with %d" % n
    if folded is not None:
        folded.append(f.value)
    return bytes(out[:n])


def images(H, W, seed=3):
    from oracle.oracle_py import synth_disp, degrade_blocks
    rs = np.random.RandomState(seed)
    out = {"noise": rs.randint(0, 256, (H, W)).astype(np.uint8), "zeros": np.zeros((H, W), np.uint8),
           "full": np.full((H, W), 255, np.uint8)}
    if H > 16 and W > 16:
        out["degraded"] = degrade_blocks(synth_disp(H, W, seed), seed)
    return out


@pytest.mark.parametrize("shape", SIZES)
def test_emulation_matches_cv2_optimize(emul, shape):
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


def test_code_length_fold_fixture(emul):
    """degrade_blocks(synth_disp(480, 640, 6), 6) at q100 is a natural image whose AC table needs codes over 16 bits."""
    from oracle.oracle_py import synth_disp, degrade_blocks
    img = degrade_blocks(synth_disp(480, 640, 6), 6)
    for lanes in (1, 7, 1024):
        folded = []
        assert emul_encode(emul, img, 100, lanes, folded) == cv2_encode(img, 100)
        assert folded[0] & 2, "the fixture no longer reaches the >16-bit adjustment"


def test_optimised_stream_decodes_like_the_standard_one(emul):
    from oracle.oracle_py import synth_disp, degrade_blocks
    img = degrade_blocks(synth_disp(131, 150, 4), 4)
    for q in (5, 50, 95):
        opt, std = emul_encode(emul, img, q, 7), cv2_encode(img, q, optimize=False)
        assert len(opt) < len(std)
        assert np.array_equal(cv2.imdecode(np.frombuffer(opt, np.uint8), 0), cv2.imdecode(np.frombuffer(std, np.uint8), 0))


def _check_hist(emul, counts, nsym=256):
    h = np.zeros(256, np.uint32)
    h[:len(counts)] = counts
    return emul.jpeg_opt_table_check(h.ctypes.data, nsym)


def test_table_builder_matches_serial_on_synthetic_histograms(emul):
    rs = np.random.RandomState(9)
    fib = [1, 1]
    while len(fib) < 26:
        fib.append(fib[-1] + fib[-2])
    cases = {
        "fibonacci 26": fib,                                              # deepest tree: lengths past 16 fold back
        "fibonacci 22 shuffled": list(rs.permutation(fib[:22])),
        "all equal": [7] * 256,
        "single symbol": [0] * 17 + [5],
        "single symbol 0": [100],
        "162 AC symbols once": [1 if (s & 15) <= 10 and ((s & 15) or s in (0, 0xF0)) else 0 for s in range(256)],
        "near 2^26": [(1 << 26) - 7, (1 << 26) - 3, 1 << 25, 3, 1],
        "near 2^22 spread": list(rs.randint((1 << 22) - 1000, 1 << 22, 14)) + [1] * 20,   # a frame's total stays below 2^26
        "powers of two": [1 << (i % 24) for i in range(60)],
        "ties everywhere": [1, 2] * 100,
    }
    assert sum(cases["162 AC symbols once"]) == 162
    for name, counts in cases.items():
        n = _check_hist(emul, np.asarray(counts, np.int64).astype(np.uint32))
        assert n == sum(1 for c in counts if c), "%s: %d" % (name, n)
    for cat in range(12):                                                # DC tables: 16 bins
        assert _check_hist(emul, [0] * cat + [9], nsym=16) == 1
    assert _check_hist(emul, [3, 1, 4, 1, 5, 9, 2, 6, 5, 3, 5, 8], nsym=16) == 12
    for trial in range(200):
        k = rs.randint(1, 257)
        counts = np.zeros(256, np.int64)
        counts[rs.choice(256, k if k < 256 else 256, replace=False)] = rs.geometric(rs.uniform(0.01, 0.9), min(k, 256))
        n = _check_hist(emul, counts.astype(np.uint32))
        assert n == int((counts > 0).sum()), "random histogram %d" % trial


def test_optimised_bound(emul):
    # 328 header bytes + EOI + ((12 + 11) + 63 * (16 + 10) bits per block) * 2 for stuffing; the standard bound is unchanged
    assert emul.jpeg_enc_opt_bound(8, 8, 1) == 330 + 2 * ((1661 + 7) // 8)
    assert emul.jpeg_enc_opt_bound(1080, 1920, 1) == 330 + 2 * ((32400 * 1661 + 7) // 8)
    assert emul.jpeg_enc_opt_bound(1080, 1920, 0) == 330 + 2 * ((32400 * 1658 + 7) // 8)
    rs = np.random.RandomState(1)
    for H, W in ((8, 8), (64, 64), (480, 640), (1080, 1920)):
        yy, xx = np.mgrid[:H, :W]
        cases = {"noise": rs.randint(0, 256, (H, W)).astype(np.uint8),
                 "checker1": np.where((yy + xx) % 2 == 0, 0, 255).astype(np.uint8),
                 "checker2": np.where(((yy // 2) + (xx // 2)) % 2 == 0, 255, 0).astype(np.uint8)}
        bound = emul.jpeg_enc_opt_bound(H, W, 1)
        for kind, img in cases.items():
            for q in (95, 100):
                n = len(cv2_encode(img, q))
                assert n <= bound, "%dx%d %s q%d: %d > bound %d" % (H, W, kind, q, n, bound)


def test_table_dedup_matches_linear_scan(emul):
    """The hashed de-duplication of the decoder's parser gives the pools and indices of the linear first-occurrence scan,
    on streams whose tables repeat (same image and quality, standard tables across qualities) and differ (optimised)."""
    from depthmapcompression_b200.filters import pack_streams
    rs = np.random.RandomState(4)
    imgs = [rs.randint(0, 256, (24, 40)).astype(np.uint8), np.zeros((24, 40), np.uint8),
            np.clip(rs.normal(100, 30, (24, 40)), 0, 255).astype(np.uint8)]
    streams = []
    for rep in range(3):
        for i, img in enumerate(imgs):
            for q in (10, 50, 50, 90):
                streams.append(cv2_encode(img, q, optimize=(rep + i) % 2 == 0))
    order = rs.permutation(len(streams))
    streams = [streams[i] for i in order]
    blob, offsets = pack_streams(streams)
    nq = C.c_int(0)
    nh = emul.jpeg_dedup_check(blob.ctypes.data, offsets.ctypes.data, len(streams), C.byref(nq))
    assert nh > 2 and nq.value == 3, (nh, nq.value)
