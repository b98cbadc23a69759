"""The optimised-table JPEG extensions of include/filter_ext.h (jpegEncodeGray(..., true), degradeJPEGGray(..., true))
through cv::Mat: the streams must equal cv2.imencode with IMWRITE_JPEG_OPTIMIZE byte for byte, the default call must stay
the standard stream, and the round trip must equal cv2.imdecode of the stream, for whole images and ROIs."""
import os
import subprocess

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_jpeg_ext_opt.cpp")


def _build(tmp_path):
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "test_jpeg_ext_opt")
    lib = os.path.join(ROOT, "depthmapcompression_b200")
    subprocess.check_call(["g++", "-O1", "-std=gnu++14", "-msse4.1", "-w", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "refshim"),
                           "-o", exe, SRC, "-L" + lib, "-ldmc_b200", "-ldl", "-Wl,-rpath," + lib])
    return exe


def test_jpeg_ext_opt_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


def _enc(img, q, optimize=True):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize)])
    assert ok
    return bytes(buf)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,q", [((480, 640), 50), ((480, 640), 100), ((131, 150), 80), ((1, 1), 95), ((37, 3), 0)])
def test_jpeg_ext_opt_matches_cv2(tmp_path, shape, q):
    from oracle.oracle_py import synth_disp, degrade_blocks
    exe = _build(tmp_path)
    H, W = shape
    img = degrade_blocks(synth_disp(H, W, 6), 6) if H > 16 else np.random.RandomState(2).randint(0, 256, shape).astype(np.uint8)
    raw = tmp_path / "in.raw"
    img.tofile(str(raw))
    res = subprocess.run([exe, str(raw), str(H), str(W), str(q), str(tmp_path)], capture_output=True, text=True, timeout=300)
    print(res.stdout, res.stderr)
    assert res.returncode == 0 and "ALL OK" in res.stdout
    want = _enc(img, q)
    assert (tmp_path / "stream.jpg").read_bytes() == want
    assert (tmp_path / "standard.jpg").read_bytes() == _enc(img, q, optimize=False)
    dec = np.fromfile(str(tmp_path / "degraded.raw"), np.uint8).reshape(H, W)
    assert np.array_equal(dec, cv2.imdecode(np.frombuffer(want, np.uint8), 0))
    assert "bytes %d %d" % (len(want), len(want)) in res.stdout
    if H > 2 and W > 2:
        roi = np.ascontiguousarray(img[1:-1, 1:-1])
        rwant = _enc(roi, q)
        assert (tmp_path / "roi.jpg").read_bytes() == rwant
        rdec = np.fromfile(str(tmp_path / "roi_degraded.raw"), np.uint8).reshape(H - 2, W - 2)
        assert np.array_equal(rdec, cv2.imdecode(np.frombuffer(rwant, np.uint8), 0))
        assert "roi %d %d" % (len(rwant), len(rwant)) in res.stdout
