"""jpegRateDistortionGray of include/filter_ext.h through cv::Mat: the stream sizes must equal cv2.imencode's, the PSNR of
the decoded image cv2.PSNR against cv2.imdecode's, and the PSNR of the filtered image cv2.PSNR against the port's
PostFilterSet()(decoded, 2, 1, 3, 5, 10), in both Huffman modes."""
import os
import subprocess

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_rd_sweep_ext.cpp")
QUALITIES = (0, 10, 50, 95, 100)


def _build(tmp_path):
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "test_rd_sweep_ext")
    lib = os.path.join(ROOT, "depthmapcompression_b200")
    subprocess.check_call(["g++", "-O1", "-std=gnu++14", "-msse4.1", "-w", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "refshim"),
                           "-o", exe, SRC, "-L" + lib, "-ldmc_b200", "-ldl", "-Wl,-rpath," + lib])
    return exe


def test_rd_sweep_ext_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_rd_sweep_ext_matches_cv2_and_port(tmp_path):
    from _util import load_png
    from oracle.oracle_py import Port
    exe = _build(tmp_path)
    img = load_png("kinect_meeting_q50.png")
    H, W = img.shape
    raw = tmp_path / "in.raw"
    img.tofile(str(raw))
    res = subprocess.run([exe, str(raw), str(H), str(W)] + [str(q) for q in QUALITIES], capture_output=True, text=True, timeout=600)
    print(res.stdout, res.stderr)
    assert res.returncode == 0 and "ALL OK" in res.stdout
    got = {}
    for line in res.stdout.splitlines():
        if line.startswith("rd "):
            _, opt, q, nb, pc, pf = line.split()
            got[(int(opt), int(q))] = (int(nb), float(pc), float(pf))
    port = Port()
    for q in QUALITIES:
        for opt in (0, 1):
            ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, opt])
            assert ok
            dec = cv2.imdecode(buf, 0)
            filt = port.post_filter_set(dec, 2, 1, 3, 5, 10)
            nb, pc, pf = got[(opt, q)]
            assert nb == len(buf), (opt, q)
            assert abs(pc - cv2.PSNR(img, dec)) < 1e-9, (opt, q)
            assert abs(pf - cv2.PSNR(img, filt)) < 1e-9, (opt, q)
