"""jpegDecodeColor of include/filter_ext.h through cv::Mat: equal to cv2.imdecode(buf, IMREAD_COLOR) for colour streams of
every sampling and for a one-component stream; a progressive stream is refused with its reason."""
import os
import subprocess

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_jpeg_color_ext.cpp")


def _build(tmp_path):
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "test_jpeg_color_ext")
    lib = os.path.join(ROOT, "depthmapcompression_b200")
    subprocess.check_call(["g++", "-O1", "-std=gnu++14", "-msse4.1", "-w", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "refshim"),
                           "-o", exe, SRC, "-L" + lib, "-ldmc_b200", "-ldl", "-Wl,-rpath," + lib])
    return exe


def test_jpeg_color_ext_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_jpeg_color_ext_matches_cv2(tmp_path):
    exe = _build(tmp_path)
    rs = np.random.RandomState(4)
    img = rs.randint(0, 256, (37, 61, 3)).astype(np.uint8)
    files, want = [], {}
    for name, sf in (("444", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444), ("422", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422),
                     ("420", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420), ("440", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440),
                     ("411", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411)):
        ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 80, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf])
        files.append((name, buf))
    files.append(("gray", cv2.imencode(".jpg", img[:, :, 1], [cv2.IMWRITE_JPEG_QUALITY, 70])[1]))
    files.append(("progressive", cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1]))
    paths = []
    for name, buf in files:
        p = tmp_path / (name + ".jpg")
        p.write_bytes(bytes(buf))
        paths.append(str(p))
        want[name] = cv2.imdecode(buf, cv2.IMREAD_COLOR)
    res = subprocess.run([exe] + paths, capture_output=True, text=True, timeout=300)
    print(res.stdout, res.stderr)
    assert res.returncode == 0 and "ALL OK" in res.stdout
    for name, _ in files:
        p = tmp_path / (name + ".jpg")
        if name == "progressive":
            assert "refused %s" % p in res.stdout and "progressive" in res.stdout
            continue
        got = np.fromfile(str(p) + ".bgr", np.uint8).reshape(37, 61, 3)
        assert np.array_equal(got, want[name]), name
