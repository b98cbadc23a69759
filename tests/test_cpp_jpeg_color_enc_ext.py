"""jpegEncodeColor and degradeJPEGColor of include/filter_ext.h through cv::Mat: the streams equal cv2.imencode's bytes
for every sampling (and 4:2:0 by default), the round trips equal cv2.imdecode of them with their byte counts, and a CV_8UC1
source is refused."""
import os
import subprocess

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_jpeg_color_enc_ext.cpp")
SAMPLINGS = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
             "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411}


def _build(tmp_path):
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "test_jpeg_color_enc_ext")
    lib = os.path.join(ROOT, "depthmapcompression_b200")
    subprocess.check_call(["g++", "-O1", "-std=gnu++14", "-msse4.1", "-w", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "refshim"),
                           "-o", exe, SRC, "-L" + lib, "-ldmc_b200", "-ldl", "-Wl,-rpath," + lib])
    return exe


def test_jpeg_color_enc_ext_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_jpeg_color_enc_ext_matches_cv2(tmp_path):
    exe = _build(tmp_path)
    rows, cols, q = 37, 61, 80
    rs = np.random.RandomState(4)
    img = rs.randint(0, 256, (rows, cols, 3)).astype(np.uint8)
    src = tmp_path / "frame.bgr"
    img.tofile(str(src))
    res = subprocess.run([exe, str(src), str(rows), str(cols), str(q)], capture_output=True, text=True, timeout=300)
    print(res.stdout, res.stderr)
    assert res.returncode == 0 and "ALL OK" in res.stdout and "refused gray" in res.stdout
    for name, sf in SAMPLINGS.items():
        want = bytes(cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf])[1])
        assert (tmp_path / ("frame.bgr.%s.jpg" % name)).read_bytes() == want, name
        got = np.fromfile(str(tmp_path / ("frame.bgr.%s.bgr" % name)), np.uint8).reshape(rows, cols, 3)
        assert np.array_equal(got, cv2.imdecode(np.frombuffer(want, np.uint8), cv2.IMREAD_COLOR)), name
        assert "sampling %s %d %d" % (name, len(want), len(want)) in res.stdout
    assert (tmp_path / "frame.bgr.default.jpg").read_bytes() == bytes(cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])[1])
