"""prepareDisparityBatch and renderViewBatch of include/filter_ext.h through cv::Mat: the disparities (one and two passes)
and the views of the prepared depth must equal what the Python prepareDisparityBatch and renderViewBatch return."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_pointcloud_batch_ext.cpp")
FB, AMP = 75.0 * 575.0, 2.6


def _build(tmp_path):
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "test_pointcloud_batch_ext")
    lib = os.path.join(ROOT, "depthmapcompression_b200")
    subprocess.check_call(["g++", "-O1", "-std=gnu++14", "-msse4.1", "-w", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "refshim"),
                           "-o", exe, SRC, "-L" + lib, "-ldmc_b200", "-ldl", "-Wl,-rpath," + lib])
    return exe


def test_pointcloud_batch_ext_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_pointcloud_batch_ext_matches_python(tmp_path):
    from _util import load_png
    import depthmapcompression_b200 as dmc
    exe = _build(tmp_path)
    d16 = load_png("kinect_meeting_depth16_crop.png")
    H, W = d16.shape
    rs = np.random.RandomState(4)
    frames = np.stack([d16, np.roll(d16, 17, axis=1), np.where(rs.rand(H, W) < 0.3, 0, d16).astype(np.uint16)])
    n = len(frames)
    tex = rs.randint(0, 256, (n, H, W, 3)).astype(np.uint8)
    f, tx = 510.0, 100.0
    frames.tofile(str(tmp_path / "depth16.raw")); tex.tofile(str(tmp_path / "tex.raw"))
    res = subprocess.run([exe, str(tmp_path / "depth16.raw"), str(tmp_path / "tex.raw"), str(n), str(H), str(W), repr(f), repr(tx), str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    print(res.stdout, res.stderr)
    assert res.returncode == 0 and "ALL OK" in res.stdout
    for passes in (1, 2):
        got = np.fromfile(str(tmp_path / ("disp%d.raw" % passes)), np.uint8).reshape(n, H, W)
        assert np.array_equal(got, dmc.prepareDisparityBatch(frames, FB, AMP, passes=passes)), passes
    disp = dmc.prepareDisparityBatch(frames, FB, AMP, passes=2)
    depth = np.stack([dmc.disp8U2depth32F(x, None, FB, AMP, 0.0) for x in disp])
    K = np.eye(3) * f; K[0, 2] = (W - 1) * 0.5; K[1, 2] = (H - 1) * 0.5; K[2, 2] = 1.0
    R = np.stack([np.eye(3)] * 2); t = np.array([[tx, 0., 0.], [-tx, 0., 0.]])
    want = dmc.renderViewBatch(depth, tex, f, R, t, K, isSub=True)
    got = np.fromfile(str(tmp_path / "views.raw"), np.uint8).reshape(want.shape)
    assert np.array_equal(got, want)
