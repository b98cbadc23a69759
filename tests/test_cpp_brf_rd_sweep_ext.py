"""The BRF overloads of jpegRateDistortionGray and jpegViewRateDistortionGray (include/filter_ext.h) through cv::Mat: stream
sizes and the PSNR of the coded, post-filtered and boundary-reconstructed frames and views must equal what
jpegRateDistortion / jpegViewRateDistortion report with brf=brf_params((13, 13), 1, 1, 1), in both Huffman modes."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_brf_rd_sweep_ext.cpp")
QUALITIES = (0, 20, 70, 100)


def _build(tmp_path):
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "test_brf_rd_sweep_ext")
    lib = os.path.join(ROOT, "depthmapcompression_b200")
    subprocess.check_call(["g++", "-O1", "-std=gnu++14", "-msse4.1", "-w", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "refshim"),
                           "-o", exe, SRC, "-L" + lib, "-ldmc_b200", "-ldl", "-Wl,-rpath," + lib])
    return exe


def test_brf_rd_sweep_ext_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_brf_rd_sweep_ext_matches_python(tmp_path):
    from _util import load_png
    import depthmapcompression_b200 as dmc
    from depthmapcompression_b200 import capi
    exe = _build(tmp_path)
    disp = load_png("kinect_meeting_q80.png")
    H, W = disp.shape
    tex = np.stack([disp, 255 - disp, disp // 2 + 1], -1)
    f, tx = 510.0, 100.0
    disp.tofile(str(tmp_path / "disp.raw")); tex.tofile(str(tmp_path / "tex.raw"))
    res = subprocess.run([exe, str(tmp_path / "disp.raw"), str(tmp_path / "tex.raw"), str(H), str(W), repr(f), repr(tx)] + [str(q) for q in QUALITIES],
                         capture_output=True, text=True, timeout=600)
    print(res.stdout, res.stderr)
    assert res.returncode == 0 and "ALL OK" in res.stdout
    gray, view = {}, {}
    for line in res.stdout.splitlines():
        w = line.split()
        if w and w[0] == "gray":
            gray[(int(w[1]), int(w[2]))] = (int(w[3]), float(w[4]), float(w[5]), float(w[6]))
        elif w and w[0] == "view":
            view[(int(w[1]), int(w[2]), int(w[3]))] = (int(w[4]), float(w[5]), float(w[6]), float(w[7]))
    b = dmc.brf_params((13, 13), 1.0, 1.0, 1.0)
    K = np.eye(3) * f; K[0, 2] = (W - 1) * 0.5; K[1, 2] = (H - 1) * 0.5; K[2, 2] = 1.0
    R = np.stack([np.eye(3)] * 2); t = np.array([[tx, 0., 0.], [-tx, 0., 0.]])
    pg = dmc.filters.chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10)
    pv = dmc.filters.chain_params(capi.CHAIN_DEPTH32F, 1, 0, 1, 3, 65.0, focus=75.0, baseline=575.0, amp=2.6)
    for opt in (0, 1):
        r = dmc.jpegRateDistortion(disp, QUALITIES, pg, optimize=bool(opt), brf=b)
        rv = dmc.jpegViewRateDistortion(disp, tex, QUALITIES, pv, f, R, t, K, isSub=True, optimize=bool(opt), brf=b)
        for k, q in enumerate(QUALITIES):
            assert gray[(opt, q)] == (r["bytes"][k, 0], r["psnr_coded"][k, 0], r["psnr_filtered"][k, 0], r["psnr_brf"][k, 0]), (opt, q)
            for v in range(2):
                assert view[(opt, q, v)] == (rv["bytes"][k, 0], rv["psnr_view_coded"][k, v, 0], rv["psnr_view_filtered"][k, v, 0],
                                             rv["psnr_view_brf"][k, v, 0]), (opt, q, v)
