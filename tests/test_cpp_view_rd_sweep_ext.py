"""jpegViewRateDistortionGray of include/filter_ext.h through cv::Mat: the stream sizes and the PSNR of the views rendered
from the coded and from the filtered depth must equal what jpegViewRateDistortion reports for the same frame, cameras and
chain, in both Huffman modes."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_view_rd_sweep_ext.cpp")
QUALITIES = (0, 20, 70, 100)


def _build(tmp_path):
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "test_view_rd_sweep_ext")
    lib = os.path.join(ROOT, "depthmapcompression_b200")
    subprocess.check_call(["g++", "-O1", "-std=gnu++14", "-msse4.1", "-w", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "refshim"),
                           "-o", exe, SRC, "-L" + lib, "-ldmc_b200", "-ldl", "-Wl,-rpath," + lib])
    return exe


def test_view_rd_sweep_ext_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_view_rd_sweep_ext_matches_python(tmp_path):
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
    got = {}
    for line in res.stdout.splitlines():
        if line.startswith("view "):
            _, opt, q, v, nb, pc, pf = line.split()
            got[(int(opt), int(q), int(v))] = (int(nb), float(pc), float(pf))
    K = np.eye(3) * f; K[0, 2] = (W - 1) * 0.5; K[1, 2] = (H - 1) * 0.5; K[2, 2] = 1.0
    R = np.stack([np.eye(3)] * 2); t = np.array([[tx, 0., 0.], [-tx, 0., 0.]])
    p = dmc.filters.chain_params(capi.CHAIN_DEPTH32F, 1, 0, 1, 3, 65.0, focus=75.0, baseline=575.0, amp=2.6)
    for opt in (0, 1):
        r = dmc.jpegViewRateDistortion(disp, tex, QUALITIES, p, f, R, t, K, isSub=True, optimize=bool(opt))
        for k, q in enumerate(QUALITIES):
            for v in range(2):
                nb, pc, pf = got[(opt, q, v)]
                assert nb == r["bytes"][k, 0], (opt, q, v)
                assert pc == r["psnr_view_coded"][k, v, 0] and pf == r["psnr_view_filtered"][k, v, 0], (opt, q, v)
