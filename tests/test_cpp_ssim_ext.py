"""structuralSimilarity (include/filter_ext.h) through cv::Mat: the SSIM of CV_8UC3 and CV_8UC1 images, of a region of interest
with a wider row step and of an image with itself must equal, bit for bit, what frameSSIM reports for the same pixels."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_ssim_ext.cpp")


def _build(tmp_path):
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "test_ssim_ext")
    lib = os.path.join(ROOT, "depthmapcompression_b200")
    subprocess.check_call(["g++", "-O1", "-std=gnu++14", "-msse4.1", "-w", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "refshim"),
                           "-o", exe, SRC, "-L" + lib, "-ldmc_b200", "-ldl", "-Wl,-rpath," + lib])
    return exe


def test_ssim_ext_compiles_and_links(tmp_path):
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_ssim_ext_matches_python(tmp_path):
    import depthmapcompression_b200 as dmc
    from oracle.oracle_py import synth_disp, degrade_blocks
    exe = _build(tmp_path)
    H, W = 97, 131
    d = synth_disp(H, W, 4)
    a = np.stack([d, 255 - d, (d // 3).astype(np.uint8)], -1)
    b = np.stack([degrade_blocks(a[..., c], 5 + c) for c in range(3)], -1)
    a.tofile(str(tmp_path / "a.raw")); b.tofile(str(tmp_path / "b.raw"))
    res = subprocess.run([exe, str(tmp_path / "a.raw"), str(tmp_path / "b.raw"), str(H), str(W)], capture_output=True, text=True, timeout=600)
    print(res.stdout, res.stderr)
    assert res.returncode == 0 and "ALL OK" in res.stdout
    got = dict((w[0], float(w[1])) for w in (line.split() for line in res.stdout.splitlines()) if len(w) == 2 and w[0] != "ALL")
    want = {"c3": dmc.frameSSIM(a, b)[0], "c1": dmc.frameSSIM(a[..., 0], b[..., 0])[0],
            "roi": dmc.frameSSIM(a[2:H - 3, 3:W - 4, 0], b[2:H - 3, 3:W - 4, 0])[0], "self": dmc.frameSSIM(a, a)[0]}
    for k, v in want.items():
        assert got[k] == v, (k, got[k], v)
    assert want["self"] == 1.0 or abs(want["self"] - 1.0) < 1e-12
