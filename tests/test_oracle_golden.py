"""The CPU restatement (oracle/dmc_oracle.c) and, where present, the compiled reference
(oracle/_ref/libdmc_ref.so) against the committed golden vectors (tests/golden/golden.json)."""
import numpy as np
import pytest

from _util import crc, load_golden, load_png
from oracle.oracle_py import SEPARABLE_KERNEL, FILL_DISPARITY

FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6
GOLD = load_golden()
CHAIN_INPUTS = [k for k in GOLD["inputs"] if "depth16" not in k]


def run_chain_op(L, key, img):
    fb = FOCUS * BASELINE
    if key == "pfs_2_1_3_5_10": return L.post_filter_set(img, 2, 1, 3, 5, 10)
    if key == "pfs_1_0_1_3_10": return L.post_filter_set(img, 1, 0, 1, 3, 10)
    if key == "pfs_2_1_3_5_10_sep": return L.post_filter_set(img, 2, 1, 3, 5, 10, SEPARABLE_KERNEL)
    if key == "depth32f_1_0_1_3_65": return L.filter_disp8u_depth32f(img, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0)
    if key == "depth16u_1_0_1_3_65": return L.filter_disp8u_depth16u(img, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0)
    if key == "disp32f_1_0_1_3_10": return L.filter_disp8u_disp32f(img, 1, 0, 1, 3, 10.0)
    if key == "depth32f2disp8u": return L.depth32f2disp8u(L.filter_disp8u_depth32f(img, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0), fb, AMP, 0.0)
    if key == "reproject_xyz_510": return L.reproject_xyz(L.filter_disp8u_depth32f(img, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0), 510.0)
    if key == "brf_13_1_1_1": return L.brf(img, 13, 13, 1, 1, 1)
    if key == "brf_7_1_2_05": return L.brf(img, 7, 7, 1, 2, 0.5)
    if key.startswith("bwrf8u_r"): r = int(key[8]); return L.bwrf(img, 2 * r + 1, 2 * r + 1, 10)
    if key == "bwrf8u_sep_11_th10": return L.bwrf(img, 11, 11, 10, SEPARABLE_KERNEL)
    if key == "bwrf32f_r3_th65": return L.bwrf(img.astype(np.float32) * 16.0, 7, 7, 65.0)
    if key == "bwrf32f_r5_th65": return L.bwrf(img.astype(np.float32) * 16.0, 11, 11, 65.0)
    if key == "bwrf16u_r2_th160": return L.bwrf(img.astype(np.uint16) * 16, 5, 5, 160.0)
    if key.startswith("minmax_r"): return L.blur_remove_minmax(img, int(key[8:]))
    if key.startswith("median_k"): return L.median_blur(img, int(key[8:]))
    if key.startswith("gauss_gr"): gr = int(key[8:]); return L.small_gaussian(img, 2 * gr + 1, gr + 0.5)
    if key == "disp8u2depth32f": return L.disp8u2depth32f(img, fb, AMP, 0.0)
    raise KeyError(key)


def run_depth16_op(L, key, d16):
    fb = FOCUS * BASELINE
    if key == "depth16u2disp8u": return L.depth16u2disp8u(d16, fb, AMP, 0.0)
    if key == "fill_disparity_1pass": return L.fill_occlusion(L.depth16u2disp8u(d16, fb, AMP, 0.0), 0, FILL_DISPARITY)
    if key == "fill_disparity_2pass":
        f = L.fill_occlusion(L.depth16u2disp8u(d16, fb, AMP, 0.0), 0, FILL_DISPARITY)
        t = L.fill_occlusion(np.ascontiguousarray(f.T), 0, FILL_DISPARITY)
        return np.ascontiguousarray(t.T)
    if key == "reproject_xyz_16u_510": return L.reproject_xyz(d16, 510.0)
    raise KeyError(key)


def test_fixture_files_intact():
    assert GOLD["survey_8c_known_answers_reproduced"] is True
    for name, ent in GOLD["inputs"].items():
        assert crc(load_png(name)) == ent["crc"], name


@pytest.mark.parametrize("name", CHAIN_INPUTS)
def test_port_matches_golden_chain(port, name):
    img = load_png(name)
    for key, want in GOLD["inputs"][name]["golden"].items():
        assert crc(run_chain_op(port, key, img)) == want, (name, key)


def test_port_matches_golden_depth16(port):
    name = "kinect_meeting_depth16_crop.png"; d16 = load_png(name)
    for key, want in GOLD["inputs"][name]["golden"].items():
        assert crc(run_depth16_op(port, key, d16)) == want, key


@pytest.mark.parametrize("name", CHAIN_INPUTS[:2])
def test_reference_build_matches_golden(ref_build, name):
    """Guards against shim / compiler-flag drift of oracle/_ref."""
    img = load_png(name)
    for key, want in GOLD["inputs"][name]["golden"].items():
        assert crc(run_chain_op(ref_build, key, img)) == want, (name, key)
