"""Property-style parity: hypothesis draws shapes, radii, thresholds, types and methods (the matrix of SURVEY.md 7.4)
and every drawn case must match the CPU oracle bit for bit."""
import numpy as np
import pytest

from _util import assert_bits_equal

hyp = pytest.importorskip("hypothesis")
from hypothesis import given, settings, strategies as st, HealthCheck  # noqa: E402

pytestmark = pytest.mark.gpu
COMMON = dict(max_examples=60, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def _image(seed, H, W, dtype, cn, smooth):
    rs = np.random.RandomState(seed)
    shape = (H, W) if cn == 1 else (H, W, cn)
    if smooth:
        blk = rs.randint(0, 256, size=((H + 5) // 6, (W + 5) // 6) + (() if cn == 1 else (cn,)))
        a = np.kron(blk, np.ones((6, 6) + (() if cn == 1 else (1,))))[:H, :W] + rs.randint(-5, 6, size=shape)
        a = np.clip(a, 0, 255)
    else:
        a = rs.randint(0, 256, size=shape)
    if dtype == np.uint16: a = a * 150 + rs.randint(0, 40, size=shape)
    elif dtype == np.int16: a = a * 150 - 19000
    elif dtype == np.float32: a = a * 2.5 + 0.5 * rs.randint(0, 3, size=shape)
    return np.ascontiguousarray(a.astype(dtype))


@settings(**COMMON)
@given(H=st.integers(1, 70), W=st.integers(1, 150), seed=st.integers(0, 10**6), smooth=st.booleans(),
       mr=st.integers(0, 3), gr=st.integers(0, 3), mmr=st.integers(0, 6), br=st.integers(0, 7), th=st.integers(0, 255),
       entry=st.sampled_from(["disp8u", "depth32f", "depth16u", "disp32f"]), method=st.sampled_from([0, 2]))
def test_chain_entry_points(dmc, port, H, W, seed, smooth, mr, gr, mmr, br, th, entry, method):
    a = np.maximum(_image(seed, H, W, np.uint8, 1, smooth), 1)
    pfs = dmc.PostFilterSet()
    if entry == "disp8u":
        assert_bits_equal(pfs(a, None, mr, gr, mmr, br, th, method), port.post_filter_set(a, mr, gr, mmr, br, th, method), "operator()")
    elif entry == "depth32f":
        assert_bits_equal(pfs.filterDisp8U2Depth32F(a, None, 75, 575, 2.6, mr, gr, mmr, br, th * 4.25, method),
                          port.filter_disp8u_depth32f(a, 75, 575, 2.6, mr, gr, mmr, br, th * 4.25, method), "Depth32F")
    elif entry == "depth16u":
        assert_bits_equal(pfs.filterDisp8U2Depth16U(a, None, 75, 575, 2.6, mr, gr, mmr, br, th * 4.25, method),
                          port.filter_disp8u_depth16u(a, 75, 575, 2.6, mr, gr, mmr, br, th * 4.25, method), "Depth16U")
    else:
        assert_bits_equal(pfs.filterDisp8U2Disp32F(a, None, mr, gr, mmr, br, th + 0.5, method),
                          port.filter_disp8u_disp32f(a, mr, gr, mmr, br, th + 0.5, method), "Disp32F")


@settings(**COMMON)
@given(H=st.integers(1, 60), W=st.integers(1, 140), seed=st.integers(0, 10**6), smooth=st.booleans(),
       kw=st.integers(0, 15), kh=st.integers(0, 15), th=st.floats(0, 255.9), method=st.sampled_from([0, 1, 2]),
       tc=st.sampled_from([(np.uint8, 1), (np.uint8, 3), (np.uint16, 1), (np.int16, 1), (np.uint16, 3), (np.int16, 3), (np.float32, 1), (np.float32, 3)]))
def test_range_filter(dmc, port, H, W, seed, smooth, kw, kh, th, method, tc):
    dt, cn = tc
    b = _image(seed, H, W, dt, cn, smooth)
    init = _image(seed + 1, H, W, dt, cn, False)
    want = port.bwrf(b, kw, kh, th, method, dst_init=init)
    got = dmc.binalyWeightedRangeFilter(b, init.copy(), (kw, kh), th, method)
    if dt != np.uint8 and (kw >> 1) % 8 == 5 and W % 4 == 0:        # reference reads past its padded buffer (undefined pixels)
        if method == 2: got[-(kh >> 1) - 1:, -1] = want[-(kh >> 1) - 1:, -1]
        elif (kh >> 1) == 0: got[-1, -1] = want[-1, -1]
    assert_bits_equal(got, want, "bwrf %dx%d th%.2f %sC%d m%d" % (kw, kh, th, dt.__name__, cn, method))


@settings(**COMMON)
@given(H=st.integers(1, 50), W=st.integers(1, 120), seed=st.integers(0, 10**6), smooth=st.booleans(), r=st.integers(0, 10),
       k=st.sampled_from([1, 3, 5, 7, 9]), dt=st.sampled_from([np.uint8, np.uint16, np.int16, np.float32, np.float64]),
       f=st.floats(0, 3), c=st.floats(0, 3), s=st.floats(0, 3))
def test_minmax_and_boundary_reconstruction(dmc, port, H, W, seed, smooth, r, k, dt, f, c, s):
    b = _image(seed, H, W, dt, 1, smooth) if dt != np.float64 else _image(seed, H, W, np.float32, 1, smooth).astype(np.float64)
    assert_bits_equal(dmc.blurRemoveMinMax(b, None, r), port.blur_remove_minmax(b, r), "blurRemoveMinMax")
    assert_bits_equal(dmc.boundaryReconstructionFilter(b, None, (k, k), f, c, s), port.brf(b, k, k, np.float32(f), np.float32(c), np.float32(s)), "BRF")
