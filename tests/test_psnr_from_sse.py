"""The PSNR of the rate-distortion sweep (dmc_psnr_from_sse, psnrFromSSE) against cv2.PSNR.  Host only: the formula is
evaluated on the CPU and needs no GPU; the SSE is computed here with numpy."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def dmc():
    import __graft_entry__ as g
    g.build()
    import depthmapcompression_b200 as m
    return m


def np_sse(a, b):
    return int(((a.astype(np.int64) - b) ** 2).sum())


def test_psnr_from_sse_matches_cv2(dmc):
    from depthmapcompression_b200 import capi
    rs = np.random.RandomState(11)
    sses, pixels, want = [], [], []
    for H, W, spread in [(1, 1, 255), (5, 1, 3), (7, 13, 40), (83, 131, 1), (480, 640, 20), (1080, 1920, 255), (3, 10000, 2)]:
        for _ in range(4):
            a = rs.randint(0, 256, (H, W)).astype(np.uint8)
            b = np.clip(a.astype(np.int16) + rs.randint(-spread, spread + 1, a.shape), 0, 255).astype(np.uint8)
            s = np_sse(a, b)
            ref = cv2.PSNR(a, b)
            assert abs(capi.lib.dmc_psnr_from_sse(s, H * W) - ref) < 1e-9, (H, W, spread)
            assert abs(dmc.psnrFromSSE(s, H * W) - ref) < 1e-9
            sses.append(s); pixels.append(H * W); want.append(ref)
    got = dmc.psnrFromSSE(np.array(sses, np.uint64), np.array(pixels, np.uint64))
    assert got.shape == (len(want),) and np.all(np.abs(got - np.array(want)) < 1e-9)
    full = np_sse(np.zeros((1080, 1920), np.uint8), np.full((1080, 1920), 255, np.uint8))
    assert abs(dmc.psnrFromSSE(full, 1080 * 1920) - cv2.PSNR(np.zeros((1080, 1920), np.uint8), np.full((1080, 1920), 255, np.uint8))) < 1e-9


def test_psnr_of_identical_frames(dmc):
    from depthmapcompression_b200 import capi
    a = np.random.RandomState(3).randint(0, 256, (37, 53)).astype(np.uint8)
    assert abs(cv2.PSNR(a, a.copy()) - 361.20199909921956) < 1e-9
    assert abs(capi.lib.dmc_psnr_from_sse(0, a.size) - 361.20199909921956) < 1e-9
    assert abs(dmc.psnrFromSSE(0, a.size) - 361.20199909921956) < 1e-9
    assert np.all(np.abs(dmc.psnrFromSSE(np.zeros((2, 3), np.uint64), a.size) - 361.20199909921956) < 1e-9)
