"""The PSNR of a rendered view (psnrFromSSE over 3 * rows * cols bytes, as jpegViewRateDistortion reports it) against
cv2.PSNR of the two 8UC3 images, which averages the squared error over the channels.  Host only: the SSE is computed here
with numpy and the formula needs no GPU."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def dmc():
    import __graft_entry__ as g
    g.build()
    import depthmapcompression_b200 as m
    return m


def test_psnr_of_8uc3_views_matches_cv2(dmc):
    from depthmapcompression_b200 import capi
    rs = np.random.RandomState(23)
    for H, W, spread in [(1, 1, 255), (3, 3, 7), (17, 23, 40), (61, 83, 1), (480, 640, 20), (1080, 1920, 255)]:
        a = rs.randint(0, 256, (H, W, 3)).astype(np.uint8)
        b = np.clip(a.astype(np.int16) + rs.randint(-spread, spread + 1, a.shape), 0, 255).astype(np.uint8)
        b[: H // 2, : W // 3] = 0                                       # holes, as a render leaves them
        sse = int(((a.astype(np.int64) - b) ** 2).sum())
        ref = cv2.PSNR(a, b)
        assert abs(capi.lib.dmc_psnr_from_sse(sse, 3 * H * W) - ref) < 1e-9, (H, W)
        assert abs(dmc.psnrFromSSE(sse, 3 * H * W) - ref) < 1e-9, (H, W)
        got = dmc.psnrFromSSE(np.full((2, 3, 1), sse, np.uint64), 3 * H * W)     # the (n_q, n_views, n) shape of the sweep
        assert got.shape == (2, 3, 1) and np.all(np.abs(got - ref) < 1e-9)
    a = rs.randint(0, 256, (37, 53, 3)).astype(np.uint8)
    assert abs(cv2.PSNR(a, a.copy()) - dmc.psnrFromSSE(0, a.size)) < 1e-9
