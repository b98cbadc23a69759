"""The float64 SSIM reference the GPU tests compare with (Wang, Bovik, Sheikh and Simoncelli 2004, ssim_index.m; equal to
skimage.metrics.structural_similarity(a, b, data_range=255, gaussian_weights=True, sigma=1.5, use_sample_covariance=False),
channels averaged): separable 11-tap Gaussian moments with scipy.ndimage.correlate1d, cropped to the window positions that lie
inside the frame.  Checked here against a brute-force loop over the 2-D window, against the closed form of flat frames, and
for identical frames."""
import numpy as np
import pytest
from scipy.ndimage import correlate1d

C1, C2 = (0.01 * 255) ** 2, (0.03 * 255) ** 2
R = 5


def gauss():
    i = np.arange(-R, R + 1, dtype=np.float64)
    g = np.exp(-(i * i) / 4.5)
    return g / g.sum()


def _window(x, g):
    y = correlate1d(correlate1d(x, g, axis=0, mode="reflect"), g, axis=1, mode="reflect")
    return y[R:-R, R:-R]


def _mssim_gray(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    g = gauss()
    mx, my = _window(a, g), _window(b, g)
    sxx = _window(a * a, g) - mx * mx
    syy = _window(b * b, g) - my * my
    sxy = _window(a * b, g) - mx * my
    s = ((2 * mx * my + C1) * (2 * sxy + C2)) / ((mx * mx + my * my + C1) * (sxx + syy + C2))
    return s.mean()


def ssim_ref(a, b):
    """MSSIM of one uint8 frame pair: [rows, cols] or [rows, cols, 3] (the mean of the channels' MSSIMs)"""
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and min(a.shape[:2]) >= 2 * R + 1
    if a.ndim == 3:
        return float(np.mean([_mssim_gray(a[..., c], b[..., c]) for c in range(a.shape[2])]))
    return float(_mssim_gray(a, b))


def ssim_ref_batch(a, b):
    """float64[n] of a batch [n, rows, cols] or [n, rows, cols, 3]"""
    return np.array([ssim_ref(x, y) for x, y in zip(a, b)], np.float64)


def _brute(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    w = np.outer(gauss(), gauss())
    H, W = a.shape
    s = []
    for y in range(H - 2 * R):
        for x in range(W - 2 * R):
            pa, pb = a[y:y + 2 * R + 1, x:x + 2 * R + 1], b[y:y + 2 * R + 1, x:x + 2 * R + 1]
            mx, my = (w * pa).sum(), (w * pb).sum()
            sxx, syy, sxy = (w * pa * pa).sum() - mx * mx, (w * pb * pb).sum() - my * my, (w * pa * pb).sum() - mx * my
            s.append(((2 * mx * my + C1) * (2 * sxy + C2)) / ((mx * mx + my * my + C1) * (sxx + syy + C2)))
    return float(np.mean(s))


def test_gauss_window():
    g = gauss()
    assert abs(g.sum() - 1.0) < 1e-15 and np.array_equal(g, g[::-1])
    # the taps the kernel carries as literals (csrc/dmc_metrics.cu)
    assert g[R:].tolist() == [0.26601172486179436, 0.2130055377112537, 0.10936068950970002, 0.03600077212843083,
                              0.007598758135239185, 0.00102838008447911]


@pytest.mark.parametrize("H,W", [(11, 11), (11, 17), (19, 11), (12, 13), (23, 29)])
def test_separable_equals_brute_force(H, W):
    rs = np.random.RandomState(H * 31 + W)
    a = rs.randint(0, 256, (H, W)).astype(np.uint8)
    b = np.clip(a.astype(np.int32) + rs.randint(-40, 41, (H, W)), 0, 255).astype(np.uint8)
    c = rs.randint(0, 256, (H, W)).astype(np.uint8)
    for x, y in ((a, b), (a, c), (np.zeros_like(a), np.full_like(a, 255))):
        assert abs(ssim_ref(x, y) - _brute(x, y)) <= 1e-13


def test_colour_is_mean_of_channels():
    rs = np.random.RandomState(3)
    a = rs.randint(0, 256, (15, 16, 3)).astype(np.uint8)
    b = rs.randint(0, 256, (15, 16, 3)).astype(np.uint8)
    assert abs(ssim_ref(a, b) - np.mean([_brute(a[..., c], b[..., c]) for c in range(3)])) <= 1e-13


def test_flat_frames_closed_form():
    for u, v in ((0, 0), (0, 255), (17, 200), (255, 255)):
        a, b = np.full((14, 12), u, np.uint8), np.full((14, 12), v, np.uint8)
        assert abs(ssim_ref(a, b) - (2.0 * u * v + C1) / (u * u + v * v + C1)) <= 1e-12


def test_identical_frames_give_one():
    rs = np.random.RandomState(5)
    for shape in ((11, 11), (40, 57), (33, 21, 3)):
        a = rs.randint(0, 256, shape).astype(np.uint8)
        assert abs(ssim_ref(a, a) - 1.0) <= 1e-12
