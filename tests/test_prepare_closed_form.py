"""The closed form that dmc_prepare.cu's fill kernels compute (stated in the comment at the top of that file), restated in
numpy and checked against the oracle's serial fillOcclusion (FILL_DISPARITY, invalid 0) on every row of up to 14 pixels
over a small alphabet: invalid (0), the edge value (255) and interior values.  CPU only."""
import itertools

import numpy as np
import pytest

FILL_DISPARITY = 0


def closed_form(rows):
    """rows: uint8 [m, n], n >= 2 -> every row filled independently, as fillOcclusion fills it."""
    e = rows.astype(np.int32).copy()
    m, n = e.shape
    e[:, 0] = 255; e[:, -1] = 255
    valid = e != 0
    idx = np.broadcast_to(np.arange(n), e.shape)
    left = np.maximum.accumulate(np.where(valid, idx, 0), axis=1)                 # nearest valid at or left of p
    right = np.minimum.accumulate(np.where(valid, idx, n - 1)[:, ::-1], axis=1)[:, ::-1]   # nearest valid at or right of p
    run = right - left - 1                                                         # the run a zero lies in
    over = ((~valid) & (run > int(n * 0.5))).any(axis=1)
    f = np.where(valid, e, np.minimum(np.take_along_axis(e, left, 1), np.take_along_axis(e, right, 1)))
    f[:, 0] = f[:, 1]; f[:, -1] = f[:, -2]
    f[over] = 0
    return f.astype(np.uint8)


def serial(port, img):
    """The oracle's serial fill of img.  A row blanked to 0 reads the next row's first pixel, which is undefined past the
    last row, so a guard row that never blanks goes last."""
    guard = np.full((1, img.shape[1]), 7, np.uint8)
    return port.fill_occlusion(np.vstack([img, guard]), 0, FILL_DISPARITY)[:-1]


def all_rows(n, alphabet):
    return np.array(list(itertools.product(alphabet, repeat=n)), np.uint8)


@pytest.mark.parametrize("n", range(2, 15))
def test_closed_form_equals_serial_fill(port, n):
    alphabets = [(0, 7, 255)] + ([(0, 3, 9, 255)] if n <= 11 else [])
    for alphabet in alphabets:
        rows = all_rows(n, alphabet)
        # one image of all patterns: the serial loop reads the next row's first pixel after a blanked row, which the
        # closed form says never matters, so the row order must not matter either
        for img in (rows, rows[::-1].copy()):
            want = serial(port, img)
            assert np.array_equal(closed_form(img), want), (n, alphabet)


def test_closed_form_column_pass_equals_two_serial_passes(port):
    """pointcloudTest's second pass (transpose, fill, transpose) is the closed form down every column."""
    rs = np.random.RandomState(3)
    for H, W in ((2, 2), (3, 17), (17, 3), (61, 83), (40, 9)):
        for p0 in (0.2, 0.5, 0.8):
            img = np.where(rs.rand(H, W) < p0, 0, rs.randint(1, 256, (H, W))).astype(np.uint8)
            one = serial(port, img)
            assert np.array_equal(closed_form(img), one)
            two = serial(port, np.ascontiguousarray(one.T)).T
            assert np.array_equal(closed_form(np.ascontiguousarray(one.T)).T, two), (H, W, p0)
