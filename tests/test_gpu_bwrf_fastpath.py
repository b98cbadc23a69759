"""The flat-warp path of the 8-bit range filter (dmc_bwrf8u_h2.cu): warps whose footprint lies within th of every
centre compute the disc mean instead of running the tap loop.  Inputs are built so that fast warps, slow warps and
tiles mixing both occur, at the test's boundary (max(F) - min(centres) == th and th + 1), at every image edge, on
partial tiles and unaligned device pointers, for every radius on both sides of the FLUSH limit; each output is compared
bit for bit with the CPU oracle.  Run with `-m gpu` on a B200."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)          # raises loudly without a GPU / without the built library
    return m


def ntaps(r):
    n = 0
    for dy in range(-r, r + 1):
        lim, j = r * r - dy * dy, 0
        while (j + 1) * (j + 1) <= lim:
            j += 1
        n += 2 * j + 1
    return n


def flat_mix(rs, H, W, amp, noisy_share=0.3):
    """plateaus of 64 x 16 pixels with noise of +-amp, a share of them replaced by full-range noise"""
    by, bx = (H + 15) // 16, (W + 63) // 64
    lvl = rs.randint(20, 236, size=(by, bx))
    a = np.kron(lvl, np.ones((16, 64), np.int64))[:H, :W] + rs.randint(-amp, amp + 1, size=(H, W))
    noisy = np.kron(rs.rand(by, bx) < noisy_share, np.ones((16, 64), bool))[:H, :W]
    a[noisy] = rs.randint(0, 256, size=int(noisy.sum()))
    return np.clip(a, 0, 255).astype(np.uint8)


def bwrf(dmc, img, r, th):
    return dmc.binalyWeightedRangeFilter(img, None, (2 * r + 1, 2 * r + 1), th, dmc.FULL_KERNEL)


def check(dmc, port, img, r, th, what=""):
    got, want = bwrf(dmc, img, r, th), port.bwrf(img, 2 * r + 1, 2 * r + 1, th)
    bad = np.argwhere(got != want)
    assert bad.size == 0, "%s r=%d th=%d shape=%s: %d pixels differ, first at %s" % (what, r, th, img.shape, len(bad), bad[:3].tolist())


@pytest.mark.parametrize("r", range(1, 11))
def test_every_radius_both_sides_of_flush(dmc, port, r):
    """ntaps*th <= 2048 runs the half accumulator alone, above it the FLUSH variant; (2r+1)*th <= 2048 bounds th"""
    rs = np.random.RandomState(100 + r)
    for th in sorted({0, 1, 2048 // ntaps(r), 2048 // ntaps(r) + 1, 2048 // (2 * r + 1)}):
        img = flat_mix(rs, 96, 300, amp=max(1, th // 4))
        check(dmc, port, img, r, th, "flat_mix")


@pytest.mark.parametrize("r", [1, 2, 5, 7, 10])
def test_threshold_boundary(dmc, port, r):
    """one halo pixel at c0 + th (the warp passes: max(F) - min(centres) == th) and at c0 + th + 1 (it does not), in
    every position around a warp block, both above and below the plateau"""
    rs = np.random.RandomState(7)
    th, c0 = 10, 120
    for delta in (th, th + 1, -th, -(th + 1)):
        img = np.full((64, 256), c0, np.uint8)
        for y, x in [(3, 63), (4, 64), (0, 0), (63, 255), (16 + r, 130), (20, 64 + 63 + r), (33, 128 - r)]:
            img[y, x] = c0 + delta
        img[40:48, 160:200] = c0 + rs.randint(-th // 2, th // 2 + 1, size=(8, 40))
        check(dmc, port, img, r, th, "boundary %+d" % delta)


@pytest.mark.parametrize("r", [1, 3, 5, 10])
def test_th0_constant_regions(dmc, port, r):
    rs = np.random.RandomState(3)
    img = np.kron(rs.randint(0, 256, size=(6, 5)), np.ones((24, 80), np.int64)).astype(np.uint8)
    img[100:110, 10:20] = rs.randint(0, 256, size=(10, 10))
    check(dmc, port, img, r, 0, "th0")
    check(dmc, port, np.full((50, 333), 255, np.uint8), r, 0, "th0 const")


@pytest.mark.parametrize("shape", [(1, 1), (1, 129), (7, 1), (17, 127), (37, 53), (83, 131), (100, 1023), (257, 385), (1080, 1920)])
def test_fast_warps_touch_every_edge(dmc, port, shape):
    """smooth frames (every warp fast) and frames with plateaus reaching all four borders, incl. partial tiles"""
    H, W = shape
    rs = np.random.RandomState(H * 7 + W)
    yy, xx = np.mgrid[0:H, 0:W]
    smooth = (100 + 3 * np.sin(yy / 9.0) + 3 * np.cos(xx / 11.0)).round().astype(np.uint8)
    for r in (1, 5, 10):
        check(dmc, port, smooth, r, 10, "smooth")
    check(dmc, port, flat_mix(rs, H, W, 2), 5, 10, "flat_mix")


@pytest.mark.parametrize("offs", [(0, 0), (1, 0), (0, 1), (3, 5), (15, 17)])
@pytest.mark.parametrize("shape", [(64, 128), (61, 131), (33, 1919)])
def test_unaligned_device_pointers(dmc, port, offs, shape):
    """device images at odd byte offsets (16-byte staging loads and 2-byte stores are off) and odd widths"""
    import torch
    from depthmapcompression_b200.capi import DmcImage, lib
    H, W = shape
    rs = np.random.RandomState(H + W + offs[0])
    img = flat_mix(rs, H, W, 3)
    so, do = offs
    d_in = torch.zeros(H * W + 64, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(H * W + 64, dtype=torch.uint8, device="cuda")
    d_in[so:so + H * W] = torch.from_numpy(img.reshape(-1)).cuda()
    torch.cuda.synchronize()                # the copy runs on torch's stream, the filter on the context's own
    ctx = dmc.default_context(0)
    for r in (2, 5):
        s8 = DmcImage(d_in.data_ptr() + so, H, W, 0, W, 1)
        o8 = DmcImage(d_out.data_ptr() + do, H, W, 0, W, 1)
        ctx.check(lib.dmc_bwrf(ctx.h, C.byref(s8), C.byref(o8), 2 * r + 1, 2 * r + 1, 10.0, 0, 1))
        torch.cuda.synchronize()
        got = d_out[do:do + H * W].cpu().numpy().reshape(H, W)
        assert np.array_equal(got, port.bwrf(img, 2 * r + 1, 2 * r + 1, 10)), (r, offs, shape)


def test_bench_video_frames_through_chain(dmc, port):
    """two frames of bench.py's 1080p video through PostFilterSet()(2,1,3,5,10) and the range filter on its real input"""
    import cv2
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    y = cv2.imread(os.path.join(root, "tests", "golden", "x264_depth_y.png"), cv2.IMREAD_UNCHANGED)
    base = np.ascontiguousarray(np.tile(y, (3, 3))[:1080, :1920])
    pfs = dmc.PostFilterSet()
    for f in (0, 500):
        frame = np.ascontiguousarray(np.roll(base, (f % 1080, (2 * f) % 1920), axis=(0, 1)))
        assert np.array_equal(pfs(frame, None, 2, 1, 3, 5, 10), port.post_filter_set(frame, 2, 1, 3, 5, 10)), f
        rf_in = port.blur_remove_minmax(port.small_gaussian(port.median_blur(frame, 5), 3, 1.5), 3)
        check(dmc, port, rf_in, 5, 10, "video frame %d" % f)
