"""The per-strip flat test and the strip regrouping of the 8-bit range filter (dmc_bwrf8u_h2.cu).  A thread's strip is
2 pixels by R rows, a tile is 128 pixels by 4R rows (256 strips), and the CTA hands flat strips to its first threads and
tap strips to the rest.  The inputs choose, strip by strip, which strips take the tap loop: a tap strip gets centres
c0 - a and c0 + a with 2a > th, a flat strip c0, so every strip next to a tap strip still passes (its footprint lies
within a <= th of its centres) and each tile holds exactly the number of tap strips asked for.  Every output is
compared bit for bit with the CPU oracle.  Run with `-m gpu` on a B200."""
import ctypes as C

import numpy as np
import pytest

from _util import ntaps

pytestmark = pytest.mark.gpu

C0 = 128


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)          # raises loudly without a GPU / without the built library
    return m


def rows_per_thread(r, H, W):
    """R of the launch, as launch_rad picks it (few tiles: R = 2)"""
    R = 8 if r <= 3 else (4 if r <= 6 else (2 if r <= 8 else 1))
    if R > 2 and ((W + 127) // 128) * ((H + 4 * R - 1) // (4 * R)) < 2 * 148:
        R = 2
    return R


def words_each_side(r):
    return 6 if r <= 6 else (8 if r <= 8 else 10)


def strip_image(tap, H, W, R, a):
    """tap[sy, sx] per strip (R rows x 2 pixels): tap strips get c0 +- a in a checkerboard, the others c0"""
    yy, xx = np.mgrid[0:H, 0:W]
    t = tap[yy // R, xx // 2]
    img = np.full((H, W), C0, np.int64)
    img[t] = (C0 + np.where((yy + xx) % 2 == 0, a, -a))[t]
    return np.clip(img, 0, 255).astype(np.uint8)


def taps_per_tile(rs, H, W, R, counts):
    """tap-strip mask with counts[i % len(counts)] tap strips (at random places) in the i-th tile; a partial tile gets
    as many of its in-image strips as it has"""
    sy, sx = (H + R - 1) // R, (W + 1) // 2
    tap = np.zeros((sy, sx), bool)
    i = 0
    for ty in range(0, sy, 4):
        for tx in range(0, sx, 64):
            blk = tap[ty:ty + 4, tx:tx + 64]
            k = min(counts[i % len(counts)], blk.size)
            blk[np.unravel_index(rs.choice(blk.size, k, replace=False), blk.shape)] = True
            i += 1
    return tap


def bwrf(dmc, img, r, th):
    return dmc.binalyWeightedRangeFilter(img, None, (2 * r + 1, 2 * r + 1), th, dmc.FULL_KERNEL)


def check(dmc, port, img, r, th, what=""):
    got, want = bwrf(dmc, img, r, th), port.bwrf(img, 2 * r + 1, 2 * r + 1, th)
    bad = np.argwhere(got != want)
    assert bad.size == 0, "%s r=%d th=%d shape=%s: %d pixels differ, first at %s" % (what, r, th, img.shape, len(bad), bad[:3].tolist())


# (H, W) with at least 296 tiles at R = 4 (the radius-5 launch keeps R = 4) and with few tiles (R = 2)
SHAPES_R5 = {"R4": (640, 1024), "R2": (64, 384)}


@pytest.mark.parametrize("path", sorted(SHAPES_R5))
def test_tap_strip_counts(dmc, port, path):
    """1, 31, 32, 33, 224 and 255 tap strips in a tile: the boundary between the flat and the tap threads falls inside a
    warp, on a warp edge and next to one"""
    H, W = SHAPES_R5[path]
    R = rows_per_thread(5, H, W)
    assert R == int(path[1])
    rs = np.random.RandomState(11)
    for counts in ([1, 31, 32, 33, 224, 255, 0, 256], [33, 31, 224, 32]):
        check(dmc, port, strip_image(taps_per_tile(rs, H, W, R, counts), H, W, R, 6), 5, 10, "counts %s" % counts)


@pytest.mark.parametrize("path", sorted(SHAPES_R5))
def test_one_strip_against_its_tile(dmc, port, path):
    """a strip of full-range noise in a constant tile, and a plateau that leaves exactly one flat strip in a noisy tile"""
    H, W = SHAPES_R5[path]
    r, th = 5, 10
    R, E = rows_per_thread(r, H, W), words_each_side(r)
    rs = np.random.RandomState(5)
    img = np.full((H, W), C0, np.uint8)
    for ty in range(0, H // (4 * R)):
        y, x = 4 * R * ty + R * (ty % 4), 128 * (ty % (W // 128)) + 2 * (7 * ty % 64)
        img[y:y + R, x:x + 2] = rs.randint(0, 256, size=(R, 2))
    check(dmc, port, img, r, th, "noisy strip")
    img = rs.randint(0, 256, size=(H, W)).astype(np.uint8)
    for ty in range(1, H // (4 * R) - 1):
        y, x = 4 * R * ty + R * (ty % 4), 128 * (ty % (W // 128)) + 2 * (7 * ty % 48) + 16
        img[y - r:y + R + r, x - E:x + 2 + E] = C0 + rs.randint(-th // 2, th // 2 + 1, size=(R + 2 * r, 2 + 2 * E))
    check(dmc, port, img, r, th, "flat strip")


@pytest.mark.parametrize("r", [1, 2, 5, 7, 10])
@pytest.mark.parametrize("path", ["main", "few"])
def test_strip_threshold_boundary(dmc, port, r, path):
    """one pixel at c0 + th (the strip passes: max(F) - min(centres) == th) and c0 + th + 1 (it does not), and the same
    below c0, at the corners of a strip's footprint and on the rim of its disc"""
    H, W = (640, 1024) if path == "main" else (48, 256)
    R, E, th = rows_per_thread(r, H, W), words_each_side(r), 10
    spots = [(-r, -E), (R - 1 + r, 1 + E), (-r, 1 + E), (R - 1 + r, -E), (0, -r), (R - 1, 1 + r), (-r, 0), (R - 1 + r, 1)]
    for delta in (th, th + 1, -th, -(th + 1)):
        img = np.full((H, W), C0, np.uint8)
        for i, (dy, dx) in enumerate(spots * 4):
            y0 = 4 * R * (1 + i % ((H - 2 * r) // (4 * R) - 2)) + R * (i % 4)
            x0 = 128 * (i % (W // 128)) + 2 * (9 * i % 64)
            if 0 <= y0 + dy < H and 0 <= x0 + dx < W:
                img[y0 + dy, x0 + dx] = C0 + delta
        check(dmc, port, img, r, th, "strip boundary %+d" % delta)


@pytest.mark.parametrize("r", range(1, 11))
def test_every_radius_both_sides_of_flush(dmc, port, r):
    """the half accumulator alone (ntaps*th <= 2048) and the FLUSH variant above it, on the main and the few-tiles path;
    partial tiles on the right and bottom edges and odd widths"""
    rs = np.random.RandomState(40 + r)
    for H, W in ((601, 2085), (75, 389)):
        R = rows_per_thread(r, H, W)
        for th in sorted({1, 2048 // ntaps(r), 2048 // ntaps(r) + 1} & set(range(1, 2048 // (2 * r + 1) + 1))):
            a = th // 2 + 1
            if a > 120:                      # every tap passes: no tap strip can be built
                img = strip_image(np.zeros(((H + R - 1) // R, (W + 1) // 2), bool), H, W, R, 0)
            else:
                img = strip_image(taps_per_tile(rs, H, W, R, [1, 31, 33, 224, 64]), H, W, R, a)
            check(dmc, port, img, r, th, "strips R=%d" % R)


@pytest.mark.parametrize("offs", [(0, 0), (1, 0), (0, 1), (3, 5)])
@pytest.mark.parametrize("shape", [(640, 1024), (61, 131), (333, 1919)])
def test_unaligned_device_pointers(dmc, port, offs, shape):
    """device images at odd byte offsets (no 16-byte staging loads, no 2-byte stores) and odd widths"""
    import torch
    from depthmapcompression_b200.capi import DmcImage, lib
    H, W = shape
    rs = np.random.RandomState(H + W + offs[0])
    so, do = offs
    d_in = torch.zeros(H * W + 64, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(H * W + 64, dtype=torch.uint8, device="cuda")
    ctx = dmc.default_context(0)
    for r in (2, 5):
        img = strip_image(taps_per_tile(rs, H, W, rows_per_thread(r, H, W), [31, 33, 1]), H, W, rows_per_thread(r, H, W), 6)
        d_in[so:so + H * W] = torch.from_numpy(img.reshape(-1)).cuda()
        torch.cuda.synchronize()            # the copy runs on torch's stream, the filter on the context's own
        s8 = DmcImage(d_in.data_ptr() + so, H, W, 0, W, 1)
        o8 = DmcImage(d_out.data_ptr() + do, H, W, 0, W, 1)
        ctx.check(lib.dmc_bwrf(ctx.h, C.byref(s8), C.byref(o8), 2 * r + 1, 2 * r + 1, 10.0, 0, 1))
        torch.cuda.synchronize()
        got = d_out[do:do + H * W].cpu().numpy().reshape(H, W)
        assert np.array_equal(got, port.bwrf(img, 2 * r + 1, 2 * r + 1, 10)), (r, offs, shape)
