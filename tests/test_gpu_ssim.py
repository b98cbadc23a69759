"""The structural similarity kernel (dmc_ssim_batch, frameSSIM) against the float64 reference of test_ssim_reference.py, to
1e-10 absolute per frame: gray and 8UC3 frames from 11 x 11 to 1080p, noise, flat frames, 0 against 255, the golden Kinect
frames and degrade_blocks of synth_disp; batches of 1, 3 and 70 frames in host and device memory, misaligned pointers and
a == b.  Every frame's result must be the same bits alone, inside a batch and on a second run; bad arguments return their
error and write nothing."""
import ctypes as C

import numpy as np
import pytest

from _util import load_png
from test_ssim_reference import ssim_ref, ssim_ref_batch

pytestmark = pytest.mark.gpu
TOL = 1e-10
SENTINEL = -12345.0


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def pairs(H, W, cn, n, seed):
    """n frame pairs of every kind: noise against noise, flat, 0 against 255, a blocky degradation of synth_disp"""
    from oracle.oracle_py import synth_disp, degrade_blocks
    rs = np.random.RandomState(seed)
    shape = (H, W) if cn == 1 else (H, W, cn)
    a, b = [], []
    for i in range(n):
        kind = i % 4
        if kind == 0:
            x = rs.randint(0, 256, shape); y = np.clip(x + rs.randint(-60, 61, shape), 0, 255)
        elif kind == 1:
            x = np.full(shape, rs.randint(0, 256)); y = np.full(shape, rs.randint(0, 256))
        elif kind == 2:
            x = np.zeros(shape); y = np.full(shape, 255)
        else:
            planes = [synth_disp(H, W, seed + i + c) for c in range(cn)]
            x = np.stack(planes, -1) if cn == 3 else planes[0]
            y = np.stack([degrade_blocks(p, seed + 7 * i + c) for c, p in enumerate(planes)], -1) if cn == 3 else degrade_blocks(planes[0], seed + i)
        a.append(x); b.append(y)
    return np.stack(a).astype(np.uint8), np.stack(b).astype(np.uint8)


@pytest.mark.parametrize("cn", [1, 3])
@pytest.mark.parametrize("H,W", [(11, 11), (11, 200), (200, 11), (12, 13), (61, 83), (480, 640)])
def test_sizes_equal_reference(dmc, H, W, cn):
    a, b = pairs(H, W, cn, 4, H * 5 + W)
    got = dmc.frameSSIM(a, b)
    want = ssim_ref_batch(a, b)
    assert np.all(np.abs(got - want) <= TOL), (got, want)
    assert np.all(np.abs(dmc.frameSSIM(a, a) - 1.0) <= 1e-12)


@pytest.mark.parametrize("cn", [1, 3])
def test_1080p_equals_reference(dmc, cn):
    a, b = pairs(1080, 1920, cn, 4, 11 + cn)
    got = dmc.frameSSIM(a, b)
    assert np.all(np.abs(got - ssim_ref_batch(a, b)) <= TOL)


def test_golden_kinect_frames(dmc):
    names = ("kinect_meeting_q50.png", "kinect_meeting_q80.png", "kinect_desk_q50.png", "kinect_desk_q80.png", "x264_depth_y.png")
    imgs = [load_png(n) for n in names]
    meeting, desk = np.stack(imgs[:2]), np.stack(imgs[2:4])
    for x, y in ((meeting[:1], meeting[1:]), (desk[:1], desk[1:])):
        assert abs(dmc.frameSSIM(x, y)[0] - ssim_ref(x[0], y[0])) <= TOL
    from oracle.oracle_py import degrade_blocks
    z = imgs[4]
    zb = degrade_blocks(z, 3)
    assert abs(dmc.frameSSIM(z, zb)[0] - ssim_ref(z, zb)) <= TOL
    bgr = np.stack([meeting[0], 255 - meeting[1], meeting[0] // 2], -1)
    bgr2 = np.stack([meeting[1], 255 - meeting[0], meeting[1] // 2], -1)
    assert abs(dmc.frameSSIM(bgr, bgr2)[0] - ssim_ref(bgr, bgr2)) <= TOL


@pytest.mark.parametrize("cn", [1, 3])
def test_batches_host_device_misaligned_and_deterministic(dmc, cn):
    import torch
    H, W = 37, 53
    a, b = pairs(H, W, cn, 70, 5 + cn)
    want = ssim_ref_batch(a, b)
    alone = np.array([dmc.frameSSIM(a[i:i + 1], b[i:i + 1])[0] for i in range(70)])
    assert np.all(np.abs(alone - want) <= TOL)
    fb = a[0].size
    for n in (1, 3, 70):
        host = dmc.frameSSIM(a[:n], b[:n])
        assert np.array_equal(host.view(np.uint64), alone[:n].view(np.uint64)), n
        assert np.array_equal(dmc.frameSSIM(a[:n], b[:n]).view(np.uint64), host.view(np.uint64)), n      # a second run
        for off_a, off_b in ((0, 0), (1, 3), (7, 0)):
            da = torch.zeros(n * fb + 16, dtype=torch.uint8, device="cuda")
            db = torch.zeros(n * fb + 16, dtype=torch.uint8, device="cuda")
            da[off_a:off_a + n * fb] = torch.from_numpy(a[:n].reshape(-1)).cuda()
            db[off_b:off_b + n * fb] = torch.from_numpy(b[:n].reshape(-1)).cuda()
            torch.cuda.synchronize()
            dev = dmc.frameSSIM((da.data_ptr() + off_a, n, H, W), (db.data_ptr() + off_b, n, H, W), channels=cn)
            assert np.array_equal(dev.view(np.uint64), alone[:n].view(np.uint64)), (n, off_a, off_b)
            same = dmc.frameSSIM((da.data_ptr() + off_a, n, H, W), (da.data_ptr() + off_a, n, H, W), channels=cn)
            assert np.all(np.abs(same - 1.0) <= 1e-12)
    # a == b from host memory (one staging copy) and misaligned host frames
    assert np.array_equal(dmc.frameSSIM(a[:3], a[:3]).view(np.uint64), np.array([dmc.frameSSIM(a[i], a[i])[0] for i in range(3)]).view(np.uint64))
    buf = np.zeros(3 * fb + 1, np.uint8)
    mis = buf[1:].reshape(a[:3].shape)
    mis[...] = a[:3]
    assert np.array_equal(dmc.frameSSIM(mis, b[:3]).view(np.uint64), alone[:3].view(np.uint64))


def test_argument_rules(dmc):
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    a = np.random.RandomState(1).randint(0, 256, (2, 20, 20, 3)).astype(np.uint8)
    DP = C.POINTER(C.c_double)

    def call(pa=a.ctypes.data, pb=a.ctypes.data, n=2, rows=20, cols=20, cn=3, mem=capi.MEM_HOST, out=True):
        o = np.full(2, SENTINEL)
        rc = capi.lib.dmc_ssim_batch(ctx.h, C.c_void_p(pa), C.c_void_p(pb), n, rows, cols, cn, mem, o.ctypes.data_as(DP) if out else None)
        return rc, bool(np.all(o == SENTINEL))

    assert call()[0] == capi.DMC_OK
    assert call(rows=10) == (capi.DMC_ERR_SIZE, True)
    assert call(cols=10) == (capi.DMC_ERR_SIZE, True)
    assert call(rows=10, cols=10, cn=1) == (capi.DMC_ERR_SIZE, True)
    for cn in (0, 2, 4):
        assert call(cn=cn) == (capi.DMC_ERR_ARG, True), cn
    assert call(pa=None) == (capi.DMC_ERR_SIZE, True)
    assert call(pb=None) == (capi.DMC_ERR_SIZE, True)
    assert call(out=False)[0] == capi.DMC_ERR_SIZE
    assert call(n=-1) == (capi.DMC_ERR_SIZE, True)
    for mem in (2, -1):
        assert call(mem=mem) == (capi.DMC_ERR_ARG, True), mem
    assert call(n=0) == (capi.DMC_OK, True)
    with pytest.raises(dmc.DmcError):
        dmc.frameSSIM(a[:, :10, :10], a[:, :10, :10])
    with pytest.raises(dmc.DmcError):
        dmc.frameSSIM(a, a[..., 0])
