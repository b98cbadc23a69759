"""boundaryReconstructionFilter on frame batches (dmc_brf_batch, boundaryReconstructionFilterBatch): one launch covers many
frames, with the frame taken from the grid's z.  Every frame of a batch must equal dmc_boundary_reconstruction of that frame
alone and the oracle port, bit for bit, for the five depths, from host memory (streamed in chunks) and from device memory, in
place and through scratch; frames of one launch may take different per-CTA paths (flat tile, ranked tile, > 256 values,
float NaN / -0); argument errors write nothing."""
import ctypes as C
import os

import numpy as np
import pytest

from _util import assert_bits_equal, load_png

pytestmark = pytest.mark.gpu

DTYPES = [np.uint8, np.uint16, np.int16, np.float32, np.float64]
KS = (13, 13)


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


@pytest.fixture(scope="module")
def port():
    from oracle.oracle_py import Port
    p = Port()
    p.set_num_threads(0)
    return p


def frames_of(rs, n, H, W, dt):
    """smooth ramps with a few values, block noise and a flat frame, cycling"""
    out = []
    for i in range(n):
        yy, xx = np.mgrid[0:H, 0:W]
        kind = i % 3
        if kind == 0:
            a = (xx // 3 + yy // 5 + i) % 200 + rs.randint(0, 3, size=(H, W))
        elif kind == 1:
            a = np.kron(rs.randint(0, 200, ((H + 3) // 4, (W + 3) // 4)), np.ones((4, 4), np.int64))[:H, :W]
        else:
            a = np.full((H, W), 17 + i % 50)
        out.append(a)
    a = np.stack(out)
    if dt == np.uint8:
        return a.astype(dt)
    if dt in (np.uint16, np.int16):
        return (a * 37 - (3000 if dt == np.int16 else -1000)).astype(dt)
    return (a * 0.37 - 11.0).astype(dt)


def single(dmc, a, ks=KS, p=(1.0, 1.0, 1.0)):
    return np.stack([dmc.boundaryReconstructionFilter(x, None, ks, *p) for x in a])


@pytest.mark.parametrize("dt", DTYPES)
def test_batch_equals_single_and_port(dmc, port, dt):
    rs = np.random.RandomState(11)
    for (H, W) in [(3, 3), (17, 23), (61, 83)]:
        for n in (1, 3, 70):
            a = frames_of(rs, n, H, W, dt)
            got = dmc.boundaryReconstructionFilterBatch(a, None, KS, 1.0, 1.0, 1.0)
            assert got.dtype == a.dtype and got.shape == a.shape
            assert_bits_equal(got, single(dmc, a), "batch vs single %s %dx%d n=%d" % (np.dtype(dt).name, H, W, n))
            for i in sorted({0, n // 2, n - 1}):
                assert_bits_equal(got[i], port.brf(a[i], KS[0], KS[1], 1.0, 1.0, 1.0), "batch vs port %s %dx%d n=%d i=%d" % (np.dtype(dt).name, H, W, n, i))
    # a non-square window and other weights
    a = frames_of(rs, 5, 40, 70, dt)
    assert_bits_equal(dmc.boundaryReconstructionFilterBatch(a, None, (5, 9), 1.0, 0.5, 2.0), single(dmc, a, (5, 9), (1.0, 0.5, 2.0)), "5x9")


def test_batch_1080p_equals_single_and_port(dmc, port):
    img = load_png("kinect_desk_q50.png")
    big = np.ascontiguousarray(np.tile(img, (3, 3))[:1080, :1920])
    a = np.stack([big, np.roll(big, 37, axis=1)])
    got = dmc.boundaryReconstructionFilterBatch(a, None, KS, 1.0, 1.0, 1.0)
    assert_bits_equal(got, single(dmc, a), "1080p batch vs single")
    assert_bits_equal(got[1], port.brf(a[1], 13, 13, 1.0, 1.0, 1.0), "1080p batch vs port")


def test_mixed_paths_in_one_launch(dmc, port):
    """flat, ranked, > 256 distinct values and a float frame holding NaN / -0 next to a plain one, in one batch"""
    rs = np.random.RandomState(12)
    H, W = 48, 80
    for dt in (np.uint16, np.float32, np.float64):
        flat = np.full((H, W), 7, dt)
        ranked = frames_of(rs, 1, H, W, dt)[0]
        many = rs.randint(0, 30000, (H, W)).astype(dt)
        special = ranked.copy()
        if dt != np.uint16:
            special[5, 7] = -0.0; special[30, 60] = np.nan; special[31, 61] = np.inf
        a = np.stack([flat, ranked, many, special, ranked.copy()])
        got = dmc.boundaryReconstructionFilterBatch(a, None, (7, 7), 1.0, 1.0, 1.0)
        for i in range(len(a)):
            assert_bits_equal(got[i], port.brf(a[i], 7, 7, 1.0, 1.0, 1.0), "mixed %s frame %d" % (np.dtype(dt).name, i))
        assert_bits_equal(got, single(dmc, a, (7, 7)), "mixed %s vs single" % np.dtype(dt).name)


def test_host_chunks_device_in_place_and_overlap(dmc, monkeypatch):
    import torch
    rs = np.random.RandomState(13)
    for dt, tdt in ((np.uint8, torch.uint8), (np.int16, torch.int16), (np.float32, torch.float32)):
        a = frames_of(rs, 70, 61, 83, dt)
        want = single(dmc, a)
        monkeypatch.setenv("DMC_CHUNK_MB", "1")                  # 61 x 83 frames: several chunks per slot
        assert_bits_equal(dmc.boundaryReconstructionFilterBatch(a, None, KS, 1.0, 1.0, 1.0), want, "host chunks")
        b = a.copy()
        assert dmc.boundaryReconstructionFilterBatch(b, b, KS, 1.0, 1.0, 1.0) is b
        assert_bits_equal(b, want, "host in place")
        buf = np.concatenate([a, a[:1]])                          # dst = src shifted by one frame, both views of one array
        dmc.boundaryReconstructionFilterBatch(buf[:-1], buf[1:], KS, 1.0, 1.0, 1.0)
        assert_bits_equal(buf[1:], want, "host overlapping")
        monkeypatch.delenv("DMC_CHUNK_MB")
        monkeypatch.setenv("DMC_GROUP_MB", "1")                   # device groups
        ctx = dmc.default_context()
        d = torch.from_numpy(a).cuda(); o = torch.empty_like(d); torch.cuda.synchronize()
        dev = (d.data_ptr(), 70, 61, 83, dt)
        dmc.boundaryReconstructionFilterBatch(dev, o.data_ptr(), KS, 1.0, 1.0, 1.0); ctx.synchronize()
        assert_bits_equal(o.cpu().numpy(), want, "device")
        dmc.boundaryReconstructionFilterBatch(dev, d.data_ptr(), KS, 1.0, 1.0, 1.0); ctx.synchronize()
        assert_bits_equal(d.cpu().numpy(), want, "device in place")
        e = torch.from_numpy(np.concatenate([a, a[:1]])).cuda(); torch.cuda.synchronize()
        fb = a[0].nbytes
        dmc.boundaryReconstructionFilterBatch((e.data_ptr(), 70, 61, 83, dt), e.data_ptr() + fb, KS, 1.0, 1.0, 1.0); ctx.synchronize()
        assert_bits_equal(e.cpu().numpy()[1:], want, "device overlapping")
        monkeypatch.delenv("DMC_GROUP_MB")


def test_device_groups_8u_in_place_and_overlapping(dmc, monkeypatch):
    """several device groups of 8-bit frames (the depth the sweeps filter): into a separate dst, in place, and with dst a frame
    above or below src, where the groups go through group-sized scratch in memmove order"""
    import torch
    rs = np.random.RandomState(15)
    n, H, W = 23, 480, 640                                       # 300 KB frames: 1 MB groups of 3 frames, 8 groups
    a = frames_of(rs, n, H, W, np.uint8)
    want = single(dmc, a)
    ctx = dmc.default_context()
    fb = a[0].nbytes
    monkeypatch.setenv("DMC_GROUP_MB", "1")
    d = torch.from_numpy(a).cuda(); o = torch.empty_like(d); torch.cuda.synchronize()
    dmc.boundaryReconstructionFilterBatch((d.data_ptr(), n, H, W), o.data_ptr(), KS, 1.0, 1.0, 1.0); ctx.synchronize()
    assert_bits_equal(o.cpu().numpy(), want, "device groups")
    dmc.boundaryReconstructionFilterBatch((d.data_ptr(), n, H, W), d.data_ptr(), KS, 1.0, 1.0, 1.0); ctx.synchronize()
    assert_bits_equal(d.cpu().numpy(), want, "device groups in place")
    for shift in (1, -1, 2):                                     # dst = src + shift frames (2: across a group boundary)
        lo = max(0, -shift)
        e = torch.zeros((n + abs(shift),) + a.shape[1:], dtype=torch.uint8, device="cuda")
        e[lo:lo + n] = torch.from_numpy(a).cuda(); torch.cuda.synchronize()
        sp = e.data_ptr() + lo * fb
        dmc.boundaryReconstructionFilterBatch((sp, n, H, W), sp + shift * fb, KS, 1.0, 1.0, 1.0); ctx.synchronize()
        assert_bits_equal(e.cpu().numpy()[lo + shift:lo + shift + n], want, "device groups, dst = src %+d frames" % shift)
    # the host path with dst a frame below src, too
    monkeypatch.setenv("DMC_CHUNK_MB", "1")
    buf = np.concatenate([a[:1], a])
    dmc.boundaryReconstructionFilterBatch(buf[1:], buf[:-1], KS, 1.0, 1.0, 1.0)
    assert_bits_equal(buf[:-1], want, "host, dst = src - 1 frame")


def test_argument_rules(dmc):
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    a = frames_of(np.random.RandomState(14), 3, 17, 23, np.uint8)

    def call(depth=capi.CV_8U, b=None, n=3, rows=17, cols=23, mem=capi.MEM_HOST, src=True, dst=True):
        out = np.full(a.shape, 0xA5, np.uint8)
        bp = dmc.brf_params(KS) if b is None else b
        rc = capi.lib.dmc_brf_batch(ctx.h, C.c_void_p(a.ctypes.data if src else None), C.c_void_p(out.ctypes.data if dst else None), n, rows, cols, depth,
                                    C.byref(bp) if bp is not False else None, mem)
        return rc, bool(np.all(out == 0xA5))

    assert call() == (capi.DMC_OK, False)
    assert call(b=False) == (capi.DMC_ERR_ARG, True)
    for ks in ((0, 13), (13, 0), (-1, 3), (22, 13), (13, 22), (23, 23)):
        assert call(b=dmc.brf_params(ks)) == (capi.DMC_ERR_ARG, True), ks
    assert call(b=dmc.brf_params((21, 1))) == (capi.DMC_OK, False)
    for depth in (1, 4, 7, -1, 8):
        assert call(depth=depth) == (capi.DMC_ERR_TYPE, True), depth
    for mem in (2, -1):
        assert call(mem=mem) == (capi.DMC_ERR_ARG, True), mem
    for kw in (dict(n=-1), dict(rows=0), dict(cols=0), dict(rows=-5), dict(src=False), dict(dst=False)):
        assert call(**kw) == (capi.DMC_ERR_SIZE, True), kw
    assert call(n=0) == (capi.DMC_OK, True)
    assert capi.lib.dmc_brf_batch(None, None, None, 1, 1, 1, 0, None, 0) == capi.DMC_ERR_ARG
    with pytest.raises(dmc.DmcError):
        dmc.boundaryReconstructionFilterBatch(a.astype(np.int32), None, KS)
    with pytest.raises(dmc.DmcError):
        dmc.boundaryReconstructionFilterBatch((0, 3, 17, 23), None, KS)
