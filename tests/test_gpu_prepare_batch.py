"""pointcloudTest's preparation on frame batches (dmc_prepare_disp_batch, prepareDisparityBatch): every output frame must
equal, bit for bit, the library's single-image calls on that frame (depth16U2disp8U -> fillOcclusion(0, FILL_DISPARITY),
and for two passes transpose -> fillOcclusion -> transpose) and the port's serial restatement, over sizes, batch sizes,
groups, host and device memory, and rows built to hit every branch of the fill."""
import ctypes as C

import numpy as np
import pytest

from _util import canon_crc, load_golden, load_png

pytestmark = pytest.mark.gpu

FB, AMP = 75.0 * 575.0, 2.6
FILL_DISPARITY = 0


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def adversarial(H, W, seed):
    """16U frame whose rows and columns carry the fill's edge cases.  Depth 0 converts to disparity 0 (invalid); depths of
    32768 and more convert to 0 in the converter's SIMD body and to a small value in its scalar tail."""
    rs = np.random.RandomState(seed)
    d = rs.randint(300, 20000, (H, W)).astype(np.uint16)
    half = W // 2                                     # (int)(cols * 0.5): a run of half fills, half + 1 blanks the row
    for y in range(H):
        k = (y + seed) % 8
        if k == 0: d[y, 1:1 + half] = 0
        elif k == 1: a = max(1, W // 3 - 1); d[y, a:a + half + 1] = 0
        elif k == 2: d[y] = 0
        elif k == 3: d[y, W // 2:] = 0; d[(y + 1) % H, 0] = 0          # a run up to the row end, the next row's first pixel invalid
        elif k == 4: d[y, W // 2:] = 0; d[(y + 1) % H, 0] = 1000       # ... and valid
        elif k == 5: d[y] = rs.randint(32768, 65536, W)
        elif k == 6: d[y, rs.rand(W) < 0.4] = 0
    hv = H // 2
    for x in range(0, W, 5):                          # the same cases down columns, for the second pass
        k = (x // 5 + seed) % 4
        if k == 0: d[1:1 + hv, x] = 0
        elif k == 1: d[max(1, H // 3 - 1):max(1, H // 3 - 1) + hv + 1, x] = 0
        elif k == 2: d[:, x] = 0
    return d


def batch(H, W, n, seed):
    return np.stack([adversarial(H, W, seed + 13 * i) for i in range(n)])


def single_calls(dmc, frame, passes, fb=FB, a=AMP, b=0.0):
    """The library's single-image calls, as simpleTest (one pass) and pointcloudTest (two) make them."""
    x = dmc.depth16U2disp8U(frame, None, fb, a, b)
    dmc.fillOcclusion(x, 0, dmc.FILL_DISPARITY)
    if passes == 2:
        x = dmc.transpose(dmc.fillOcclusion(dmc.transpose(x), 0, dmc.FILL_DISPARITY))
    return x


def port_fill(port, x):
    """The port's serial fill.  Past the last row its read is undefined (the single-image kernel reads `invalid`); the
    closed form (tests/test_prepare_closed_form.py) shows the read never matters, so a guard row stands in for it."""
    g = np.vstack([x, np.full((1, x.shape[1]), 7, np.uint8)])
    return port.fill_occlusion(g, 0, FILL_DISPARITY)[:-1]


def port_prepare(port, frame, passes, fb=FB, a=AMP, b=0.0):
    x = port_fill(port, port.depth16u2disp8u(frame, fb, a, b))
    if passes == 2:
        x = np.ascontiguousarray(port_fill(port, np.ascontiguousarray(x.T)).T)
    return x


def device_prepare(dmc, frames, passes, fb=FB, a=AMP, b=0.0):
    import torch
    n, H, W = frames.shape
    src = torch.from_numpy(frames.view(np.int16)).cuda()
    dst = torch.full((n, H, W), 0xA5, dtype=torch.uint8, device="cuda")
    dmc.prepareDisparityBatch((src.data_ptr(), n, H, W), fb, a, b, passes=passes, dst=dst.data_ptr())
    dmc.default_context().synchronize()
    return dst.cpu().numpy()


def check(dmc, port, frames, passes, with_port=True, **kw):
    host = dmc.prepareDisparityBatch(frames, kw.get("fb", FB), kw.get("a", AMP), kw.get("b", 0.0), passes=passes)
    dev = device_prepare(dmc, frames, passes, **kw)
    assert host.shape == frames.shape and host.dtype == np.uint8
    assert np.array_equal(host, dev), (frames.shape, passes)
    for i, f in enumerate(frames):
        assert np.array_equal(host[i], single_calls(dmc, f, passes, **kw)), (frames.shape, passes, i)
        if with_port:
            assert np.array_equal(host[i], port_prepare(port, f, passes, **kw)), (frames.shape, passes, i)
    return host


@pytest.mark.parametrize("H,W", [(2, 2), (1, 5), (3, 17), (17, 3), (61, 83), (480, 640), (1080, 1920)])
def test_batch_equals_single_calls_and_port(dmc, port, H, W):
    for passes in (1, 2):
        if passes == 2 and H < 2:
            continue
        for n in (1, 3):
            frames = batch(H, W, n, H + W + n)
            check(dmc, port, frames, passes, with_port=H * W <= 480 * 640 or n == 1)


def test_converter_quirks_per_frame(dmc, port):
    """The SIMD body / scalar tail split is per frame: area % 16 != 0, values >= 32768 in both parts, b != 0."""
    rs = np.random.RandomState(5)
    for H, W in ((7, 9), (5, 13), (31, 33)):
        assert (H * W) % 16 != 0
        frames = rs.randint(0, 65536, (4, H, W)).astype(np.uint16)
        frames[:, :, ::3] = rs.randint(32768, 65536, (4, H, (W + 2) // 3))
        for passes in (1, 2):
            check(dmc, port, frames, passes)
            check(dmc, port, frames, passes, fb=1200.0, a=1.0, b=2.5)


def test_70_frames_in_groups_and_chunks(dmc, port, monkeypatch):
    frames = batch(61, 83, 70, 1)
    want = {p: np.stack([single_calls(dmc, f, p) for f in frames]) for p in (1, 2)}
    for mb in (None, "1"):                           # 1 MiB: several device groups and host chunks
        if mb:
            monkeypatch.setenv("DMC_GROUP_MB", mb); monkeypatch.setenv("DMC_CHUNK_MB", mb)
        for p in (1, 2):
            assert np.array_equal(dmc.prepareDisparityBatch(frames, FB, AMP, passes=p), want[p]), (mb, p)
            assert np.array_equal(device_prepare(dmc, frames, p), want[p]), (mb, p)
    big = batch(480, 640, 70, 2)
    monkeypatch.setenv("DMC_GROUP_MB", "16"); monkeypatch.setenv("DMC_CHUNK_MB", "8")
    got = device_prepare(dmc, big, 2)
    assert np.array_equal(dmc.prepareDisparityBatch(big, FB, AMP, passes=2), got)
    for i in (0, 1, 33, 68, 69):
        assert np.array_equal(got[i], single_calls(dmc, big[i], 2)), i
        assert np.array_equal(got[i], port_prepare(port, big[i], 2)), i


def test_kinect_crop_reproduces_golden_crcs(dmc):
    name = "kinect_meeting_depth16_crop.png"
    d16 = load_png(name)
    g = load_golden()["inputs"][name]["golden"]
    H, W = d16.shape
    others = batch(H, W, 4, 9)
    for passes, key in ((1, "fill_disparity_1pass"), (2, "fill_disparity_2pass")):
        assert canon_crc(dmc.prepareDisparityBatch(d16, FB, AMP, passes=passes)) == g[key]
        for pos in (0, 2, 4):
            frames = np.concatenate([others[:pos], d16[None], others[pos:]])
            for out in (dmc.prepareDisparityBatch(frames, FB, AMP, passes=passes), device_prepare(dmc, frames, passes)):
                assert canon_crc(out[pos]) == g[key], (passes, pos)


def test_argument_rules(dmc):
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    src = batch(8, 10, 2, 3)
    dst = np.full(src.shape, 0xA5, np.uint8)

    def call(s=src.ctypes.data, d=dst.ctypes.data, n=2, rows=8, cols=10, passes=2, mem=capi.MEM_HOST):
        return capi.lib.dmc_prepare_disp_batch(ctx.h, C.c_void_p(s), C.c_void_p(d), n, rows, cols, FB, AMP, 0.0, passes, mem)

    for passes in (0, 3, -1):
        assert call(passes=passes) == capi.DMC_ERR_ARG and np.all(dst == 0xA5), passes
    for mem in (2, -1):
        assert call(mem=mem) == capi.DMC_ERR_ARG and np.all(dst == 0xA5), mem
    assert call(cols=1) == capi.DMC_ERR_SIZE and np.all(dst == 0xA5)
    assert call(cols=1, passes=1) == capi.DMC_ERR_SIZE and np.all(dst == 0xA5)
    assert call(rows=1, passes=2) == capi.DMC_ERR_SIZE and np.all(dst == 0xA5)
    for bad in (dict(n=-1), dict(rows=0), dict(cols=-2), dict(d=0)):
        assert call(**bad) == capi.DMC_ERR_SIZE and np.all(dst == 0xA5), bad
    assert call(n=0) == capi.DMC_OK and np.all(dst == 0xA5)
    # depth16 and disp8 overlapping, in host and device memory
    buf = np.full(src.nbytes + dst.nbytes, 0x5A, np.uint8)
    buf[:src.nbytes] = src.view(np.uint8).ravel()
    keep = buf.copy()
    for off in (0, 7, src.nbytes - 1):
        assert call(s=buf.ctypes.data, d=buf.ctypes.data + off) == capi.DMC_ERR_ARG and np.array_equal(buf, keep), off
    import torch
    t = torch.from_numpy(buf).cuda()
    for off in (0, 100):
        assert call(s=t.data_ptr(), d=t.data_ptr() + off, mem=capi.MEM_DEVICE) == capi.DMC_ERR_ARG, off
    torch.cuda.synchronize()
    assert np.array_equal(t.cpu().numpy(), keep)
    with pytest.raises(dmc.DmcError):
        dmc.prepareDisparityBatch(src, FB, AMP, passes=3)
    with pytest.raises(dmc.DmcError):
        dmc.prepareDisparityBatch(src.astype(np.float32), FB, AMP)
    # rows < 2 is fine for one pass (simpleTest's call on a one-row image)
    one = batch(1, 5, 2, 4)
    assert np.array_equal(dmc.prepareDisparityBatch(one, FB, AMP, passes=1)[1], single_calls(dmc, one[1], 1))
