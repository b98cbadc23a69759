"""The distortion metric and the JPEG rate-distortion sweep on the GPU: dmc_sse_gray_batch must equal the int64 sum of
squared differences numpy computes, and dmc_jpeg_rd_sweep must report for every frame and quality the size of
cv2.imencode's stream, the SSE of cv2.imdecode's frame and the SSE of the port's PostFilterSet()(decoded, 2,1,3,5,10),
in both Huffman modes, from host and device sources, and equal the composition of the public GPU calls."""
import ctypes as C

import numpy as np
import pytest

from _util import load_png

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu

SSE_SIZES = [(1, 1), (1, 5), (5, 1), (7, 13), (83, 131), (100, 1023), (480, 640), (1080, 1920), (3, 10000)]
QUALITIES = (0, 1, 5, 50, 80, 95, 100)
CHAIN = (2, 1, 3, 5, 10)
U64 = C.POINTER(C.c_uint64)


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def np_sse(a, b):
    a = a.reshape(-1, a.shape[-2], a.shape[-1]); b = b.reshape(a.shape)
    return np.array([int(((x.astype(np.int64) - y) ** 2).sum()) for x, y in zip(a, b)], np.uint64)


def kinds(H, W, seed=3):
    from oracle.oracle_py import synth_disp, degrade_blocks
    rs = np.random.RandomState(seed)
    out = [rs.randint(0, 256, (H, W)).astype(np.uint8), np.zeros((H, W), np.uint8), np.full((H, W), 255, np.uint8)]
    if H > 16 and W > 16:
        out.append(degrade_blocks(synth_disp(H, W, seed), seed))
    return np.stack(out)


@pytest.mark.parametrize("shape", SSE_SIZES)
def test_sse_matches_numpy_host_and_device(dmc, shape):
    import torch
    rs = np.random.RandomState(shape[0] * 7 + shape[1])
    for n in (1, 3, 70):
        a = rs.randint(0, 256, (n,) + shape).astype(np.uint8)
        b = np.clip(a.astype(np.int16) + rs.randint(-40, 41, a.shape), 0, 255).astype(np.uint8)
        b[n // 2] = rs.randint(0, 256, shape)            # one frame far from its reference
        want = np_sse(a, b)
        assert np.array_equal(dmc.frameSSE(a, b), want), (shape, n, "host")
        da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        got = dmc.frameSSE((da.data_ptr(), n, *shape), (db.data_ptr(), n, *shape))
        assert np.array_equal(got, want), (shape, n, "device")
        # b one byte off a's 16-byte alignment: the byte-wise path
        buf = torch.zeros(a.size + 16, dtype=torch.uint8, device="cuda")
        buf[1:1 + a.size] = db.reshape(-1)
        torch.cuda.synchronize()                         # (the library's stream does not wait for torch's)
        got = dmc.frameSSE((da.data_ptr(), n, *shape), (buf.data_ptr() + 1, n, *shape))
        assert np.array_equal(got, want), (shape, n, "device, misaligned")


def test_sse_special_frames_and_aliasing(dmc):
    import torch
    H, W = 1080, 1920
    zero, full = np.zeros((2, H, W), np.uint8), np.full((2, H, W), 255, np.uint8)
    assert list(dmc.frameSSE(zero, full)) == [255 * 255 * H * W] * 2
    d0, d1 = torch.from_numpy(zero).cuda(), torch.from_numpy(full).cuda()
    assert list(dmc.frameSSE((d0.data_ptr(), 2, H, W), (d1.data_ptr(), 2, H, W))) == [255 * 255 * 2073600] * 2
    rs = np.random.RandomState(5)
    x = rs.randint(0, 256, (3, 83, 131)).astype(np.uint8)
    assert list(dmc.frameSSE(x, x.copy())) == [0, 0, 0]
    assert list(dmc.frameSSE(x, x)) == [0, 0, 0]                    # the same host pointer
    dx = torch.from_numpy(x).cuda()
    assert list(dmc.frameSSE((dx.data_ptr(), 3, 83, 131), (dx.data_ptr(), 3, 83, 131))) == [0, 0, 0]
    assert dmc.frameSSE(np.zeros((0, 4, 4), np.uint8), np.zeros((0, 4, 4), np.uint8)).shape == (0,)


def rd_frames():
    golden = np.stack([load_png(n) for n in ("kinect_meeting_q50.png", "kinect_desk_q50.png", "x264_depth_y.png")])
    return [golden, kinds(61, 83, seed=4), kinds(480, 640, seed=9)]


def check_against_cv2(dmc, frames, qualities):
    from oracle.oracle_py import Port
    port = Port()
    n = len(frames)
    res = {opt: dmc.jpegRateDistortion(frames, qualities, dmc.filters.chain_params(0, *CHAIN), optimize=opt) for opt in (False, True)}
    for k, q in enumerate(qualities):
        for i in range(n):
            ok, buf = cv2.imencode(".jpg", frames[i], [cv2.IMWRITE_JPEG_QUALITY, q])
            ok2, obuf = cv2.imencode(".jpg", frames[i], [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, 1])
            assert ok and ok2
            dec = cv2.imdecode(buf, 0)
            filt = port.post_filter_set(dec, *CHAIN)
            sc, sf = np_sse(frames[i], dec)[0], np_sse(frames[i], filt)[0]
            for opt, nb in ((False, len(buf)), (True, len(obuf))):
                r = res[opt]
                where = (frames.shape, i, q, opt)
                assert r["bytes"][k, i] == nb, where
                assert r["sse_coded"][k, i] == sc, where
                assert r["sse_filtered"][k, i] == sf, where
                assert r["psnr_coded"][k, i] == dmc.psnrFromSSE(sc, frames[0].size), where
    for opt in (False, True):
        assert set(res[opt]) == {"bytes", "sse_coded", "psnr_coded", "sse_filtered", "psnr_filtered"}
        assert all(v.shape == (len(qualities), n) for v in res[opt].values())


def test_rd_sweep_matches_cv2_and_port(dmc):
    for frames in rd_frames():
        check_against_cv2(dmc, frames, QUALITIES)


def test_rd_sweep_200_frames_1080p_equals_public_calls(dmc):
    import torch
    import bench
    base = bench.base_frame()
    n, H, W = 200, base.shape[0], base.shape[1]
    frames = np.stack([bench.frame_np(base, 7 * f) for f in range(n)])
    qs = (20, 50, 90)
    params = dmc.filters.chain_params(0, *CHAIN)
    ctx = dmc.default_context()
    d_src = torch.from_numpy(frames).cuda()
    for opt in (False, True):
        host = dmc.jpegRateDistortion(frames, qs, params, optimize=opt)
        dev = dmc.jpegRateDistortion((d_src.data_ptr(), n, H, W), qs, params, optimize=opt)
        for key in host:
            assert np.array_equal(host[key], dev[key]), (opt, key)
        d_dec = torch.empty_like(d_src); d_filt = torch.empty_like(d_src)
        for k, q in enumerate(qs):
            _, nbytes = dmc.degradeJPEG((d_src.data_ptr(), n, H, W), q, dst=d_dec.data_ptr(), optimize=opt)
            ctx.chain_batch(d_dec.data_ptr(), d_filt.data_ptr(), n, H, W, params, device=True)
            ctx.synchronize()
            assert np.array_equal(host["bytes"][k], nbytes), (opt, q)
            assert np.array_equal(host["sse_coded"][k], dmc.frameSSE((d_src.data_ptr(), n, H, W), (d_dec.data_ptr(), n, H, W))), (opt, q)
            assert np.array_equal(host["sse_filtered"][k], dmc.frameSSE((d_src.data_ptr(), n, H, W), (d_filt.data_ptr(), n, H, W))), (opt, q)
    # spot check against cv2 and the port on two frames of the batch
    check_against_cv2(dmc, frames[[0, 199]], (50,))


def sweep(dmc, frames, qualities, params, flags=0, n=None, rows=None, cols=None, sse_filtered=True, sentinel=0xA5A5A5A5A5A5A5A5):
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    n = frames.shape[0] if n is None else n
    rows = frames.shape[1] if rows is None else rows
    cols = frames.shape[2] if cols is None else cols
    q = np.ascontiguousarray(qualities, np.int32)
    m = max(len(q), 1) * max(n, 1)
    out = [np.full(m, sentinel, np.uint64) for _ in range(3)]
    rc = capi.lib.dmc_jpeg_rd_sweep(ctx.h, C.c_void_p(frames.ctypes.data), capi.MEM_HOST, n, rows, cols, q.ctypes.data_as(C.POINTER(C.c_int)), len(q), flags,
                                    C.byref(params) if params is not None else None, out[0].ctypes.data_as(U64), out[1].ctypes.data_as(U64),
                                    out[2].ctypes.data_as(U64) if sse_filtered else None)
    return rc, out


def test_rd_sweep_without_chain_leaves_sse_filtered_untouched(dmc):
    from depthmapcompression_b200 import capi
    frames = kinds(61, 83, seed=2)
    rc, (nb, sc, sf) = sweep(dmc, frames, (30, 70), None)
    assert rc == capi.DMC_OK
    assert np.all(sf == 0xA5A5A5A5A5A5A5A5)
    r = dmc.jpegRateDistortion(frames, (30, 70), dmc.filters.chain_params(0, *CHAIN))
    assert np.array_equal(nb.reshape(2, -1), r["bytes"]) and np.array_equal(sc.reshape(2, -1), r["sse_coded"])
    rc, _ = sweep(dmc, frames, (30,), None, sse_filtered=False)            # sse_filtered may be NULL
    assert rc == capi.DMC_OK
    r = dmc.jpegRateDistortion(frames, (30,))
    assert set(r) == {"bytes", "sse_coded", "psnr_coded"}


def test_rd_sweep_quality_zero_acts_as_one(dmc):
    frames = kinds(61, 83, seed=6)
    r = dmc.jpegRateDistortion(frames, (0, 1), dmc.filters.chain_params(0, *CHAIN))
    for key in r:
        assert np.array_equal(r[key][0], r[key][1]), key


def test_rd_sweep_argument_rules(dmc):
    from depthmapcompression_b200 import capi
    frames = kinds(61, 83, seed=1)
    good = dmc.filters.chain_params(0, *CHAIN)
    untouched = lambda out: all(np.all(o == 0xA5A5A5A5A5A5A5A5) for o in out)     # noqa: E731
    for qs in ((), (-1,), (101,), (50, 101), (50, -5, 60)):
        rc, out = sweep(dmc, frames, qs, good)
        assert rc == capi.DMC_ERR_ARG and untouched(out), qs
    for flags in (2, 3, -1, 1 << 30):
        rc, out = sweep(dmc, frames, (50,), good, flags=flags)
        assert rc == capi.DMC_ERR_ARG and untouched(out), flags
    for chain in (capi.CHAIN_DEPTH32F, capi.CHAIN_DEPTH16U, capi.CHAIN_DISP32F, 4, -1):
        rc, out = sweep(dmc, frames, (50,), dmc.filters.chain_params(chain, *CHAIN, focus=75.0, baseline=575.0, amp=2.6))
        assert rc == capi.DMC_ERR_ARG and untouched(out), chain
    for bad in ((11, 1, 3, 5, 10), (2, -1, 3, 5, 10), (2, 1, 11, 5, 10), (2, 1, 3, 11, 10)):       # check_chain_params' radii
        rc, out = sweep(dmc, frames, (50,), dmc.filters.chain_params(0, *bad))
        assert rc == capi.DMC_ERR_ARG and untouched(out), bad
    rc, out = sweep(dmc, frames, (50,), dmc.filters.chain_params(0, *CHAIN, brange_method=capi.FULL_KERNEL_PAIR))
    assert rc == capi.DMC_ERR_ARG and untouched(out)
    rc, out = sweep(dmc, frames, (50,), dmc.filters.chain_params(0, *CHAIN, brange_method=capi.SEPARABLE_KERNEL))
    assert rc == capi.DMC_OK
    rc, out = sweep(dmc, frames, (50,), good, n=0)
    assert rc == capi.DMC_OK and untouched(out)
    for rows, cols in ((0, 83), (61, 0), (65536, 8), (8, 65536), (-3, 83)):                       # dmc_jpeg_encode_bound_ex's sizes
        rc, out = sweep(dmc, frames, (50,), good, rows=rows, cols=cols, n=0)
        assert rc == capi.DMC_ERR_SIZE and untouched(out), (rows, cols)
    rc, out = sweep(dmc, frames, (50,), good, n=-1)
    assert rc == capi.DMC_ERR_SIZE and untouched(out)
    rc, out = sweep(dmc, frames, (50,), good, sse_filtered=False)           # a chain needs somewhere to put its SSE
    assert rc == capi.DMC_ERR_SIZE and untouched(out)
    with pytest.raises(dmc.DmcError):
        dmc.jpegRateDistortion(frames, (), good)
