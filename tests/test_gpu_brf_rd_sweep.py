"""The boundary reconstruction filter as a third arm of both rate-distortion sweeps (dmc_jpeg_rd_sweep_ex,
dmc_jpeg_view_rd_sweep_ex; brf= of jpegRateDistortion / jpegViewRateDistortion).  With B = boundaryReconstructionFilter on the
8-bit decoded disparity, sse_brf must equal SSE(frame, port.brf(cv2.imdecode(stream))) and sse_view_brf the SSE of the port's
view of D(B(decoded)) against the reference view, bit for bit; the other outputs must be those of the entry points without
the arm; a 40-frame 1080p batch must equal the public calls degradeJPEG -> boundaryReconstructionFilterBatch -> render / SSE."""
import ctypes as C

import numpy as np
import pytest

from _util import load_png
from test_pointcloud import intel_host
from test_gpu_view_rd_sweep import (AMP, BASELINE, CHAIN, FOCUS, SENTINEL, cameras, intrinsics, mixed_batch, np_sse, params,
                                    texture_of)

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu

BRF = ((13, 13), 1.0, 1.0, 1.0)                   # main.cpp:306-311
GRAY_CHAIN = (2, 1, 3, 5, 10)


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


def coded(disp, q, opt):
    ok, buf = cv2.imencode(".jpg", disp, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, int(opt)])
    assert ok
    return len(buf), cv2.imdecode(buf, 0)


def B(port, x, brf=BRF):
    (kw, kh), frec, color, space = brf
    return port.brf(x, kw, kh, frec, color, space)


def gray_check(dmc, port, frames, qualities, brf=BRF):
    from depthmapcompression_b200 import capi
    p = dmc.filters.chain_params(capi.CHAIN_DISP8U, *GRAY_CHAIN)
    b = dmc.brf_params(*brf)
    for opt in (False, True):
        r = dmc.jpegRateDistortion(frames, qualities, p, optimize=opt, brf=b)
        old = dmc.jpegRateDistortion(frames, qualities, p, optimize=opt)
        for key in old:
            assert np.array_equal(r[key], old[key]), (opt, key)
        for k, q in enumerate(qualities):
            for i in range(len(frames)):
                nb, dec = coded(frames[i], q, opt)
                assert r["bytes"][k, i] == nb
                assert r["sse_brf"][k, i] == np_sse(frames[i], B(port, dec, brf)), (frames.shape, q, opt, i)
        assert np.array_equal(r["psnr_brf"], dmc.psnrFromSSE(r["sse_brf"], frames[0].size))
        nobrf = dmc.jpegRateDistortion(frames, qualities, None, optimize=opt, brf=b)
        assert np.array_equal(nobrf["sse_brf"], r["sse_brf"]) and "sse_filtered" not in nobrf


def view_expect(port, disp, tex, qualities, f, cams, K, sub, rcp, opt, brf=BRF):
    def D(x):
        return port.disp8u2depth32f(x, FOCUS * BASELINE, AMP, 0.0)

    def view(depth, img, R, t):
        return port.fill_small_hole(port.project_image(img, port.reproject_xyz(depth, f), R, t, K, sub, rcp=rcp)[0])

    sb = np.zeros((len(qualities), len(cams), len(disp)), np.uint64)
    for i in range(len(disp)):
        ref = [view(D(disp[i]), tex[i], R, t) for R, t in cams]
        for k, q in enumerate(qualities):
            dz = D(B(port, coded(disp[i], q, opt)[1], brf))
            for v, (R, t) in enumerate(cams):
                sb[k, v, i] = np_sse(ref[v], view(dz, tex[i], R, t))
    return sb


def view_check(dmc, port, disp, tex, qualities, f, cams, sub, opts=(False, True)):
    K = intrinsics(f, disp.shape[1], disp.shape[2])
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    b = dmc.brf_params(*BRF)
    for rcp in [False] + ([True] if intel_host() else []):
        for opt in opts:
            r = dmc.jpegViewRateDistortion(disp, tex, qualities, params(dmc), f, R, t, K, isSub=sub, optimize=opt, exact_divide=not rcp, brf=b)
            old = dmc.jpegViewRateDistortion(disp, tex, qualities, params(dmc), f, R, t, K, isSub=sub, optimize=opt, exact_divide=not rcp)
            for key in old:
                assert np.array_equal(r[key], old[key]), (key, rcp, opt)
            sb = view_expect(port, disp, tex, qualities, f, cams, K, sub, rcp, opt)
            assert np.array_equal(r["sse_view_brf"], sb), (disp.shape, sub, rcp, opt)
            assert np.array_equal(r["psnr_view_brf"], dmc.psnrFromSSE(sb, sb.dtype.type(3 * disp[0].size)))


@pytest.mark.parametrize("H,W", [(3, 3), (17, 23), (61, 83)])
def test_small_sizes_equal_port(dmc, port, H, W):
    from oracle.oracle_py import synth_disp
    rs = np.random.RandomState(H * 7 + W)
    disp = np.stack([rs.randint(1, 256, (H, W)).astype(np.uint8), synth_disp(H, W, 3), np.full((H, W), 40, np.uint8)])
    gray_check(dmc, port, disp, (5, 50, 95))
    tex = rs.randint(0, 256, (3, H, W, 3)).astype(np.uint8)
    for sub in (False, True):
        view_check(dmc, port, disp, tex, (5, 50, 95), 20.0, cameras(tx=30.0), sub)


def test_golden_kinect_frames_equal_port(dmc, port):
    disp = np.stack([load_png(n) for n in ("kinect_meeting_q80.png", "kinect_desk_q80.png")])
    gray_check(dmc, port, disp, (10, 60, 100))
    tex = np.stack([cv2.cvtColor(d, cv2.COLOR_GRAY2BGR) for d in disp])
    view_check(dmc, port, disp, tex, (10, 60, 100), 510.0, cameras(), True)


def test_1080p_equals_port(dmc, port):
    from oracle.oracle_py import synth_disp
    d = synth_disp(1080, 1920, 5)
    gray_check(dmc, port, d[None], (20, 90))
    view_check(dmc, port, d[None], texture_of(d)[None], (20, 90), 1100.0, cameras()[1:], True)


def test_mixed_batch_equals_frames_alone(dmc):
    disp, tex = mixed_batch()
    f = 100.0
    K = intrinsics(f, *disp.shape[1:])
    cams = cameras(30.0)[:2]
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    b = dmc.brf_params(*BRF)
    batch = dmc.jpegViewRateDistortion(disp, tex, (15, 75), params(dmc), f, R, t, K, exact_divide=True, brf=b)
    for i in range(len(disp)):
        one = dmc.jpegViewRateDistortion(disp[i:i + 1], tex[i:i + 1], (15, 75), params(dmc), f, R, t, K, exact_divide=True, brf=b)
        for key in one:
            assert np.array_equal(batch[key][..., i:i + 1], one[key]), (i, key)


def test_40_frames_1080p_equal_public_calls(dmc, port):
    import torch
    import bench
    base = bench.base_frame()
    n, H, W = 40, base.shape[0], base.shape[1]
    disp = np.stack([bench.frame_np(base, 7 * i) for i in range(n)])
    tex = np.stack([texture_of(d) for d in disp])
    qs, f = (30, 90), 1100.0
    cams = cameras()[:1]
    K = intrinsics(f, H, W)
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    b = dmc.brf_params(*BRF)
    from depthmapcompression_b200 import capi
    pg = dmc.filters.chain_params(capi.CHAIN_DISP8U, *GRAY_CHAIN)
    d_src, d_tex = torch.from_numpy(disp).cuda(), torch.from_numpy(tex).cuda()
    d_dec, d_brf = torch.empty_like(d_src), torch.empty_like(d_src)
    torch.cuda.synchronize()
    ctx = dmc.default_context()

    def view(depth, img, Rv, tv):
        return dmc.fillSmallHole(dmc.projectImagefromXYZ(img, None, dmc.reprojectXYZ(depth, None, f), Rv, tv, K, isSub=True))

    def sse3(a, c):
        return int(dmc.frameSSE(a.reshape(1, H, 3 * W), c.reshape(1, H, 3 * W))[0])

    ref = [[view(dmc.disp8U2depth32F(disp[i], None, FOCUS * BASELINE, AMP, 0.0), tex[i], Rv, tv) for Rv, tv in cams] for i in range(n)]
    for opt in (False, True):
        host = dmc.jpegRateDistortion(disp, qs, pg, optimize=opt, brf=b)
        dev = dmc.jpegRateDistortion((d_src.data_ptr(), n, H, W), qs, pg, optimize=opt, brf=b)
        vhost = dmc.jpegViewRateDistortion(disp, tex, qs, params(dmc), f, R, t, K, optimize=opt, brf=b)
        vdev = dmc.jpegViewRateDistortion((d_src.data_ptr(), n, H, W), (d_tex.data_ptr(), n, H, W), qs, params(dmc), f, R, t, K, optimize=opt, brf=b)
        for key in host:
            assert np.array_equal(host[key], dev[key]), (opt, key)
        for key in vhost:
            assert np.array_equal(vhost[key], vdev[key]), (opt, key)
        for k, q in enumerate(qs):
            _, nb = dmc.degradeJPEG((d_src.data_ptr(), n, H, W), q, dst=d_dec.data_ptr(), optimize=opt)
            dmc.boundaryReconstructionFilterBatch((d_dec.data_ptr(), n, H, W), d_brf.data_ptr(), *BRF)
            ctx.synchronize()
            assert np.array_equal(host["bytes"][k], nb) and np.array_equal(vhost["bytes"][k], nb), (opt, q)
            sb = dmc.frameSSE((d_src.data_ptr(), n, H, W), (d_brf.data_ptr(), n, H, W))
            assert np.array_equal(host["sse_brf"][k], sb), (opt, q)
            bb = d_brf.cpu().numpy()
            for i in range(n):
                z = dmc.disp8U2depth32F(bb[i], None, FOCUS * BASELINE, AMP, 0.0)
                for v, (Rv, tv) in enumerate(cams):
                    assert vhost["sse_view_brf"][k, v, i] == sse3(ref[i][v], view(z, tex[i], Rv, tv)), (opt, q, i, v)
    # and against the CPU port on one frame of the batch
    assert host["sse_brf"][1, 13] == np_sse(disp[13], B(port, coded(disp[13], 90, True)[1]))


def test_argument_rules(dmc):
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    disp, tex = mixed_batch(24, 32)
    n = len(disp)
    U64, DP = C.POINTER(C.c_uint64), C.POINTER(C.c_double)
    pg = dmc.filters.chain_params(capi.CHAIN_DISP8U, *GRAY_CHAIN)
    pv = params(dmc)
    q = np.array([50], np.int32)
    cams = cameras(30.0)[:2]
    R = np.ascontiguousarray(np.stack([c[0] for c in cams])); t = np.ascontiguousarray(np.stack([c[1] for c in cams]))
    K = np.ascontiguousarray(intrinsics(20.0, 24, 32))

    def gray(b, p=pg, outs=(True,) * 4):
        out = [np.full(n, SENTINEL, np.uint64) for _ in range(4)]
        rc = capi.lib.dmc_jpeg_rd_sweep_ex(ctx.h, C.c_void_p(disp.ctypes.data), capi.MEM_HOST, n, 24, 32, q.ctypes.data_as(C.POINTER(C.c_int)), 1, 0,
                                           C.byref(p) if p is not None else None, C.byref(b) if b is not None else None,
                                           *[o.ctypes.data_as(U64) if ok else None for o, ok in zip(out, outs)])
        return rc, all(np.all(o == SENTINEL) for o in out), out

    def view(b, p=pv, outs=(True,) * 4):
        out = [np.full(2 * n, SENTINEL, np.uint64) for _ in range(4)]
        rc = capi.lib.dmc_jpeg_view_rd_sweep_ex(ctx.h, C.c_void_p(disp.ctypes.data), C.c_void_p(tex.ctypes.data), capi.MEM_HOST, n, 24, 32,
                                                q.ctypes.data_as(C.POINTER(C.c_int)), 1, 0, C.byref(p) if p is not None else None,
                                                C.byref(b) if b is not None else None, 20.0, R.ctypes.data_as(DP), t.ctypes.data_as(DP), 2,
                                                K.ctypes.data_as(DP), 1, 0, *[o.ctypes.data_as(U64) if ok else None for o, ok in zip(out, outs)])
        return rc, all(np.all(o == SENTINEL) for o in out), out

    good = dmc.brf_params(*BRF)
    for fn in (gray, view):
        rc, untouched, out = fn(good)
        assert rc == capi.DMC_OK and not np.any(out[3] == SENTINEL), fn.__name__
        rc, untouched, out = fn(None)                           # no BRF arm: sse_brf is not written
        assert rc == capi.DMC_OK and np.all(out[3] == SENTINEL), fn.__name__
        rc, untouched, out = fn(None, outs=(True, True, True, False))
        assert rc == capi.DMC_OK, fn.__name__
        for ks in ((0, 13), (13, 0), (23, 23), (13, 22), (-1, 1)):
            rc, untouched, _ = fn(dmc.brf_params(ks))
            assert rc == capi.DMC_ERR_ARG and untouched, (fn.__name__, ks)
        rc, untouched, _ = fn(good, outs=(True, True, True, False))
        assert rc == capi.DMC_ERR_SIZE and untouched, fn.__name__
    rc, untouched, out = gray(good, p=None, outs=(True, True, False, True))      # the BRF arm without the chain
    assert rc == capi.DMC_OK and not np.any(out[3] == SENTINEL)
    rc, untouched, _ = view(good, p=None)                                         # the view sweep still needs p for D
    assert rc == capi.DMC_ERR_ARG and untouched
    # the old entry points are the _ex ones with b = NULL
    r_old = [np.full(n, SENTINEL, np.uint64) for _ in range(3)]
    assert capi.lib.dmc_jpeg_rd_sweep(ctx.h, C.c_void_p(disp.ctypes.data), capi.MEM_HOST, n, 24, 32, q.ctypes.data_as(C.POINTER(C.c_int)), 1, 0,
                                      C.byref(pg), *[o.ctypes.data_as(U64) for o in r_old]) == capi.DMC_OK
    rc, _, out = gray(None)
    assert all(np.array_equal(a, c) for a, c in zip(r_old, out[:3]))
