"""SSIM outputs of both rate-distortion sweeps (dmc_jpeg_rd_sweep_ssim, dmc_jpeg_view_rd_sweep_ssim; ssim=True of
jpegRateDistortion / jpegViewRateDistortion).  Every SSIM output must equal, bit for bit, frameSSIM of the frames the public
calls produce (degradeJPEG -> chain_batch / boundaryReconstructionFilterBatch -> renderViewBatch), in both Huffman modes, over
more than one group, from host and device sources; on samples it must equal the float64 reference on cv2 and the CPU port
to 1e-10.  bytes and the SSE outputs must not change with SSIM, NULL SSIM outputs must be the _ex entry points, and bad
arguments must return their error and write nothing."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_brf_rd_sweep import BRF, GRAY_CHAIN, B, coded
from test_gpu_view_rd_sweep import AMP, BASELINE, FOCUS, SENTINEL, cameras, intrinsics, mixed_batch, params, texture_of
from test_ssim_reference import ssim_ref

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu
TOL = 1e-10


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def gray_params(dmc):
    from depthmapcompression_b200 import capi
    return dmc.filters.chain_params(capi.CHAIN_DISP8U, *GRAY_CHAIN)


def depth_params(dmc, radii=(0, 0, 0, 0, 0.0)):
    return params(dmc, radii=radii)


def public_arms(dmc, disp, tex, q, opt, f, R, t, K, views=True):
    """SSIM of every arm through the public calls, host memory: (gray coded, filtered, brf [n]), (view coded, filtered, brf
    [n_views, n]).  D(x) = disp8U2depth32F is the 32F chain with radii 0 (the same views, see dmc_c.h)."""
    ctx = dmc.default_context()
    n, H, W = disp.shape
    dec, _ = dmc.degradeJPEG(disp, q, optimize=opt)
    filt = np.empty_like(disp)
    ctx.chain_batch(dec, filt, n, H, W, gray_params(dmc))
    brf = dmc.boundaryReconstructionFilterBatch(dec, None, *BRF)
    gray = tuple(dmc.frameSSIM(disp, x) for x in (dec, filt, brf))
    if not views:
        return gray, None

    def depth(x, p):
        z = np.empty(x.shape, np.float32)
        ctx.chain_batch(x, z, n, H, W, p)
        return z

    def render(z):
        return dmc.renderViewBatch(z, tex, f, R, t, K, isSub=True)

    ref = render(depth(disp, depth_params(dmc)))
    arms = (render(depth(dec, depth_params(dmc))), render(depth(dec, params(dmc))), render(depth(brf, depth_params(dmc))))
    view = tuple(np.stack([dmc.frameSSIM(ref[v], x[v]) for v in range(len(R))]) for x in arms)
    return gray, view


def check_against_public(dmc, disp, tex, qs, f, cams, device_too):
    import torch
    n, H, W = disp.shape
    K = intrinsics(f, H, W)
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    b = dmc.brf_params(*BRF)
    if device_too:
        d_src, d_tex = torch.from_numpy(disp).cuda(), torch.from_numpy(np.ascontiguousarray(tex)).cuda()
        torch.cuda.synchronize()
    for opt in (False, True):
        g = dmc.jpegRateDistortion(disp, qs, gray_params(dmc), optimize=opt, brf=b, ssim=True)
        v = dmc.jpegViewRateDistortion(disp, tex, qs, params(dmc), f, R, t, K, optimize=opt, brf=b, ssim=True)
        g0 = dmc.jpegRateDistortion(disp, qs, gray_params(dmc), optimize=opt, brf=b)
        v0 = dmc.jpegViewRateDistortion(disp, tex, qs, params(dmc), f, R, t, K, optimize=opt, brf=b)
        assert set(g) - set(g0) == {"ssim_coded", "ssim_filtered", "ssim_brf"}
        assert set(v) - set(v0) == {"ssim_view_coded", "ssim_view_filtered", "ssim_view_brf"}
        for key in g0:
            assert np.array_equal(g[key], g0[key]), (opt, key)
        for key in v0:
            assert np.array_equal(v[key], v0[key]), (opt, key)
        if device_too:
            gd = dmc.jpegRateDistortion((d_src.data_ptr(), n, H, W), qs, gray_params(dmc), optimize=opt, brf=b, ssim=True)
            vd = dmc.jpegViewRateDistortion((d_src.data_ptr(), n, H, W), (d_tex.data_ptr(), n, H, W), qs, params(dmc), f, R, t, K,
                                            optimize=opt, brf=b, ssim=True)
            for key in g:
                assert np.array_equal(gd[key], g[key]), (opt, key)
            for key in v:
                assert np.array_equal(vd[key], v[key]), (opt, key)
        for k, q in enumerate(qs):
            gray, view = public_arms(dmc, disp, tex, q, opt, f, R, t, K)
            for arm, x in zip(("coded", "filtered", "brf"), gray):
                assert np.array_equal(g["ssim_" + arm][k].view(np.uint64), x.view(np.uint64)), (opt, q, arm)
            for arm, x in zip(("coded", "filtered", "brf"), view):
                assert np.array_equal(v["ssim_view_" + arm][k].view(np.uint64), x.view(np.uint64)), (opt, q, arm)


def test_40_frames_1080p_equal_public_calls(dmc):
    import bench
    base = bench.base_frame()
    disp = np.stack([bench.frame_np(base, 7 * i) for i in range(40)])
    tex = np.stack([texture_of(d) for d in disp])
    check_against_public(dmc, disp, tex, (30, 90), 1100.0, cameras()[:1], device_too=True)


def test_more_than_one_group_of_small_frames(dmc):
    """2100 frames: the sweeps' groups hold at most 2048 frames"""
    from oracle.oracle_py import synth_disp
    disp = np.stack([synth_disp(16, 24, i % 50) for i in range(2100)])
    tex = np.stack([texture_of(d) for d in disp])
    check_against_public(dmc, disp, tex, (40,), 20.0, cameras(30.0)[:2], device_too=False)


def test_samples_equal_float64_reference(dmc, port):
    from oracle.oracle_py import synth_disp
    from _util import load_png
    rs = np.random.RandomState(9)
    small = np.stack([synth_disp(61, 83, 2), np.clip(synth_disp(61, 83, 3).astype(np.int16) + rs.randint(-30, 31, (61, 83)), 1, 255).astype(np.uint8)])
    kinect = load_png("kinect_meeting_q80.png")[None]
    for disp, f, qs in ((small, 20.0, (10, 70)), (kinect, 510.0, (50,))):
        n, H, W = disp.shape
        tex = np.stack([texture_of(d) for d in disp])
        cams = cameras(30.0 if H < 100 else 100.0)[:2]
        K = intrinsics(f, H, W)
        R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
        b = dmc.brf_params(*BRF)
        g = dmc.jpegRateDistortion(disp, qs, gray_params(dmc), optimize=True, brf=b, ssim=True)
        v = dmc.jpegViewRateDistortion(disp, tex, qs, params(dmc), f, R, t, K, optimize=True, exact_divide=True, brf=b, ssim=True)

        def D(x):
            return port.disp8u2depth32f(x, FOCUS * BASELINE, AMP, 0.0)

        def view(depth, img, Rv, tv):
            return port.fill_small_hole(port.project_image(img, port.reproject_xyz(depth, f), Rv, tv, K, True, rcp=False)[0])

        for i in range(n):
            ref = [view(D(disp[i]), tex[i], Rv, tv) for Rv, tv in cams]
            for k, q in enumerate(qs):
                dec = coded(disp[i], q, True)[1]
                filt = port.post_filter_set(dec, *GRAY_CHAIN)
                bd = B(port, dec)
                for arm, x in (("coded", dec), ("filtered", filt), ("brf", bd)):
                    assert abs(g["ssim_" + arm][k, i] - ssim_ref(disp[i], x)) <= TOL, (H, q, i, arm)
                zs = {"coded": D(dec), "filtered": port.filter_disp8u_depth32f(dec, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0), "brf": D(bd)}
                for vi, (Rv, tv) in enumerate(cams):
                    for arm, z in zs.items():
                        assert abs(v["ssim_view_" + arm][k, vi, i] - ssim_ref(ref[vi], view(z, tex[i], Rv, tv))) <= TOL, (H, q, i, vi, arm)


def test_argument_rules(dmc):
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    U64, DP, IP = C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(C.c_int)
    q = np.array([50], np.int32)
    pg, pv, good = gray_params(dmc), params(dmc), dmc.brf_params(*BRF)

    def run(disp, tex, fn, p, b, q_outs, sse_outs=(True,) * 4, ex=False):
        n, H, W = disp.shape
        nv = 2 if fn == "view" else 1
        sse = [np.full(nv * n, SENTINEL, np.uint64) for _ in range(4)]
        qq = [np.full(nv * n, -7.0) for _ in range(3)]
        s_args = [o.ctypes.data_as(U64) if ok else None for o, ok in zip(sse, sse_outs)]
        q_args = [] if ex else [o.ctypes.data_as(DP) if ok else None for o, ok in zip(qq, q_outs)]
        pp = C.byref(p) if p is not None else None
        bb = C.byref(b) if b is not None else None
        if fn == "gray":
            f = capi.lib.dmc_jpeg_rd_sweep_ex if ex else capi.lib.dmc_jpeg_rd_sweep_ssim
            rc = f(ctx.h, C.c_void_p(disp.ctypes.data), capi.MEM_HOST, n, H, W, q.ctypes.data_as(IP), 1, 0, pp, bb, *s_args, *q_args)
        else:
            cams = cameras(30.0)[:2]
            R = np.ascontiguousarray(np.stack([c[0] for c in cams])); t = np.ascontiguousarray(np.stack([c[1] for c in cams]))
            K = np.ascontiguousarray(intrinsics(20.0, H, W))
            f = capi.lib.dmc_jpeg_view_rd_sweep_ex if ex else capi.lib.dmc_jpeg_view_rd_sweep_ssim
            rc = f(ctx.h, C.c_void_p(disp.ctypes.data), C.c_void_p(tex.ctypes.data), capi.MEM_HOST, n, H, W, q.ctypes.data_as(IP), 1, 0, pp, bb,
                   20.0, R.ctypes.data_as(DP), t.ctypes.data_as(DP), 2, K.ctypes.data_as(DP), 1, 0, *s_args, *q_args)
        untouched = all(np.all(o == SENTINEL) for o in sse) and all(np.all(o == -7.0) for o in qq)
        return rc, untouched, sse, qq

    disp, tex = mixed_batch(24, 32)
    for fn, p in (("gray", pg), ("view", pv)):
        rc, _, sse, qq = run(disp, tex, fn, p, good, (True,) * 3)
        assert rc == capi.DMC_OK and all(np.all((o > -1) & (o <= 1)) for o in qq), fn
        rc_ex, _, sse_ex, _ = run(disp, tex, fn, p, good, (True,) * 3, ex=True)           # NULL SSIM outputs: the _ex entry point
        rc_n, untouched_q, sse_n, qq_n = run(disp, tex, fn, p, good, (False,) * 3)
        assert rc_ex == rc_n == capi.DMC_OK and all(np.array_equal(x, y) and np.array_equal(x, z) for x, y, z in zip(sse, sse_ex, sse_n)), fn
        assert all(np.all(o == -7.0) for o in qq_n), fn
        for outs in ((True, False, True), (True, True, False)):                          # filtered / BRF SSIM missing
            rc, untouched, _, _ = run(disp, tex, fn, p, good, outs)
            assert rc == capi.DMC_ERR_SIZE and untouched, (fn, outs)
        rc, _, _, qq = run(disp, tex, fn, p, None, (True, True, False))                 # no BRF arm: its SSIM is not needed
        assert rc == capi.DMC_OK and np.all(qq[2] == -7.0), fn
        tiny, ttex = np.ascontiguousarray(disp[:, :10, :12]), np.ascontiguousarray(tex[:, :10, :12])
        rc, untouched, _, _ = run(tiny, ttex, fn, p, good, (True,) * 3)                 # under 11 x 11 with SSIM
        assert rc == capi.DMC_ERR_SIZE and untouched, fn
        rc, _, _, _ = run(tiny, ttex, fn, p, good, (False,) * 3)                        # ... and without
        assert rc == capi.DMC_OK, fn
    rc, _, _, qq = run(disp, tex, "gray", None, good, (True, False, True), sse_outs=(True, True, False, True))   # no chain: no filtered SSIM
    assert rc == capi.DMC_OK and np.all(qq[1] == -7.0) and np.all(qq[2] != -7.0)
    with pytest.raises(dmc.DmcError):
        dmc.jpegRateDistortion(np.zeros((1, 10, 30), np.uint8), (50,), ssim=True)
