"""The view-synthesis rate-distortion sweep on the GPU (dmc_jpeg_view_rd_sweep, jpegViewRateDistortion): for every frame,
quality and camera it must report the size of cv2.imencode's stream and, bit for bit, the SSE between the reference view
and the views rendered from the decoded and from the filtered depth, where a view is the port's
fill_small_hole(project_image(texture, reproject_xyz(depth, f), R, t, K, isSub)) and the depths come from the port's
disp8u2depth32f / filter_disp8u_depth32f of cv2.imdecode's frame.  The batched renderer must give every frame of a batch
what it gives the frame alone, and the sweep must equal the composition of the library's public single-frame calls."""
import ctypes as C

import numpy as np
import pytest

from _util import load_png
from test_pointcloud import VIEWS, intel_host, rot

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu

FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6
CHAIN = (1, 0, 1, 3, 65.0)                       # pointcloudTest's filterDisp8U2Depth32F (main.cpp:341)
SENTINEL = 0xA5A5A5A5A5A5A5A5


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


@pytest.fixture(scope="module")
def port():
    from oracle.oracle_py import Port
    return Port()


def params(dmc, chain=None, radii=CHAIN, **kw):
    from depthmapcompression_b200 import capi
    return dmc.filters.chain_params(capi.CHAIN_DEPTH32F if chain is None else chain, *radii, focus=FOCUS, baseline=BASELINE, amp=AMP, **kw)


def intrinsics(f, H, W):
    K = np.eye(3) * f; K[0, 2] = (W - 1) * 0.5; K[1, 2] = (H - 1) * 0.5; K[2, 2] = 1.0      # main.cpp:132-136
    return K


def cameras(tx=100.0):
    rv = dict((n, (R, t)) for n, R, t in VIEWS)["rot"]
    return [(np.eye(3), np.array([tx, 0., 0.])), (np.eye(3), np.array([-tx, 0., 0.])), rv]


def np_sse(a, b):
    return int(((a.astype(np.int64) - b) ** 2).sum())


def texture_of(d):
    return np.stack([d, ((d.astype(np.int32) * 7) & 255).astype(np.uint8), 255 - d], -1)


def expect(port, disp, tex, qualities, f, cams, K, sub, rcp, radii=CHAIN):
    """The composition the sweep stands for, on the CPU: -> (bytes [2, n_q, n], sse_coded, sse_filtered [n_q, n_views, n])"""
    n = len(disp)
    nb = np.zeros((2, len(qualities), n), np.uint64)
    sc = np.zeros((len(qualities), len(cams), n), np.uint64); sf = np.zeros_like(sc)

    def D(x):
        return port.disp8u2depth32f(x, FOCUS * BASELINE, AMP, 0.0)

    def view(depth, img, R, t):
        return port.fill_small_hole(port.project_image(img, port.reproject_xyz(depth, f), R, t, K, sub, rcp=rcp)[0])

    for i in range(n):
        ref = [view(D(disp[i]), tex[i], R, t) for R, t in cams]
        for k, q in enumerate(qualities):
            for opt in (0, 1):
                ok, buf = cv2.imencode(".jpg", disp[i], [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, opt])
                assert ok
                nb[opt, k, i] = len(buf)
            dec = cv2.imdecode(buf, 0)
            filt = port.filter_disp8u_depth32f(dec, FOCUS, BASELINE, AMP, *radii)
            for v, (R, t) in enumerate(cams):
                sc[k, v, i] = np_sse(ref[v], view(D(dec), tex[i], R, t))
                sf[k, v, i] = np_sse(ref[v], view(filt, tex[i], R, t))
    return nb, sc, sf


def check(dmc, port, disp, tex, qualities, f, cams, sub, radii=CHAIN):
    K = intrinsics(f, disp.shape[1], disp.shape[2])
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    for rcp in [False] + ([True] if intel_host() else []):
        nb, sc, sf = expect(port, disp, tex, qualities, f, cams, K, sub, rcp, radii)
        for opt in (False, True):
            r = dmc.jpegViewRateDistortion(disp, tex, qualities, params(dmc, radii=radii), f, R, t, K, isSub=sub, optimize=opt, exact_divide=not rcp)
            where = (disp.shape, sub, rcp, opt)
            assert np.array_equal(r["bytes"], nb[int(opt)]), where
            assert np.array_equal(r["sse_view_coded"], sc), where
            assert np.array_equal(r["sse_view_filtered"], sf), where
            assert r["psnr_view_coded"].shape == sc.shape and r["psnr_view_filtered"].shape == sf.shape
            assert np.array_equal(r["psnr_view_filtered"], dmc.psnrFromSSE(sf, sf.dtype.type(3 * disp[0].size))), where


@pytest.mark.parametrize("H,W", [(3, 3), (17, 23), (61, 83)])
def test_view_sweep_small_sizes_equal_port(dmc, port, H, W):
    from oracle.oracle_py import synth_disp
    rs = np.random.RandomState(H * 31 + W)
    disp = np.stack([rs.randint(1, 256, (H, W)).astype(np.uint8), synth_disp(H, W, 3), np.full((H, W), 40, np.uint8)])
    tex = rs.randint(0, 256, (3, H, W, 3)).astype(np.uint8)
    for sub in (False, True):
        check(dmc, port, disp, tex, (5, 50, 95), 20.0, cameras(tx=30.0), sub)


def test_view_sweep_golden_kinect_frames_equal_port(dmc, port):
    disp = np.stack([load_png(n) for n in ("kinect_meeting_q80.png", "kinect_desk_q80.png")])
    tex = np.stack([cv2.cvtColor(d, cv2.COLOR_GRAY2BGR) for d in disp])         # the "depth map view" (main.cpp:345-349)
    for sub in (False, True):
        check(dmc, port, disp, tex, (10, 60, 100), 510.0, cameras(), sub)


def test_view_sweep_1080p_equals_port(dmc, port):
    from oracle.oracle_py import synth_disp
    d = synth_disp(1080, 1920, 5)
    check(dmc, port, d[None], texture_of(d)[None], (20, 90), 1100.0, cameras()[1:], True)


def test_zero_radii_chain_is_the_unfiltered_depth(dmc, port):
    from oracle.oracle_py import synth_disp
    rs = np.random.RandomState(8)
    frames = [synth_disp(61, 83, 2), rs.randint(0, 256, (61, 83)).astype(np.uint8), np.zeros((17, 23), np.uint8), load_png("kinect_desk_q50.png")]
    pfs = dmc.PostFilterSet()
    for x in frames:
        d = dmc.disp8U2depth32F(x, None, FOCUS * BASELINE, AMP, 0.0)
        z = pfs.filterDisp8U2Depth32F(x, None, FOCUS, BASELINE, AMP, 0, 0, 0, 0, 65.0)
        valid = x != 0
        assert np.array_equal(d.view(np.uint32)[valid], z.view(np.uint32)[valid]), x.shape
        # disparity 0: the converter gives +inf, the 1-tap range filter inf - inf = NaN; neither point is ever drawn
        assert np.all(np.isposinf(d[~valid])) and np.all(np.isnan(z[~valid])), x.shape
        assert np.array_equal(d.view(np.uint32), port.disp8u2depth32f(x, FOCUS * BASELINE, AMP, 0.0).view(np.uint32)), x.shape
        pz = port.filter_disp8u_depth32f(x, FOCUS, BASELINE, AMP, 0, 0, 0, 0, 65.0)          # (NaN payloads differ between GPU and x86)
        assert np.array_equal(z.view(np.uint32)[valid], pz.view(np.uint32)[valid]) and np.all(np.isnan(pz[~valid])), x.shape
    # so the sweep with all radii 0 renders the same view from the coded and from the "filtered" depth
    disp = np.stack(frames[:2]); tex = np.stack([texture_of(x) for x in disp])
    r = dmc.jpegViewRateDistortion(disp, tex, (10, 70), params(dmc, radii=(0, 0, 0, 0, 65.0)), 20.0,
                                   np.stack([c[0] for c in cameras(30.0)]), np.stack([c[1] for c in cameras(30.0)]), intrinsics(20.0, 61, 83), exact_divide=True)
    assert np.array_equal(r["sse_view_coded"], r["sse_view_filtered"])
    assert r["sse_view_coded"].any()


def mixed_batch(H=120, W=160):
    """Frames that need different numbers of fixed-point iterations under one camera: a flat frame, a near frame whose
    points collapse onto a few pixels in the far view, and occlusion-heavy content."""
    from oracle.oracle_py import synth_disp
    rs = np.random.RandomState(17)
    flat = np.full((H, W), 90, np.uint8)
    near = (200 + rs.randint(0, 50, (H, W))).astype(np.uint8)
    blocks = np.kron(rs.randint(1, 256, (H // 4, W // 4)), np.ones((4, 4), np.int64)).astype(np.uint8)
    noisy = np.clip(synth_disp(H, W, 4).astype(np.int16) + rs.randint(-60, 61, (H, W)), 1, 255).astype(np.uint8)
    disp = np.stack([flat, near, blocks, noisy, flat.copy()])
    return disp, np.stack([texture_of(d) for d in disp])


def test_mixed_batch_equals_frames_alone_and_port(dmc, port):
    disp, tex = mixed_batch()
    f = 100.0
    K = intrinsics(f, *disp.shape[1:])
    cams = [(np.eye(3), np.array([0., 0., 3e4])), (rot(0.3, -0.2), np.array([150., -40., -100.]))]
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    qs = (15, 75)
    for sub in (False, True):
        batch = dmc.jpegViewRateDistortion(disp, tex, qs, params(dmc), f, R, t, K, isSub=sub, exact_divide=True)
        for i in range(len(disp)):
            one = dmc.jpegViewRateDistortion(disp[i:i + 1], tex[i:i + 1], qs, params(dmc), f, R, t, K, isSub=sub, exact_divide=True)
            for key in one:
                assert np.array_equal(batch[key][..., i:i + 1], one[key]), (sub, i, key)
        nb, sc, sf = expect(port, disp, tex, qs, f, cams, K, sub, False)
        assert np.array_equal(batch["sse_view_coded"], sc) and np.array_equal(batch["sse_view_filtered"], sf), sub
        assert np.array_equal(batch["bytes"], nb[0]), sub


def public_calls(dmc, d_src, tex, n, qs, f, cams, K, opt):
    """The sweep through the library's public calls: degradeJPEG -> filterDisp8U2Depth32F -> reprojectXYZ ->
    projectImagefromXYZ -> fillSmallHole -> frameSSE."""
    import torch
    H, W = tex.shape[1:3]
    pfs = dmc.PostFilterSet()

    def view(depth, img, R, t):
        xyz = dmc.reprojectXYZ(depth, None, f)
        return dmc.fillSmallHole(dmc.projectImagefromXYZ(img, None, xyz, R, t, K, isSub=True))

    def sse(a, b):
        return int(dmc.frameSSE(a.reshape(1, H, 3 * W), b.reshape(1, H, 3 * W))[0])

    src = d_src.cpu().numpy()
    ref = [[view(dmc.disp8U2depth32F(src[i], None, FOCUS * BASELINE, AMP, 0.0), tex[i], R, t) for R, t in cams] for i in range(n)]
    nb = np.zeros((len(qs), n), np.uint64)
    sc = np.zeros((len(qs), len(cams), n), np.uint64); sf = np.zeros_like(sc)
    d_dec = torch.empty_like(d_src)
    for k, q in enumerate(qs):
        _, nb[k] = dmc.degradeJPEG((d_src.data_ptr(), n, H, W), q, dst=d_dec.data_ptr(), optimize=opt)
        dmc.default_context().synchronize()
        dec = d_dec.cpu().numpy()
        for i in range(n):
            dz = dmc.disp8U2depth32F(dec[i], None, FOCUS * BASELINE, AMP, 0.0)
            fz = pfs.filterDisp8U2Depth32F(dec[i], None, FOCUS, BASELINE, AMP, *CHAIN)
            for v, (R, t) in enumerate(cams):
                sc[k, v, i] = sse(ref[i][v], view(dz, tex[i], R, t))
                sf[k, v, i] = sse(ref[i][v], view(fz, tex[i], R, t))
    return nb, sc, sf


def test_view_sweep_40_frames_1080p_equals_public_calls(dmc, port):
    import torch
    import bench
    base = bench.base_frame()
    n, H, W = 40, base.shape[0], base.shape[1]
    disp = np.stack([bench.frame_np(base, 7 * i) for i in range(n)])
    tex = np.stack([texture_of(d) for d in disp])
    qs, f = (30, 90), 1100.0
    cams = cameras()[:2]
    K = intrinsics(f, H, W)
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    d_src, d_tex = torch.from_numpy(disp).cuda(), torch.from_numpy(tex).cuda()
    torch.cuda.synchronize()
    for opt in (False, True):
        host = dmc.jpegViewRateDistortion(disp, tex, qs, params(dmc), f, R, t, K, optimize=opt)
        dev = dmc.jpegViewRateDistortion((d_src.data_ptr(), n, H, W), (d_tex.data_ptr(), n, H, W), qs, params(dmc), f, R, t, K, optimize=opt)
        for key in host:
            assert np.array_equal(host[key], dev[key]), (opt, key)
        nb, sc, sf = public_calls(dmc, d_src, tex, n, qs, f, cams, K, opt)
        assert np.array_equal(host["bytes"], nb), opt
        assert np.array_equal(host["sse_view_coded"], sc), opt
        assert np.array_equal(host["sse_view_filtered"], sf), opt
    # and against the CPU port on one frame of the batch
    check(dmc, port, disp[[13]], tex[[13]], (30,), f, cams[:1], True)


def sweep(dmc, disp, tex, qs, p, f=20.0, R=None, t=None, K=None, n_views=None, flags=0, render_flags=0, n=None, rows=None, cols=None,
          outputs=(True, True, True)):
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    n = disp.shape[0] if n is None else n
    rows = disp.shape[1] if rows is None else rows
    cols = disp.shape[2] if cols is None else cols
    cams = cameras(30.0)[:2]
    R = np.ascontiguousarray(np.stack([c[0] for c in cams]) if R is None else R, np.float64)
    t = np.ascontiguousarray(np.stack([c[1] for c in cams]) if t is None else t, np.float64)
    K = np.ascontiguousarray(intrinsics(f, disp.shape[1], disp.shape[2]) if K is None else K, np.float64)
    nv = len(R) if n_views is None else n_views
    q = np.ascontiguousarray(qs, np.int32)
    m = max(len(q), 1) * max(n, 1)
    out = [np.full(m, SENTINEL, np.uint64), np.full(m * max(len(R), 1), SENTINEL, np.uint64), np.full(m * max(len(R), 1), SENTINEL, np.uint64)]
    DP, U64 = C.POINTER(C.c_double), C.POINTER(C.c_uint64)
    ptr = lambda a, ok=True: a.ctypes.data_as(DP if a.dtype == np.float64 else U64) if ok and a is not None else None     # noqa: E731
    rc = capi.lib.dmc_jpeg_view_rd_sweep(ctx.h, C.c_void_p(disp.ctypes.data), C.c_void_p(tex.ctypes.data), capi.MEM_HOST, n, rows, cols,
                                         q.ctypes.data_as(C.POINTER(C.c_int)), len(q), flags, C.byref(p) if p is not None else None, f,
                                         ptr(R), ptr(t), nv, ptr(K), 1, render_flags, ptr(out[0], outputs[0]), ptr(out[1], outputs[1]), ptr(out[2], outputs[2]))
    return rc, out


def test_view_sweep_argument_rules(dmc):
    from depthmapcompression_b200 import capi
    disp, tex = mixed_batch(24, 32)
    good = params(dmc)
    untouched = lambda out: all(np.all(o == SENTINEL) for o in out)     # noqa: E731
    rc, out = sweep(dmc, disp, tex, (50,), good)
    assert rc == capi.DMC_OK and not untouched(out)
    for qs in ((), (-1,), (101,), (50, 101), (50, -5, 60)):
        rc, out = sweep(dmc, disp, tex, qs, good)
        assert rc == capi.DMC_ERR_ARG and untouched(out), qs
    for flags in (2, 3, -1, 1 << 30):
        rc, out = sweep(dmc, disp, tex, (50,), good, flags=flags)
        assert rc == capi.DMC_ERR_ARG and untouched(out), flags
    for rf in (2, 3, -1, 1 << 30):
        rc, out = sweep(dmc, disp, tex, (50,), good, render_flags=rf)
        assert rc == capi.DMC_ERR_ARG and untouched(out), rf
    rc, out = sweep(dmc, disp, tex, (50,), None)
    assert rc == capi.DMC_ERR_ARG and untouched(out)
    for chain in (capi.CHAIN_DISP8U, capi.CHAIN_DEPTH16U, capi.CHAIN_DISP32F, 4, -1):
        rc, out = sweep(dmc, disp, tex, (50,), params(dmc, chain=chain))
        assert rc == capi.DMC_ERR_ARG and untouched(out), chain
    for bad in ((11, 0, 1, 3, 65.0), (1, -1, 1, 3, 65.0), (1, 0, 11, 3, 65.0), (1, 0, 1, 11, 65.0)):
        rc, out = sweep(dmc, disp, tex, (50,), params(dmc, radii=bad))
        assert rc == capi.DMC_ERR_ARG and untouched(out), bad
    for method in (3, -1):                                               # the 32F chain writes nothing for these
        rc, out = sweep(dmc, disp, tex, (50,), params(dmc, brange_method=method))
        assert rc == capi.DMC_ERR_ARG and untouched(out), method
    for method in (capi.FULL_KERNEL_PAIR, capi.SEPARABLE_KERNEL):
        rc, out = sweep(dmc, disp, tex, (50,), params(dmc, brange_method=method))
        assert rc == capi.DMC_OK and not untouched(out), method
    for n_views in (0, -1):
        rc, out = sweep(dmc, disp, tex, (50,), good, n_views=n_views)
        assert rc == capi.DMC_ERR_ARG and untouched(out), n_views
    for missing in ("R", "t", "K"):
        from depthmapcompression_b200 import capi as c
        ctx = dmc.default_context()
        cams = cameras(30.0)[:2]
        arrs = {"R": np.ascontiguousarray(np.stack([x[0] for x in cams])), "t": np.ascontiguousarray(np.stack([x[1] for x in cams])),
                "K": np.ascontiguousarray(intrinsics(20.0, 24, 32))}
        arrs[missing] = None
        out = [np.full(len(disp) * 2, SENTINEL, np.uint64) for _ in range(3)]
        DP, U64 = C.POINTER(C.c_double), C.POINTER(C.c_uint64)
        q = np.array([50], np.int32)
        rc = c.lib.dmc_jpeg_view_rd_sweep(ctx.h, C.c_void_p(disp.ctypes.data), C.c_void_p(tex.ctypes.data), c.MEM_HOST, len(disp), 24, 32,
                                          q.ctypes.data_as(C.POINTER(C.c_int)), 1, 0, C.byref(good), 20.0,
                                          *[arrs[k].ctypes.data_as(DP) if arrs[k] is not None else None for k in ("R", "t")], 2,
                                          arrs["K"].ctypes.data_as(DP) if arrs["K"] is not None else None, 1, 0, *[o.ctypes.data_as(U64) for o in out])
        assert rc == capi.DMC_ERR_ARG and untouched(out), missing
    rc, out = sweep(dmc, disp, tex, (50,), good, n=0)
    assert rc == capi.DMC_OK and untouched(out)
    for rows, cols in ((0, 32), (24, 0), (65536, 8), (8, 65536), (-3, 32), (23171, 23171)):     # encoder sizes; the renderer's 2^29
        rc, out = sweep(dmc, disp, tex, (50,), good, rows=rows, cols=cols, n=0)
        assert rc == capi.DMC_ERR_SIZE and untouched(out), (rows, cols)
    rc, out = sweep(dmc, disp, tex, (50,), good, n=-1)
    assert rc == capi.DMC_ERR_SIZE and untouched(out)
    for k in range(3):
        rc, out = sweep(dmc, disp, tex, (50,), good, outputs=tuple(j != k for j in range(3)))
        assert rc == capi.DMC_ERR_SIZE and untouched(out), k
    with pytest.raises(dmc.DmcError):
        dmc.jpegViewRateDistortion(disp, tex, (), good, 20.0, np.eye(3), np.zeros(3), intrinsics(20.0, 24, 32))
    with pytest.raises(dmc.DmcError):
        dmc.jpegViewRateDistortion(disp, tex[:2], (50,), good, 20.0, np.eye(3), np.zeros(3), intrinsics(20.0, 24, 32))
