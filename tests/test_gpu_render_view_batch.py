"""Views of frame batches (dmc_render_view_batch, renderViewBatch): views[v, i] must equal, bit for bit, the single-frame
calls reprojectXYZ -> projectImagefromXYZ -> fillSmallHole (in place) on frame i with camera v, and the port's renderer,
for the four depth types, isSub on and off, exact division and the rcp table, one and three cameras, groups, host and
device memory."""
import ctypes as C

import numpy as np
import pytest

from test_pointcloud import intel_host
from test_gpu_view_rd_sweep import cameras, intrinsics, texture_of

pytestmark = pytest.mark.gpu

FOCUS, BASELINE, AMP = 75.0, 575.0, 2.6


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def depths(dmc, dtype, n, H, W, seed):
    """n frames of one depth type: 8U and 16S/16U depths straight, 32F from the 32F chain (NaN where the disparity is 0)."""
    from oracle.oracle_py import synth_disp
    rs = np.random.RandomState(seed)
    if dtype == np.float32:
        disp = np.stack([synth_disp(H, W, seed + i) for i in range(n)])
        disp[:, ::7, ::5] = 0
        pfs = dmc.PostFilterSet()
        return np.stack([pfs.filterDisp8U2Depth32F(x, None, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0) for x in disp]), disp
    hi = 256 if dtype == np.uint8 else 3000
    d = rs.randint(1 if dtype == np.uint8 else 300, hi, (n, H, W)).astype(dtype)
    d[:, ::9, ::4] = 0
    return d, (d.astype(np.int64) % 251 + 1).astype(np.uint8)


def single_calls(dmc, depth, tex, f, R, t, K, sub, exact):
    xyz = dmc.reprojectXYZ(depth, None, f)
    return dmc.fillSmallHole(dmc.projectImagefromXYZ(tex, None, xyz, R, t, K, isSub=sub, exact_divide=exact))


def port_view(port, depth, tex, f, R, t, K, sub, rcp):
    return port.fill_small_hole(port.project_image(tex, port.reproject_xyz(depth, f), R, t, K, sub, rcp=rcp)[0])


def device_views(dmc, depth, tex, f, R, t, K, sub, exact):
    import torch
    n, H, W = depth.shape
    d = torch.from_numpy(depth.view(np.int16) if depth.dtype == np.uint16 else depth).cuda()
    x = torch.from_numpy(tex).cuda()
    out = torch.full((len(R), n, H, W, 3), 0xA5, dtype=torch.uint8, device="cuda")
    dmc.renderViewBatch((d.data_ptr(), n, H, W, depth.dtype), (x.data_ptr(), n, H, W), f, R, t, K, isSub=sub, exact_divide=exact, dst=out.data_ptr())
    dmc.default_context().synchronize()
    return out.cpu().numpy()


def check(dmc, port, depth, tex, f, cams, sub, exact, frames=None, port_frames=None):
    n, H, W = depth.shape
    K = intrinsics(f, H, W)
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    host = dmc.renderViewBatch(depth, tex, f, R, t, K, isSub=sub, exact_divide=exact)
    assert host.shape == (len(cams), n, H, W, 3)
    assert np.array_equal(host, device_views(dmc, depth, tex, f, R, t, K, sub, exact)), (depth.dtype, sub, exact)
    for i in (range(n) if frames is None else frames):
        for v, (Rv, tv) in enumerate(cams):
            assert np.array_equal(host[v, i], single_calls(dmc, depth[i], tex[i], f, Rv, tv, K, sub, exact)), (depth.dtype, sub, exact, i, v)
    for i in (range(n) if port_frames is None else port_frames):
        for v, (Rv, tv) in enumerate(cams):
            assert np.array_equal(host[v, i], port_view(port, depth[i], tex[i], f, Rv, tv, K, sub, not exact)), (depth.dtype, sub, exact, i, v)
    return host


@pytest.mark.parametrize("dtype", [np.uint8, np.int16, np.uint16, np.float32])
def test_depth_types_equal_single_calls_and_port(dmc, port, dtype):
    f = 20.0 if dtype == np.uint8 else 500.0
    for H, W in ((3, 3), (61, 83)):
        for n in (1, 3):
            depth, gray = depths(dmc, dtype, n, H, W, H + n)
            tex = np.stack([texture_of(g) for g in gray])
            for exact in [True] + ([False] if intel_host() else []):
                for sub in (False, True):
                    for cams in (cameras(30.0)[:1], cameras(30.0)):
                        check(dmc, port, depth, tex, f, cams, sub, exact)


def test_chain_batch_depth32f_output_as_it_is(dmc, port):
    """dmc_chain_batch's DMC_CHAIN_DEPTH32F output goes into the render unchanged."""
    from depthmapcompression_b200 import capi
    from oracle.oracle_py import synth_disp
    n, H, W = 3, 120, 160
    disp = np.stack([synth_disp(H, W, 30 + i) for i in range(n)]); disp[:, 40:60, 50:90] = 0
    depth = np.zeros((n, H, W), np.float32)
    p = dmc.filters.chain_params(capi.CHAIN_DEPTH32F, 1, 0, 1, 3, 65.0, focus=FOCUS, baseline=BASELINE, amp=AMP)
    dmc.default_context().chain_batch(disp, depth, n, H, W, p)
    check(dmc, port, depth, np.stack([texture_of(d) for d in disp]), 150.0, cameras(40.0), True, True)


def test_1080p_batches_across_groups(dmc, port, monkeypatch):
    import bench
    base = bench.base_frame()
    H, W = base.shape
    disp = np.stack([bench.frame_np(base, 7 * i) for i in range(40)])
    tex = np.stack([texture_of(d) for d in disp])
    pfs = dmc.PostFilterSet()
    depth = np.stack([pfs.filterDisp8U2Depth32F(x, None, FOCUS, BASELINE, AMP, 1, 0, 1, 3, 65.0) for x in disp])
    f, cams = 1100.0, cameras()
    for n in (1, 3):
        check(dmc, port, depth[:n], tex[:n], f, cams, True, True, port_frames=[n - 1])
    # the default groups (4 GiB) split 40 1080p frames in two; 1 GiB groups split them in more
    full = check(dmc, port, depth, tex, f, cams, True, True, frames=[0, 1, 20, 21, 22, 39], port_frames=[21])
    monkeypatch.setenv("DMC_GROUP_MB", "1024")
    K = intrinsics(f, H, W)
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams])
    assert np.array_equal(dmc.renderViewBatch(depth, tex, f, R, t, K, exact_divide=True), full)
    assert np.array_equal(device_views(dmc, depth, tex, f, R, t, K, True, True), full)


def test_argument_rules(dmc):
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    n, H, W = 2, 12, 16
    depth = np.full((n, H, W), 900, np.uint16)
    tex = np.full((n, H, W, 3), 77, np.uint8)
    cams = cameras(30.0)[:2]
    R = np.ascontiguousarray(np.stack([c[0] for c in cams])); t = np.ascontiguousarray(np.stack([c[1] for c in cams]))
    K = np.ascontiguousarray(intrinsics(100.0, H, W))
    out = np.full((2, n, H, W, 3), 0xA5, np.uint8)
    DP = C.POINTER(C.c_double)

    def call(d=depth.ctypes.data, dt=capi.CV_16U, x=tex.ctypes.data, mem=capi.MEM_HOST, nf=n, rows=H, cols=W, Rp=R, tp=t, nv=2, Kp=K, flags=0, o=out.ctypes.data):
        ptr = lambda a: a.ctypes.data_as(DP) if a is not None else None     # noqa: E731
        return capi.lib.dmc_render_view_batch(ctx.h, C.c_void_p(d), dt, C.c_void_p(x), mem, nf, rows, cols, 100.0, ptr(Rp), ptr(tp), nv, ptr(Kp), 1, flags, C.c_void_p(o))

    untouched = lambda: np.all(out == 0xA5)     # noqa: E731
    assert call() == capi.DMC_OK and not untouched()
    out[:] = 0xA5
    for nv in (0, -1):
        assert call(nv=nv) == capi.DMC_ERR_ARG and untouched(), nv
    for miss in ("Rp", "tp", "Kp"):
        assert call(**{miss: None}) == capi.DMC_ERR_ARG and untouched(), miss
    for flags in (2, 3, -1, 1 << 30):
        assert call(flags=flags) == capi.DMC_ERR_ARG and untouched(), flags
    for dt in (capi.CV_64F, 1, 4, 7, capi.CV_8U + 16, -1):
        assert call(dt=dt) == capi.DMC_ERR_ARG and untouched(), dt
    for mem in (2, -1):
        assert call(mem=mem) == capi.DMC_ERR_ARG and untouched(), mem
    # views overlapping the depth or the texture
    buf = np.zeros(out.nbytes + tex.nbytes + depth.nbytes, np.uint8)
    buf[:depth.nbytes] = depth.view(np.uint8).ravel()
    buf[depth.nbytes:depth.nbytes + tex.nbytes] = tex.ravel()
    keep = buf.copy()
    b0 = buf.ctypes.data
    for o in (b0, b0 + depth.nbytes - 1, b0 + depth.nbytes + 5, b0 + depth.nbytes + tex.nbytes - 1):
        assert call(d=b0, x=b0 + depth.nbytes, o=o) == capi.DMC_ERR_ARG and np.array_equal(buf, keep), o - b0
    assert call(d=b0, x=b0 + depth.nbytes, o=b0 + depth.nbytes + tex.nbytes) == capi.DMC_OK
    for bad in (dict(nf=-1), dict(rows=0), dict(cols=-1), dict(o=0), dict(rows=23171, cols=23171, nf=0)):
        assert call(**bad) == capi.DMC_ERR_SIZE and untouched(), bad
    assert call(nf=0) == capi.DMC_OK and untouched()
    with pytest.raises(dmc.DmcError):
        dmc.renderViewBatch(depth.astype(np.float64), tex, 100.0, R, t, K)
    with pytest.raises(dmc.DmcError):
        dmc.renderViewBatch(depth, tex[:1], 100.0, R, t, K)
    with pytest.raises(dmc.DmcError):
        dmc.renderViewBatch(depth, tex, 100.0, R, t[:1], K)
