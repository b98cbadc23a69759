"""The colour JPEG decoder on the GPU (dmc_jpeg_decode_color_batch, jpegDecodeColorBatch): every frame must equal
cv2.imdecode(buf, IMREAD_COLOR | IMREAD_IGNORE_ORIENTATION) bit for bit over the emulation's matrix (sizes, contents,
samplings, qualities, standard / optimised tables, restart intervals), into host and device memory, in mixed batches,
across groups, for one-component streams; arguments and unsupported streams are refused with a reason; and textures
decoded to the device feed renderViewBatch exactly as cv2-decoded ones do."""
import numpy as np
import pytest

from _util import assert_bits_equal

cv2 = pytest.importorskip("cv2")
import _jpeg_color_cases as cases  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def check_batch(dmc, streams, H, W, what, device=False):
    if device:
        import torch
        out = torch.full((len(streams), H, W, 3), 0xA5, dtype=torch.uint8, device="cuda")
        dmc.jpegDecodeColorBatch(streams, H, W, dst=out.data_ptr())
        got = out.cpu().numpy()
    else:
        got = dmc.jpegDecodeColorBatch(streams, H, W)
    assert got.shape == (len(streams), H, W, 3)
    for i, s in enumerate(streams):
        assert_bits_equal(got[i], cases.reference(s), "%s frame %d" % (what, i))
    return got


@pytest.mark.parametrize("size", cases.SIZES + [(480, 640)])
def test_matrix_matches_cv2(dmc, size):
    """One batch per size: every content x sampling x quality x table kind, mixed in one call."""
    H, W = size
    streams = [cases.encode(cases.image(kind, H, W), q, sampling, tables, rst=3)
               for kind in cases.KINDS for sampling in cases.SAMPLINGS for q in cases.QUALITIES for tables in cases.TABLES]
    check_batch(dmc, streams, H, W, "%dx%d" % size)


def test_every_quality_and_device_dst(dmc):
    img = cases.image("noise", 17, 23, 5)
    streams = [cases.encode(img, q, "420", tables) for q in range(0, 101) for tables in ("standard", "optimised")]
    check_batch(dmc, streams, 17, 23, "17x23 every quality", device=True)
    check_batch(dmc, streams, 17, 23, "17x23 every quality")


def test_1080p_every_sampling(dmc):
    H, W = 1080, 1920
    img = cases.textured(H, W, 3)
    streams = [cases.encode(img, q, s, t, rst=16) for s in cases.SAMPLINGS for q, t in ((50, "standard"), (80, "optimised"), (95, "restart"))]
    streams.append(cases.encode(cases.image("flat", H, W), 50, "420"))
    check_batch(dmc, streams, H, W, "1080p", device=True)


def test_mixed_batch_equals_frames_alone(dmc):
    H, W = 61, 83
    streams = [cases.encode(cases.image(k, H, W, i), 20 + 5 * i, s, t)
               for i, (k, s, t) in enumerate(zip(cases.KINDS * 4, list(cases.SAMPLINGS) * 4, cases.TABLES * 6))]
    streams.append(cases.encode(cases.image("noise", H, W)[:, :, 2].copy(), 60))
    together = dmc.jpegDecodeColorBatch(streams, H, W)
    for i, s in enumerate(streams):
        assert_bits_equal(together[i], dmc.jpegDecodeColorBatch([s], H, W)[0], "frame %d alone" % i)
        assert_bits_equal(together[i], cases.reference(s), "frame %d" % i)


def test_batch_spanning_groups(dmc):
    """More frames than one group holds (2048): frames of both groups, mixed samplings and restart streams."""
    H, W = 16, 16
    streams = [cases.encode(cases.image("noise", H, W, i % 97), 30 + i % 70, list(cases.SAMPLINGS)[i % 5], cases.TABLES[i % 3]) for i in range(2100)]
    got = check_batch(dmc, streams, H, W, "2100 frames", device=True)
    assert got.shape[0] == 2100


def test_one_component_streams(dmc):
    for H, W in ((1, 1), (15, 17), (480, 640)):
        g = cases.image("noise", H, W)[:, :, 1].copy()
        streams = [cases.encode(g, q, tables=t) for q in (5, 50, 100) for t in cases.TABLES]
        got = check_batch(dmc, streams, H, W, "gray %dx%d" % (H, W))
        for i, s in enumerate(streams):
            assert np.array_equal(got[i, :, :, 0], cv2.imdecode(s, 0))
            assert dmc.jpegProbeColor(s) == (H, W, 1)


def test_argument_rules_and_refusals(dmc):
    img = cases.image("noise", 24, 40)
    good = cases.encode(img, 75)
    assert dmc.jpegProbeColor(good) == (24, 40, 3)
    with pytest.raises(dmc.DmcError, match="frame size differs"):
        dmc.jpegDecodeColorBatch([good], 24, 41)
    for rows, cols in ((0, 40), (24, 0), (-1, 40), (70000, 40)):
        with pytest.raises(dmc.DmcError, match="bad arguments"):
            dmc.jpegDecodeColorBatch([good], rows, cols)
    with pytest.raises(dmc.DmcError):
        dmc.jpegDecodeColorBatch([good], 24, 40, dst=np.empty((1, 24, 40), np.uint8))
    blob, offsets = dmc.pack_streams([good, good])
    bad = offsets.copy(); bad[1], bad[2] = offsets[2], offsets[1]
    with pytest.raises(dmc.DmcError, match="non-decreasing"):
        dmc.jpegDecodeColorBatch((blob, bad), 24, 40)
    assert dmc.jpegDecodeColorBatch([], 24, 40).shape == (0, 24, 40, 3)
    for stream, words in cases.refused_streams(img):
        with pytest.raises(dmc.DmcError, match=words):
            dmc.jpegProbeColor(stream)
        with pytest.raises(dmc.DmcError, match="JPEG frame 1: .*" + words):
            dmc.jpegDecodeColorBatch([good, stream], 24, 40)
    for stream in cases.accepted_variants(img):
        check_batch(dmc, [stream], 24, 40, "accepted variant")
    # the gray decoder keeps refusing colour streams
    with pytest.raises(dmc.DmcError, match="grayscale"):
        dmc.jpegProbe(good)
    # the C ABI checks what the Python wrapper cannot reach: null pointers and the memory kind
    import ctypes as C
    from depthmapcompression_b200 import capi
    ctx = dmc.default_context()
    off = np.array([0, good.size], np.uint64)
    out = np.empty((24, 40, 3), np.uint8)
    assert capi.lib.dmc_jpeg_decode_color_batch(ctx.h, None, C.c_void_p(off.ctypes.data), 1, 24, 40, C.c_void_p(out.ctypes.data), capi.MEM_HOST) == capi.DMC_ERR_SIZE
    assert capi.lib.dmc_jpeg_decode_color_batch(ctx.h, C.c_void_p(good.ctypes.data), C.c_void_p(off.ctypes.data), 1, 24, 40, C.c_void_p(out.ctypes.data), 7) == capi.DMC_ERR_ARG
    assert capi.lib.dmc_jpeg_decode_color_batch(None, C.c_void_p(good.ctypes.data), C.c_void_p(off.ctypes.data), 1, 24, 40, C.c_void_p(out.ctypes.data), capi.MEM_HOST) == capi.DMC_ERR_ARG


def test_device_textures_feed_render_view_batch(dmc):
    """Colour streams decoded to the device and passed to renderViewBatch as its texture tuple give the views of the
    same call with cv2-decoded textures."""
    import torch
    from oracle.oracle_py import synth_disp
    from test_gpu_view_rd_sweep import cameras, intrinsics
    H, W, n, f = 240, 320, 6, 300.0
    disp = np.stack([synth_disp(H, W, 20 + i) for i in range(n)])
    pfs = dmc.PostFilterSet()
    depth = np.stack([pfs.filterDisp8U2Depth32F(x, None, 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0) for x in disp])
    streams = [cases.encode(cases.textured(H, W, i), 85, list(cases.SAMPLINGS)[i % 5]) for i in range(n)]
    cams = cameras()
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams]); K = intrinsics(f, H, W)
    want = dmc.renderViewBatch(depth, np.stack([cases.reference(s) for s in streams]), f, R, t, K)
    tex = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    dmc.jpegDecodeColorBatch(streams, H, W, dst=tex.data_ptr())
    d = torch.from_numpy(depth).cuda()
    out = torch.full((len(cams), n, H, W, 3), 0xA5, dtype=torch.uint8, device="cuda")
    dmc.renderViewBatch((d.data_ptr(), n, H, W, np.float32), (tex.data_ptr(), n, H, W), f, R, t, K, dst=out.data_ptr())
    dmc.default_context().synchronize()
    assert_bits_equal(out.cpu().numpy(), want, "views from device-decoded textures")
