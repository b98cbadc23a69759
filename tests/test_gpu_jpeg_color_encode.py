"""The colour JPEG encoder on the GPU (dmc_jpeg_encode_color_batch / dmc_jpeg_degrade_color_batch, jpegEncodeColorBatch /
degradeJPEGColor): every stream must equal cv2.imencode(img, [IMWRITE_JPEG_QUALITY, q, IMWRITE_JPEG_SAMPLING_FACTOR, s])
byte for byte over the emulation's matrix (sizes, contents, the five samplings, qualities), from and to host and device
memory, in large batches and across groups; the round trip must equal cv2.imdecode of those streams, in place too; the
streams must feed jpegDecodeColorBatch and the round trip renderViewBatch; and bad arguments are refused with nothing
written."""
import ctypes as C

import numpy as np
import pytest

from _util import assert_bits_equal

cv2 = pytest.importorskip("cv2")
import _jpeg_color_cases as cases  # noqa: E402

pytestmark = pytest.mark.gpu

SIZES = cases.SIZES + [(1080, 1920), (1081, 1919), (3, 10000)]
KINDS = cases.KINDS + ("textured",)
QUALITIES = (0, 1, 5, 25, 50, 75, 90, 100)


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def image(kind, H, W):
    return cases.textured(H, W, seed=H + W) if kind == "textured" else cases.image(kind, H, W)


def enc(img, q, sampling="420"):
    return bytes(cases.encode(img, q, sampling))


def roundtrip(stream):
    return cv2.imdecode(np.frombuffer(stream, np.uint8), cv2.IMREAD_COLOR)


def streams_of(blob, offsets):
    return [bytes(blob[int(offsets[i]):int(offsets[i + 1])]) for i in range(len(offsets) - 1)]


@pytest.mark.parametrize("sampling", list(cases.SAMPLINGS))
@pytest.mark.parametrize("shape", SIZES)
def test_encode_matches_cv2(dmc, shape, sampling):
    """One batch per size of every content, at every quality (large frames: q0, 50, 90, 100)."""
    H, W = shape
    frames = np.stack([image(k, H, W) for k in KINDS])
    for q in (QUALITIES if H * W < 1 << 20 else (0, 50, 90, 100)):
        blob, offsets = dmc.jpegEncodeColorBatch(frames, q, sampling)
        assert offsets[0] == 0 and len(blob) == offsets[-1]
        for i, s in enumerate(streams_of(blob, offsets)):
            assert s == enc(frames[i], q, sampling), "%s %s %s q%d" % (shape, KINDS[i], sampling, q)


def test_every_quality_and_cv2_sampling_constants(dmc):
    img = cases.textured(37, 53, seed=12)
    for q in range(0, 101):
        blob, _ = dmc.jpegEncodeColorBatch(img, q)
        assert bytes(blob) == enc(img, q), "q%d" % q
    for name, value in cases.SAMPLINGS.items():
        assert bytes(dmc.jpegEncodeColorBatch(img, 70, value)[0]) == enc(img, 70, name)
    ok, default = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 70])
    assert bytes(dmc.jpegEncodeColorBatch(img, 70)[0]) == bytes(default)


def test_device_src_and_blob_and_empty_batch(dmc):
    import torch
    H, W = 131, 150
    frames = np.stack([image(k, H, W) for k in KINDS])
    n = len(frames)
    for sampling in ("420", "411"):
        want = [enc(f, 75, sampling) for f in frames]
        d_src = torch.from_numpy(frames).cuda()
        cap = n * dmc.jpegEncodeColorBound(H, W, sampling)
        d_blob = torch.zeros(cap, dtype=torch.uint8, device="cuda")
        _, offsets = dmc.jpegEncodeColorBatch((d_src.data_ptr(), n, H, W), 75, sampling, blob=(d_blob.data_ptr(), cap))
        assert streams_of(d_blob.cpu().numpy(), offsets) == want
        _, offsets = dmc.jpegEncodeColorBatch(frames, 75, sampling, blob=(d_blob.data_ptr(), cap))            # host src, device blob
        assert streams_of(d_blob.cpu().numpy(), offsets) == want
        blob, offsets = dmc.jpegEncodeColorBatch((d_src.data_ptr(), n, H, W), 75, sampling)                   # device src, host blob
        assert streams_of(blob, offsets) == want
    blob, offsets = dmc.jpegEncodeColorBatch(np.zeros((0, H, W, 3), np.uint8), 75)
    assert len(blob) == 0 and list(offsets) == [0]
    dec, nbytes = dmc.degradeJPEGColor(np.zeros((0, H, W, 3), np.uint8), 75)
    assert dec.shape == (0, H, W, 3) and nbytes.shape == (0,)


def test_capacity_too_small(dmc):
    import torch
    from depthmapcompression_b200 import capi
    H, W = 64, 641
    frames = np.stack([image(k, H, W) for k in KINDS])
    n = len(frames)
    need = sum(len(enc(f, 90)) for f in frames)
    ctx = dmc.default_context()
    offsets = np.zeros(n + 1, np.uint64)
    for cap in (0, 100, need - 1):
        host = np.full(need + 64, 0xA7, np.uint8)
        rc = capi.lib.dmc_jpeg_encode_color_batch(ctx.h, C.c_void_p(frames.ctypes.data), capi.MEM_HOST, n, H, W, 90, capi.DMC_JPEG_SAMPLING_420,
                                                  C.c_void_p(host.ctypes.data), capi.MEM_HOST, cap, offsets.ctypes.data_as(C.POINTER(C.c_uint64)))
        assert rc == capi.DMC_ERR_SIZE
        assert np.all(host[cap:] == 0xA7), "bytes written past the capacity %d" % cap
        dev = torch.full((need + 64,), 0xA7, dtype=torch.uint8, device="cuda")
        rc = capi.lib.dmc_jpeg_encode_color_batch(ctx.h, C.c_void_p(frames.ctypes.data), capi.MEM_HOST, n, H, W, 90, capi.DMC_JPEG_SAMPLING_420,
                                                  C.c_void_p(dev.data_ptr()), capi.MEM_DEVICE, cap, offsets.ctypes.data_as(C.POINTER(C.c_uint64)))
        assert rc == capi.DMC_ERR_SIZE
        assert bool((dev[cap:] == 0xA7).all()), "device bytes written past the capacity %d" % cap
    host = np.zeros(need, np.uint8)
    rc = capi.lib.dmc_jpeg_encode_color_batch(ctx.h, C.c_void_p(frames.ctypes.data), capi.MEM_HOST, n, H, W, 90, capi.DMC_JPEG_SAMPLING_420,
                                              C.c_void_p(host.ctypes.data), capi.MEM_HOST, need, offsets.ctypes.data_as(C.POINTER(C.c_uint64)))
    assert rc == capi.DMC_OK and int(offsets[-1]) == need


def test_batch_200_frames_1080p(dmc):
    """200 distinct 1080p frames: about 85 frames fit the 4 GB group budget at 4:2:0, so the batch spans three groups."""
    H, W, N = 1080, 1920, 200
    base = cases.textured(H, W, seed=5)
    frames = np.stack([np.roll(base, (3 * f, 7 * f), axis=(0, 1)) for f in range(N)])
    frames[::9] = np.random.RandomState(6).randint(0, 256, (H, W, 3), dtype=np.uint8)
    blob, offsets = dmc.jpegEncodeColorBatch(frames, 80)
    streams = streams_of(blob, offsets)
    for f in range(N):
        assert streams[f] == enc(frames[f], 80), "frame %d" % f
    dec, nbytes = dmc.degradeJPEGColor(frames, 80)
    assert [int(x) for x in nbytes] == [len(s) for s in streams]
    for f in (0, 1, 9, 84, 85, 86, 170, 199):
        assert_bits_equal(dec[f], roundtrip(streams[f]), "degraded frame %d" % f)


def test_batch_spanning_two_groups_of_small_frames(dmc):
    """A group holds at most 2048 frames; 2100 distinct small frames take two."""
    rs = np.random.RandomState(9)
    frames = rs.randint(0, 256, (2100, 9, 14, 3)).astype(np.uint8)
    blob, offsets = dmc.jpegEncodeColorBatch(frames, 60, "422")
    streams = streams_of(blob, offsets)
    assert all(streams[f] == enc(frames[f], 60, "422") for f in range(len(frames)))
    dec, nbytes = dmc.degradeJPEGColor(frames, 60, "422")
    assert [int(x) for x in nbytes] == [len(s) for s in streams]
    assert_bits_equal(dec, np.stack([roundtrip(s) for s in streams]), "2100 degraded frames")


def test_streams_feed_the_colour_decoder(dmc):
    import torch
    for shape in ((61, 83), (480, 640), (1081, 1919)):
        H, W = shape
        frames = np.stack([image(k, H, W) for k in KINDS])
        streams = []
        for sampling in cases.SAMPLINGS:
            blob, offsets = dmc.jpegEncodeColorBatch(frames, 85, sampling)
            streams += streams_of(blob, offsets)
            got = dmc.jpegDecodeColorBatch((blob, offsets), H, W)
            assert_bits_equal(got, np.stack([roundtrip(s) for s in streams_of(blob, offsets)]), "%s %s" % (shape, sampling))
        out = torch.empty((len(streams), H, W, 3), dtype=torch.uint8, device="cuda")
        dmc.jpegDecodeColorBatch(streams, H, W, dst=out.data_ptr())          # every sampling in one batch, device dst
        assert_bits_equal(out.cpu().numpy(), np.stack([roundtrip(s) for s in streams]), "%s mixed samplings" % (shape,))


@pytest.mark.parametrize("sampling", list(cases.SAMPLINGS))
def test_degrade_matches_roundtrip(dmc, sampling):
    import torch
    for shape in ((1, 1), (2, 3), (15, 17), (61, 83), (480, 640), (3, 10000)):
        H, W = shape
        frames = np.stack([image(k, H, W) for k in KINDS])
        for q in (1, 50, 80, 100):
            dec, nbytes = dmc.degradeJPEGColor(frames, q, sampling)
            for i, f in enumerate(frames):
                s = enc(f, q, sampling)
                assert int(nbytes[i]) == len(s)
                assert_bits_equal(dec[i], roundtrip(s), "%s %s frame %d q%d" % (shape, sampling, i, q))
    H, W = 480, 640
    frames = np.stack([image(k, H, W) for k in KINDS])
    n = len(frames)
    want = [enc(f, 50, sampling) for f in frames]
    d_src = torch.from_numpy(frames).cuda()
    d_dst = torch.empty_like(d_src)
    _, nbytes = dmc.degradeJPEGColor((d_src.data_ptr(), n, H, W), 50, sampling, dst=d_dst.data_ptr())
    assert [int(x) for x in nbytes] == [len(s) for s in want]
    assert_bits_equal(d_dst.cpu().numpy(), np.stack([roundtrip(s) for s in want]), "device round trip")
    dmc.degradeJPEGColor((d_src.data_ptr(), n, H, W), 50, sampling, dst=d_src.data_ptr())           # in place, device
    assert_bits_equal(d_src.cpu().numpy(), d_dst.cpu().numpy(), "in-place device round trip")
    host = frames.copy()
    dmc.degradeJPEGColor(host, 50, sampling, dst=host)                                               # in place, host
    assert_bits_equal(host, d_dst.cpu().numpy(), "in-place host round trip")
    one, nb = dmc.degradeJPEGColor(frames[0], 50, sampling)
    assert nb == len(want[0]) and np.array_equal(one, d_dst[0].cpu().numpy())


def test_degraded_textures_feed_render_view_batch(dmc):
    """Textures degraded on the device and passed to renderViewBatch as its texture tuple give the views of the same call
    with textures that went through cv2.imencode / cv2.imdecode."""
    import torch
    from oracle.oracle_py import synth_disp
    from test_gpu_view_rd_sweep import cameras, intrinsics
    H, W, n, f = 240, 320, 6, 300.0
    disp = np.stack([synth_disp(H, W, 20 + i) for i in range(n)])
    pfs = dmc.PostFilterSet()
    depth = np.stack([pfs.filterDisp8U2Depth32F(x, None, 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0) for x in disp])
    tex_src = np.stack([cases.textured(H, W, i) for i in range(n)])
    cams = cameras()
    R = np.stack([c[0] for c in cams]); t = np.stack([c[1] for c in cams]); K = intrinsics(f, H, W)
    want = dmc.renderViewBatch(depth, np.stack([roundtrip(enc(x, 85)) for x in tex_src]), f, R, t, K)
    tex = torch.from_numpy(tex_src).cuda()
    dmc.degradeJPEGColor((tex.data_ptr(), n, H, W), 85, dst=tex.data_ptr())
    d = torch.from_numpy(depth).cuda()
    out = torch.full((len(cams), n, H, W, 3), 0xA5, dtype=torch.uint8, device="cuda")
    dmc.renderViewBatch((d.data_ptr(), n, H, W, np.float32), (tex.data_ptr(), n, H, W), f, R, t, K, dst=out.data_ptr())
    dmc.default_context().synchronize()
    assert_bits_equal(out.cpu().numpy(), want, "views from device-degraded textures")


def test_argument_rules(dmc):
    """Bad sampling, quality, mem, size and NULL arguments are refused, and nothing is written."""
    from depthmapcompression_b200 import capi
    lib, ctx = capi.lib, dmc.default_context()
    H, W = 16, 24
    src = cases.textured(H, W)[None].copy()
    blob = np.full(1 << 16, 0xA7, np.uint8)
    dst = np.full_like(src, 0xA7)
    offsets = np.full(2, 7, np.uint64)
    nbytes = np.full(1, 7, np.uint64)
    op = offsets.ctypes.data_as(C.POINTER(C.c_uint64))
    bp = nbytes.ctypes.data_as(C.POINTER(C.c_uint64))
    S, D, B = C.c_void_p(src.ctypes.data), C.c_void_p(dst.ctypes.data), C.c_void_p(blob.ctypes.data)
    H0, S420 = capi.MEM_HOST, capi.DMC_JPEG_SAMPLING_420
    cases_ = [  # (expected code, encode call, degrade call)
        (capi.DMC_ERR_ARG, (S, H0, 1, H, W, 50, 0x222222, B, H0, blob.size, op), (S, D, 1, H, W, 50, 0x222222, H0, bp)),
        (capi.DMC_ERR_ARG, (S, H0, 1, H, W, 50, 0, B, H0, blob.size, op), (S, D, 1, H, W, 50, 0, H0, bp)),
        (capi.DMC_ERR_ARG, (S, H0, 1, H, W, -1, S420, B, H0, blob.size, op), (S, D, 1, H, W, -1, S420, H0, bp)),
        (capi.DMC_ERR_ARG, (S, H0, 1, H, W, 101, S420, B, H0, blob.size, op), (S, D, 1, H, W, 101, S420, H0, bp)),
        (capi.DMC_ERR_ARG, (S, 2, 1, H, W, 50, S420, B, H0, blob.size, op), (S, D, 1, H, W, 50, S420, 2, bp)),
        (capi.DMC_ERR_ARG, (S, H0, 1, H, W, 50, S420, B, 7, blob.size, op), (S, D, 1, H, W, 50, S420, -1, bp)),
        (capi.DMC_ERR_SIZE, (S, H0, 1, 0, W, 50, S420, B, H0, blob.size, op), (S, D, 1, 0, W, 50, S420, H0, bp)),
        (capi.DMC_ERR_SIZE, (S, H0, 1, H, 65536, 50, S420, B, H0, blob.size, op), (S, D, 1, H, 65536, 50, S420, H0, bp)),
        (capi.DMC_ERR_SIZE, (S, H0, 1, 20000, 20000, 50, S420, B, H0, blob.size, op), (S, D, 1, 20000, 20000, 50, S420, H0, bp)),
        (capi.DMC_ERR_SIZE, (None, H0, 1, H, W, 50, S420, B, H0, blob.size, op), (None, D, 1, H, W, 50, S420, H0, bp)),
        (capi.DMC_ERR_SIZE, (S, H0, 1, H, W, 50, S420, None, H0, blob.size, op), (S, None, 1, H, W, 50, S420, H0, bp)),
        (capi.DMC_ERR_SIZE, (S, H0, 1, H, W, 50, S420, B, H0, blob.size, None), (S, D, -1, H, W, 50, S420, H0, bp)),
    ]
    for code, e_args, d_args in cases_:
        assert lib.dmc_jpeg_encode_color_batch(ctx.h, *e_args) == code, e_args
        assert lib.dmc_jpeg_degrade_color_batch(ctx.h, *d_args) == code, d_args
        assert np.all(blob == 0xA7) and np.all(dst == 0xA7) and list(offsets) == [7, 7] and list(nbytes) == [7], "written on %r" % (e_args,)
    assert lib.dmc_jpeg_encode_color_batch(None, S, H0, 1, H, W, 50, S420, B, H0, blob.size, op) == capi.DMC_ERR_ARG
    assert lib.dmc_jpeg_degrade_color_batch(None, S, D, 1, H, W, 50, S420, H0, bp) == capi.DMC_ERR_ARG
    b = C.c_uint64(7)
    assert lib.dmc_jpeg_encode_color_bound(H, W, 0x222222, C.byref(b)) == capi.DMC_ERR_ARG and b.value == 7
    assert lib.dmc_jpeg_encode_color_bound(0, W, S420, C.byref(b)) == capi.DMC_ERR_SIZE and b.value == 7
    assert lib.dmc_jpeg_encode_color_bound(H, W, S420, None) == capi.DMC_ERR_ARG
    with pytest.raises(dmc.DmcError):
        dmc.jpegEncodeColorBatch(src, 50, "423")
    with pytest.raises(dmc.DmcError):
        dmc.jpegEncodeColorBatch(src[..., 0], 50)              # 8UC1 frames belong to the gray encoder
    with pytest.raises(dmc.DmcError):
        dmc.degradeJPEGColor((0, 1, H, W), 50, dst=None)       # device frames need a device dst
