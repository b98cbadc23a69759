"""SURVEY.md 8f-5, the encoder: the GPU JPEG encoder (csrc/dmc_jpeg_enc.cu) must write the very bytes cv2.imencode writes
for an 8UC1 image at the same quality, and degradeJPEG must equal cv2.imdecode(cv2.imencode(.)) -- the JPEG round trip
of the reference's pointcloudTest / simpleTest loops -- with the stream sizes as its bitrate."""
import numpy as np
import pytest

from _util import assert_bits_equal, load_png

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu

SIZES = [(1, 1), (7, 9), (8, 8), (131, 150), (64, 641), (480, 640), (1080, 1920), (3, 10000)]
QUALITIES = (1, 5, 25, 50, 75, 80, 95, 100)


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def enc(img, q):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return bytes(buf)


def kinds(H, W, seed=3):
    from oracle.oracle_py import synth_disp, degrade_blocks
    rs = np.random.RandomState(seed)
    out = [rs.randint(0, 256, (H, W)).astype(np.uint8), np.zeros((H, W), np.uint8), np.full((H, W), 255, np.uint8)]
    if H > 16 and W > 16:
        out.append(degrade_blocks(synth_disp(H, W, seed), seed))
    return np.stack(out)


def streams_of(blob, offsets):
    return [bytes(blob[int(offsets[i]):int(offsets[i + 1])]) for i in range(len(offsets) - 1)]


@pytest.mark.parametrize("shape", SIZES)
def test_encode_matches_cv2(dmc, shape):
    frames = kinds(*shape)
    for q in QUALITIES:
        blob, offsets = dmc.jpegEncodeGrayBatch(frames, q)
        assert offsets[0] == 0 and len(blob) == offsets[-1]
        for i, s in enumerate(streams_of(blob, offsets)):
            assert s == enc(frames[i], q), "%s frame %d q%d" % (shape, i, q)


def test_every_quality_and_bad_quality(dmc):
    img = np.clip(np.random.RandomState(12).normal(120, 40, (37, 53)), 0, 255).astype(np.uint8)
    for q in range(0, 101):
        blob, offsets = dmc.jpegEncodeGrayBatch(img, q)
        assert bytes(blob) == enc(img, q), "q%d" % q
    for q in (-1, 101):
        with pytest.raises(dmc.DmcError) as e:
            dmc.jpegEncodeGrayBatch(img, q)
        assert e.value.code == -4
        with pytest.raises(dmc.DmcError):
            dmc.degradeJPEG(img, q)


def test_device_src_and_blob_and_empty_batch(dmc):
    import torch
    frames = kinds(131, 150, seed=8)
    n, H, W = frames.shape
    want = [enc(f, 75) for f in frames]
    d_src = torch.from_numpy(frames).cuda()
    cap = n * dmc.jpegEncodeBound(H, W)
    d_blob = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    ptr, offsets = dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), 75, blob=(d_blob.data_ptr(), cap))
    assert streams_of(d_blob.cpu().numpy(), offsets) == want
    ptr, offsets = dmc.jpegEncodeGrayBatch(frames, 75, blob=(d_blob.data_ptr(), cap))          # host src, device blob
    assert streams_of(d_blob.cpu().numpy(), offsets) == want
    blob, offsets = dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), 75)                    # device src, host blob
    assert streams_of(blob, offsets) == want
    blob, offsets = dmc.jpegEncodeGrayBatch(np.zeros((0, H, W), np.uint8), 75)
    assert len(blob) == 0 and list(offsets) == [0]
    dec, nbytes = dmc.degradeJPEG(np.zeros((0, H, W), np.uint8), 75)
    assert dec.shape == (0, H, W) and nbytes.shape == (0,)


def test_capacity_too_small(dmc):
    import ctypes as C
    import torch
    from depthmapcompression_b200 import capi
    frames = kinds(64, 641, seed=4)
    n, H, W = frames.shape
    need = sum(len(enc(f, 90)) for f in frames)
    ctx = dmc.default_context()
    offsets = np.zeros(n + 1, np.uint64)
    for cap in (0, 100, need - 1):
        host = np.full(need + 64, 0xA7, np.uint8)
        rc = capi.lib.dmc_jpeg_encode_gray_batch(ctx.h, C.c_void_p(frames.ctypes.data), capi.MEM_HOST, n, H, W, 90, C.c_void_p(host.ctypes.data),
                                                 capi.MEM_HOST, cap, offsets.ctypes.data_as(C.POINTER(C.c_uint64)))
        assert rc == capi.DMC_ERR_SIZE
        assert np.all(host[cap:] == 0xA7), "bytes written past the capacity %d" % cap
        dev = torch.full((need + 64,), 0xA7, dtype=torch.uint8, device="cuda")
        rc = capi.lib.dmc_jpeg_encode_gray_batch(ctx.h, C.c_void_p(frames.ctypes.data), capi.MEM_HOST, n, H, W, 90, C.c_void_p(dev.data_ptr()),
                                                 capi.MEM_DEVICE, cap, offsets.ctypes.data_as(C.POINTER(C.c_uint64)))
        assert rc == capi.DMC_ERR_SIZE
        assert bool((dev[cap:] == 0xA7).all()), "device bytes written past the capacity %d" % cap
    host = np.zeros(need, np.uint8)
    rc = capi.lib.dmc_jpeg_encode_gray_batch(ctx.h, C.c_void_p(frames.ctypes.data), capi.MEM_HOST, n, H, W, 90, C.c_void_p(host.ctypes.data),
                                             capi.MEM_HOST, need, offsets.ctypes.data_as(C.POINTER(C.c_uint64)))
    assert rc == capi.DMC_OK and int(offsets[-1]) == need
    with pytest.raises(dmc.DmcError):
        dmc.jpegEncodeBound(0, 5)
    with pytest.raises(dmc.DmcError):
        dmc.jpegEncodeBound(20000, 20000)            # worst case above 256 MB


def test_batch_200_frames_1080p(dmc):
    from oracle.oracle_py import synth_disp, degrade_blocks
    H, W, N = 1080, 1920, 200
    rs = np.random.RandomState(5)
    base = [degrade_blocks(synth_disp(H, W, 300 + f, shift=(f, 2 * f)), f) for f in range(4)]
    base.append(rs.randint(0, 256, (H, W)).astype(np.uint8))
    frames = np.stack([base[f % len(base)] for f in range(N)])
    blob, offsets = dmc.jpegEncodeGrayBatch(frames, 80)
    streams = streams_of(blob, offsets)
    want = {i: enc(base[i], 80) for i in range(len(base))}
    for f in range(N):
        assert streams[f] == want[f % len(base)], "frame %d" % f
    dec, nbytes = dmc.degradeJPEG(frames, 80)
    for f in (0, 1, 4, 99, 163, 199):
        assert_bits_equal(dec[f], cv2.imdecode(np.frombuffer(want[f % len(base)], np.uint8), 0), "degraded frame %d" % f)
    assert [int(x) for x in nbytes] == [len(s) for s in streams]


def test_degrade_matches_roundtrip(dmc):
    import torch
    for shape in ((480, 640), (131, 150), (7, 9), (1, 1), (3, 10000)):
        frames = kinds(*shape, seed=6)
        for q in (1, 50, 80, 100):
            dec, nbytes = dmc.degradeJPEG(frames, q)
            for i, f in enumerate(frames):
                s = enc(f, q)
                assert int(nbytes[i]) == len(s)
                assert_bits_equal(dec[i], cv2.imdecode(np.frombuffer(s, np.uint8), 0), "%s frame %d q%d" % (shape, i, q))
    frames = kinds(480, 640, seed=7)
    n, H, W = frames.shape
    d_src = torch.from_numpy(frames).cuda()
    d_dst = torch.empty_like(d_src)
    _, nbytes = dmc.degradeJPEG((d_src.data_ptr(), n, H, W), 50, dst=d_dst.data_ptr())
    want = [enc(f, 50) for f in frames]
    assert [int(x) for x in nbytes] == [len(s) for s in want]
    for i in range(n):
        assert_bits_equal(d_dst[i].cpu().numpy(), cv2.imdecode(np.frombuffer(want[i], np.uint8), 0), "device frame %d" % i)
    dmc.degradeJPEG((d_src.data_ptr(), n, H, W), 50, dst=d_src.data_ptr())           # in place
    assert_bits_equal(d_src.cpu().numpy(), d_dst.cpu().numpy(), "in-place degrade")
    one, nb = dmc.degradeJPEG(frames[0], 50)
    assert nb == len(want[0]) and np.array_equal(one, d_dst[0].cpu().numpy())


def test_encoder_feeds_decoder_and_chain(dmc, port):
    """pointcloudTest / simpleTest from the encoder on: GPU encode -> GPU decode -> PostFilterSet()(2,1,3,5,10)."""
    from depthmapcompression_b200.filters import chain_params
    from depthmapcompression_b200 import capi
    golden = [load_png(n) for n in ("kinect_meeting_q50.png", "kinect_desk_q50.png", "x264_depth_y.png")]
    H, W = golden[0].shape
    frames = np.stack(golden * 4)
    for q in (50, 80):
        blob, offsets = dmc.jpegEncodeGrayBatch(frames, q)
        streams = streams_of(blob, offsets)
        for i, g in enumerate(golden):
            assert streams[i] == enc(g, q), "golden frame %d q%d" % (i, q)
        dec = dmc.jpegDecodeGrayBatch((blob, offsets), H, W)
        deg, _ = dmc.degradeJPEG(frames, q)
        assert_bits_equal(dec, deg, "decode(encode) vs degradeJPEG q%d" % q)
        out = np.zeros_like(frames)
        dmc.default_context().chain_batch_jpeg((blob, offsets), H, W, out, chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10))
        for i in (0, 1, 2, 11):
            ref_dec = cv2.imdecode(np.frombuffer(streams[i], np.uint8), 0)
            assert_bits_equal(dec[i], ref_dec, "decoded frame %d q%d" % (i, q))
            assert_bits_equal(out[i], port.post_filter_set(ref_dec, 2, 1, 3, 5, 10), "chain on frame %d q%d" % (i, q))
