"""The GPU JPEG encoder with optimised Huffman tables (DMC_JPEG_OPTIMIZE_HUFFMAN): every stream must equal
cv2.imencode(".jpg", f, [IMWRITE_JPEG_QUALITY, q, IMWRITE_JPEG_OPTIMIZE, 1]) byte for byte, degradeJPEG(optimize=True)
must decode to the same frames as the standard mode with the optimised stream sizes, and batches in which every frame has
its own tables must feed the decoder and the chain."""
import ctypes as C

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


def enc(img, q, optimize=True):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize)])
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
def test_encode_optimize_matches_cv2(dmc, shape):
    frames = kinds(*shape)
    for q in QUALITIES:
        blob, offsets = dmc.jpegEncodeGrayBatch(frames, q, optimize=True)
        assert offsets[0] == 0 and len(blob) == offsets[-1]
        for i, s in enumerate(streams_of(blob, offsets)):
            assert s == enc(frames[i], q), "%s frame %d q%d" % (shape, i, q)


def test_every_quality_and_fold_fixture(dmc):
    from oracle.oracle_py import synth_disp, degrade_blocks
    img = np.clip(np.random.RandomState(12).normal(120, 40, (37, 53)), 0, 255).astype(np.uint8)
    for q in range(0, 101):
        blob, _ = dmc.jpegEncodeGrayBatch(img, q, optimize=True)
        assert bytes(blob) == enc(img, q), "q%d" % q
    fixture = degrade_blocks(synth_disp(480, 640, 6), 6)          # its q100 AC table folds code lengths over 16 bits
    blob, _ = dmc.jpegEncodeGrayBatch(fixture, 100, optimize=True)
    assert bytes(blob) == enc(fixture, 100)
    dec, nbytes = dmc.degradeJPEG(fixture, 100, optimize=True)
    assert nbytes == len(blob)
    assert_bits_equal(dec, cv2.imdecode(np.frombuffer(enc(fixture, 100), np.uint8), 0), "fold fixture degrade")


def test_device_src_and_blob_and_empty_batch(dmc):
    import torch
    frames = kinds(131, 150, seed=8)
    n, H, W = frames.shape
    want = [enc(f, 75) for f in frames]
    d_src = torch.from_numpy(frames).cuda()
    cap = n * dmc.jpegEncodeBound(H, W, optimize=True)
    d_blob = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    _, offsets = dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), 75, blob=(d_blob.data_ptr(), cap), optimize=True)
    assert streams_of(d_blob.cpu().numpy(), offsets) == want
    _, offsets = dmc.jpegEncodeGrayBatch(frames, 75, blob=(d_blob.data_ptr(), cap), optimize=True)         # host src, device blob
    assert streams_of(d_blob.cpu().numpy(), offsets) == want
    blob, offsets = dmc.jpegEncodeGrayBatch((d_src.data_ptr(), n, H, W), 75, optimize=True)               # device src, host blob
    assert streams_of(blob, offsets) == want
    blob, offsets = dmc.jpegEncodeGrayBatch(np.zeros((0, H, W), np.uint8), 75, optimize=True)
    assert len(blob) == 0 and list(offsets) == [0]
    dec, nbytes = dmc.degradeJPEG(np.zeros((0, H, W), np.uint8), 75, optimize=True)
    assert dec.shape == (0, H, W) and nbytes.shape == (0,)


def test_capacity_too_small_and_bad_flags(dmc):
    import torch
    from depthmapcompression_b200 import capi
    frames = kinds(64, 641, seed=4)
    n, H, W = frames.shape
    need = sum(len(enc(f, 90)) for f in frames)
    ctx = dmc.default_context()
    offsets = np.zeros(n + 1, np.uint64)
    po = offsets.ctypes.data_as(C.POINTER(C.c_uint64))
    src = C.c_void_p(frames.ctypes.data)
    for cap in (0, 100, need - 1):
        host = np.full(need + 64, 0xA7, np.uint8)
        rc = capi.lib.dmc_jpeg_encode_gray_batch_ex(ctx.h, src, capi.MEM_HOST, n, H, W, 90, capi.JPEG_OPTIMIZE_HUFFMAN, C.c_void_p(host.ctypes.data),
                                                    capi.MEM_HOST, cap, po)
        assert rc == capi.DMC_ERR_SIZE
        assert np.all(host[cap:] == 0xA7), "bytes written past the capacity %d" % cap
        dev = torch.full((need + 64,), 0xA7, dtype=torch.uint8, device="cuda")
        rc = capi.lib.dmc_jpeg_encode_gray_batch_ex(ctx.h, src, capi.MEM_HOST, n, H, W, 90, capi.JPEG_OPTIMIZE_HUFFMAN, C.c_void_p(dev.data_ptr()),
                                                    capi.MEM_DEVICE, cap, po)
        assert rc == capi.DMC_ERR_SIZE
        assert bool((dev[cap:] == 0xA7).all()), "device bytes written past the capacity %d" % cap
    host = np.zeros(need, np.uint8)
    rc = capi.lib.dmc_jpeg_encode_gray_batch_ex(ctx.h, src, capi.MEM_HOST, n, H, W, 90, capi.JPEG_OPTIMIZE_HUFFMAN, C.c_void_p(host.ctypes.data),
                                                capi.MEM_HOST, need, po)
    assert rc == capi.DMC_OK and int(offsets[-1]) == need
    dst = np.zeros_like(frames)
    nbytes = np.zeros(n, np.uint64)
    b = C.c_uint64()
    for flags in (2, 3, -1, 1 << 30):
        assert capi.lib.dmc_jpeg_encode_gray_batch_ex(ctx.h, src, capi.MEM_HOST, n, H, W, 90, flags, C.c_void_p(host.ctypes.data),
                                                      capi.MEM_HOST, need, po) == capi.DMC_ERR_ARG
        assert capi.lib.dmc_jpeg_degrade_gray_batch_ex(ctx.h, src, C.c_void_p(dst.ctypes.data), n, H, W, 90, flags, capi.MEM_HOST,
                                                       nbytes.ctypes.data_as(C.POINTER(C.c_uint64))) == capi.DMC_ERR_ARG
        assert capi.lib.dmc_jpeg_encode_bound_ex(H, W, flags, C.byref(b)) == capi.DMC_ERR_ARG
    assert dmc.jpegEncodeBound(1080, 1920, optimize=True) == 330 + 2 * ((32400 * 1661 + 7) // 8)
    assert dmc.jpegEncodeBound(1080, 1920) == 330 + 2 * ((32400 * 1658 + 7) // 8)
    with pytest.raises(dmc.DmcError):
        dmc.jpegEncodeBound(20000, 20000, optimize=True)          # worst case above 256 MB


def test_flags_zero_ex_equals_existing_entry_points(dmc):
    from depthmapcompression_b200 import capi
    frames = kinds(480, 640, seed=11)
    n, H, W = frames.shape
    ctx = dmc.default_context()
    bound = dmc.jpegEncodeBound(H, W)
    src = C.c_void_p(frames.ctypes.data)
    for q in (0, 50, 100):
        out = []
        for ex in (False, True):
            blob = np.zeros(n * bound, np.uint8)
            offsets = np.zeros(n + 1, np.uint64)
            args = (ctx.h, src, capi.MEM_HOST, n, H, W, q) + ((0,) if ex else ()) + (C.c_void_p(blob.ctypes.data), capi.MEM_HOST, n * bound,
                                                                                      offsets.ctypes.data_as(C.POINTER(C.c_uint64)))
            fn = capi.lib.dmc_jpeg_encode_gray_batch_ex if ex else capi.lib.dmc_jpeg_encode_gray_batch
            assert fn(*args) == capi.DMC_OK
            dst = np.zeros_like(frames)
            nbytes = np.zeros(n, np.uint64)
            dargs = (ctx.h, src, C.c_void_p(dst.ctypes.data), n, H, W, q) + ((0,) if ex else ()) + (capi.MEM_HOST, nbytes.ctypes.data_as(C.POINTER(C.c_uint64)))
            fn = capi.lib.dmc_jpeg_degrade_gray_batch_ex if ex else capi.lib.dmc_jpeg_degrade_gray_batch
            assert fn(*dargs) == capi.DMC_OK
            out.append((blob[:int(offsets[-1])].tobytes(), offsets.copy(), dst, nbytes))
        assert out[0][0] == out[1][0] and np.array_equal(out[0][1], out[1][1]), "q%d streams" % q
        assert np.array_equal(out[0][2], out[1][2]) and np.array_equal(out[0][3], out[1][3]), "q%d degrade" % q
        assert streams_of(np.frombuffer(out[0][0], np.uint8), out[0][1]) == [enc(f, q, optimize=False) for f in frames]
    b0, b1 = C.c_uint64(), C.c_uint64()
    assert capi.lib.dmc_jpeg_encode_bound(H, W, C.byref(b0)) == 0 and capi.lib.dmc_jpeg_encode_bound_ex(H, W, 0, C.byref(b1)) == 0
    assert b0.value == b1.value


def test_degrade_optimize(dmc):
    import torch
    for shape in ((480, 640), (131, 150), (7, 9), (1, 1), (3, 10000)):
        frames = kinds(*shape, seed=6)
        for q in (1, 50, 80, 100):
            dec, nbytes = dmc.degradeJPEG(frames, q, optimize=True)
            std, _ = dmc.degradeJPEG(frames, q)
            assert_bits_equal(dec, std, "%s q%d optimised vs standard degrade" % (shape, q))
            for i, f in enumerate(frames):
                s = enc(f, q)
                assert int(nbytes[i]) == len(s)
                assert_bits_equal(dec[i], cv2.imdecode(np.frombuffer(s, np.uint8), 0), "%s frame %d q%d" % (shape, i, q))
    frames = kinds(480, 640, seed=7)
    n, H, W = frames.shape
    d_src = torch.from_numpy(frames).cuda()
    d_dst = torch.empty_like(d_src)
    _, nbytes = dmc.degradeJPEG((d_src.data_ptr(), n, H, W), 50, dst=d_dst.data_ptr(), optimize=True)
    want = [enc(f, 50) for f in frames]
    assert [int(x) for x in nbytes] == [len(s) for s in want]
    for i in range(n):
        assert_bits_equal(d_dst[i].cpu().numpy(), cv2.imdecode(np.frombuffer(want[i], np.uint8), 0), "device frame %d" % i)
    dmc.degradeJPEG((d_src.data_ptr(), n, H, W), 50, dst=d_src.data_ptr(), optimize=True)           # in place
    assert_bits_equal(d_src.cpu().numpy(), d_dst.cpu().numpy(), "in-place degrade")
    one, nb = dmc.degradeJPEG(frames[0], 50, optimize=True)
    assert nb == len(want[0]) and np.array_equal(one, d_dst[0].cpu().numpy())


def test_batch_200_distinct_frames_1080p(dmc, port):
    """Every frame has its own tables: the streams, the degrade round trip, the decoder and the chain."""
    from oracle.oracle_py import synth_disp, degrade_blocks
    from depthmapcompression_b200.filters import chain_params
    from depthmapcompression_b200 import capi
    H, W, N = 1080, 1920, 200
    rs = np.random.RandomState(5)
    base = [degrade_blocks(synth_disp(H, W, 300 + f, shift=(f, 2 * f)), f) for f in range(4)]
    frames = np.empty((N, H, W), np.uint8)
    for f in range(N):                                            # distinct frames: a base frame with a few pixels changed
        frames[f] = base[f % 4]
        ys, xs = rs.randint(0, H, 8 + f), rs.randint(0, W, 8 + f)
        frames[f, ys, xs] = rs.randint(0, 256, len(ys))
    blob, offsets = dmc.jpegEncodeGrayBatch(frames, 80, optimize=True)
    streams = streams_of(blob, offsets)
    want = [enc(frames[f], 80) for f in range(N)]
    assert len(set(s[:400] for s in want)) > N // 2              # most frames carry tables of their own
    for f in range(N):
        assert streams[f] == want[f], "frame %d" % f
    dec, nbytes = dmc.degradeJPEG(frames, 80, optimize=True)
    assert [int(x) for x in nbytes] == [len(s) for s in want]
    for f in (0, 1, 4, 99, 163, 199):
        assert_bits_equal(dec[f], cv2.imdecode(np.frombuffer(want[f], np.uint8), 0), "degraded frame %d" % f)
    decb = dmc.jpegDecodeGrayBatch((blob, offsets), H, W)
    assert_bits_equal(decb, dec, "decode(encode optimised) vs degradeJPEG")
    # the golden frames: encode -> decode -> chain against the port
    golden = [load_png(n) for n in ("kinect_meeting_q50.png", "kinect_desk_q50.png", "x264_depth_y.png")]
    gh, gw = golden[0].shape
    gframes = np.stack(golden * 4)
    for q in (50, 80):
        gblob, goffs = dmc.jpegEncodeGrayBatch(gframes, q, optimize=True)
        gstreams = streams_of(gblob, goffs)
        for i, g in enumerate(golden):
            assert gstreams[i] == enc(g, q), "golden frame %d q%d" % (i, q)
        gdec = dmc.jpegDecodeGrayBatch((gblob, goffs), gh, gw)
        out = np.zeros_like(gframes)
        dmc.default_context().chain_batch_jpeg((gblob, goffs), gh, gw, out, chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10))
        for i in (0, 1, 2, 11):
            ref_dec = cv2.imdecode(np.frombuffer(gstreams[i], np.uint8), 0)
            assert_bits_equal(gdec[i], ref_dec, "decoded golden frame %d q%d" % (i, q))
            assert_bits_equal(out[i], port.post_filter_set(ref_dec, 2, 1, 3, 5, 10), "chain on golden frame %d q%d" % (i, q))


def test_decode_more_than_one_group_of_per_frame_tables(dmc):
    """More than 2048 cv2-optimised streams of mixed qualities: two decode groups, every frame with its own tables."""
    rs = np.random.RandomState(21)
    H, W, N = 24, 40, 2300
    base = np.clip(rs.normal(110, 35, (H, W)), 0, 255).astype(np.uint8)
    frames = np.repeat(base[None], N, axis=0)
    for f in range(N):
        ys, xs = rs.randint(0, H, 12), rs.randint(0, W, 12)
        frames[f, ys, xs] = rs.randint(0, 256, 12)
    qs = [int(q) for q in rs.randint(5, 100, N)]
    streams = [enc(frames[f], qs[f]) for f in range(N)]
    dec = dmc.jpegDecodeGrayBatch(streams, H, W)
    for f in range(N):
        assert_bits_equal(dec[f], cv2.imdecode(np.frombuffer(streams[f], np.uint8), 0), "frame %d" % f)
