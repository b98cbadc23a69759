"""SURVEY.md 8f-1, the decode that feeds the chain: the frame-parallel GPU JPEG decoder must reproduce libjpeg-turbo's
default (ISLOW) decoder bit for bit -- the decoder the reference reaches through cv::imdecode(buf, 0) (main.cpp:284,
:521) -- so that chain parity carries through from the bitstream.  The oracle here is cv2.imdecode itself."""
import numpy as np
import pytest

from _util import assert_bits_equal, load_png, make_image

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dmc():
    import depthmapcompression_b200 as m
    m.default_context(0)
    return m


def enc(img, q, *extra):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q] + list(extra))
    assert ok
    return buf


def test_decode_matches_libjpeg_turbo(dmc):
    from oracle.oracle_py import synth_disp, degrade_blocks
    rs = np.random.RandomState(31)
    for (H, W) in [(480, 640), (131, 150), (8, 8), (1, 1), (7, 9), (64, 641), (1080, 1920)]:
        for kind in ("synth", "pw", "noise"):
            img = synth_disp(H, W, 3) if kind == "synth" and H > 16 else make_image(rs, H, W, kind="noise" if kind == "noise" else "pw")
            for q in (5, 25, 50, 80, 95, 100):
                streams = [enc(img, q), enc(img, q, cv2.IMWRITE_JPEG_OPTIMIZE, 1), enc(img, q, cv2.IMWRITE_JPEG_RST_INTERVAL, 3)]
                got = dmc.jpegDecodeGrayBatch(streams, H, W)
                for i, s in enumerate(streams):
                    assert_bits_equal(got[i], cv2.imdecode(s, 0), "%dx%d %s q%d variant %d" % (H, W, kind, q, i))


def test_decode_golden_kinect_and_chain_from_bitstream(dmc, port):
    """simpleTest() from the bitstream on: JPEG q50 -> decode -> PostFilterSet()(2,1,3,5,10), all on the device."""
    import torch
    from depthmapcompression_b200.filters import chain_params
    from depthmapcompression_b200 import capi
    frames = [load_png(n) for n in ("kinect_meeting_q50.png", "kinect_desk_q50.png", "x264_depth_y.png")]
    H, W = frames[0].shape
    streams = [enc(f, 50) for f in frames] * 40            # a 120-frame batch
    n = len(streams)
    d_dec = torch.empty((n, H, W), dtype=torch.uint8, device="cuda"); d_out = torch.empty_like(d_dec)
    ctx = dmc.default_context()
    dmc.jpegDecodeGrayBatch(streams, H, W, dst=d_dec.data_ptr())
    ctx.chain_batch(d_dec.data_ptr(), d_out.data_ptr(), n, H, W, chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10), device=True)
    ctx.synchronize()
    dec = d_dec.cpu().numpy(); out = d_out.cpu().numpy()
    for i in (0, 1, 2, 60, 119):
        ref_dec = cv2.imdecode(streams[i], 0)
        assert_bits_equal(dec[i], ref_dec, "decode frame %d" % i)
        assert_bits_equal(out[i], port.post_filter_set(ref_dec, 2, 1, 3, 5, 10), "chain on decoded frame %d" % i)


def test_unsupported_streams_are_refused(dmc):
    img = np.full((16, 16), 90, np.uint8)
    with pytest.raises(dmc.DmcError):
        dmc.jpegDecodeGrayBatch([enc(img, 50, cv2.IMWRITE_JPEG_PROGRESSIVE, 1)], 16, 16)
    with pytest.raises(dmc.DmcError):
        dmc.jpegDecodeGrayBatch([enc(np.dstack([img, img, img]), 50)], 16, 16)
    with pytest.raises(dmc.DmcError):
        dmc.jpegDecodeGrayBatch([enc(img, 50)], 16, 24)          # size differs from the batch size
    with pytest.raises(dmc.DmcError):
        dmc.jpegDecodeGrayBatch([b"not a jpeg at all"], 16, 16)


def test_streamed_bitstream_to_chain_1080p(dmc, port):
    """dmc_chain_batch_jpeg: host JPEG blobs -> decode -> chain -> host (and -> device), 1080p x 70 frames, a few of them with
    restart intervals (legacy decode path inside the same chunk).  Reference path: main.cpp:276-303."""
    import torch
    from oracle.oracle_py import synth_disp, degrade_blocks
    from depthmapcompression_b200.filters import chain_params
    from depthmapcompression_b200 import capi
    H, W, N = 1080, 1920, 70
    rs = np.random.RandomState(77)
    base = [degrade_blocks(synth_disp(H, W, 1000 + f, shift=(2 * f, f)), f) for f in range(5)]
    base.append(np.clip(base[0].astype(int) + rs.randint(-12, 13, (H, W)), 0, 255).astype(np.uint8))       # noisy: long scans
    streams = []
    for f in range(N):
        extra = (cv2.IMWRITE_JPEG_RST_INTERVAL, 7) if f % 23 == 5 else ()
        streams.append(enc(base[f % len(base)], (50, 80, 95)[f % 3], *extra))
    ctx = dmc.default_context()
    p8 = chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10)
    out = np.zeros((N, H, W), np.uint8)
    ctx.chain_batch_jpeg(streams, H, W, out, p8)
    check = (0, 1, 5, 17, 28, 51, 69)
    for i in check:
        ref_dec = cv2.imdecode(streams[i], 0)
        assert_bits_equal(out[i], port.post_filter_set(ref_dec, 2, 1, 3, 5, 10), "bitstream -> chain, frame %d" % i)
    # a second call reuses every buffer; device destination; the depth chain
    p32 = chain_params(capi.CHAIN_DEPTH32F, 1, 0, 1, 3, 65.0, focus=75.0, baseline=575.0, amp=2.6)
    d32 = torch.zeros((N, H, W), dtype=torch.float32, device="cuda")
    ctx.chain_batch_jpeg(streams, H, W, d32.data_ptr(), p32, device=True); ctx.synchronize()
    for i in (0, 5, 69):
        ref_dec = cv2.imdecode(streams[i], 0)
        assert_bits_equal(d32[i].cpu().numpy(), port.filter_disp8u_depth32f(ref_dec, 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.0), "bitstream -> Depth32F, frame %d" % i)
    out2 = np.zeros((N, H, W), np.uint8)
    ctx.chain_batch_jpeg(streams, H, W, out2, p8)
    assert_bits_equal(out2, out, "second streamed call")


def _streams_1080p(n):
    """n 1080p q80 streams cycling over three degraded synthetic frames -> (streams, index of each frame's base)"""
    from oracle.oracle_py import synth_disp, degrade_blocks
    base = [enc(degrade_blocks(synth_disp(1080, 1920, 2000 + k, shift=(3 * k, k)), k), 80) for k in range(3)]
    return [base[f % 3] for f in range(n)], base


def test_streamed_error_in_a_later_chunk(dmc, port, monkeypatch):
    """dmc_chain_batch_jpeg stops at a malformed stream found while earlier chunks are still in flight, drains its slots
    and leaves the context usable.  DMC_CHUNK_MB=1 makes every 1080p frame a chunk of its own, so the slots come round
    three times in a 12-frame batch."""
    from depthmapcompression_b200.filters import chain_params
    from depthmapcompression_b200 import capi
    monkeypatch.setenv("DMC_CHUNK_MB", "1")
    H, W, N = 1080, 1920, 12
    streams, base = _streams_1080p(N)
    p8 = chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10)
    ctx = dmc.Context(0)
    bad = list(streams); bad[9] = b"not a jpeg at all"
    with pytest.raises(dmc.DmcError, match="JPEG frame 9"):
        ctx.chain_batch_jpeg(bad, H, W, np.zeros((N, H, W), np.uint8), p8)
    out = np.zeros((N, H, W), np.uint8)
    ctx.chain_batch_jpeg(streams, H, W, out, p8)
    want = [port.post_filter_set(cv2.imdecode(s, 0), 2, 1, 3, 5, 10) for s in base]
    for i in range(N):
        assert_bits_equal(out[i], want[i % 3], "call after the failed one, frame %d" % i)
    ctx.close()


def test_streamed_jpeg_through_gateway(dmc, monkeypatch):
    """dmc_chain_batch_jpeg with dmc_set_gateway: the bitstreams and results travel over another device's link, the kernels
    reach its buffers over NVLink.  Results equal the own-link ones, on repeated calls (buffers and events reused) and for a
    device destination.  Needs two GPUs with peer access (skipped on a one-GPU box)."""
    import torch
    from depthmapcompression_b200.filters import chain_params
    from depthmapcompression_b200 import capi
    if capi.lib.dmc_device_count() < 2:
        pytest.skip("needs two GPUs")
    monkeypatch.setenv("DMC_CHUNK_MB", "1")
    H, W, N = 1080, 1920, 12
    streams, _ = _streams_1080p(N)
    p8 = chain_params(capi.CHAIN_DISP8U, 2, 1, 3, 5, 10)
    ctx = dmc.Context(0)
    own = np.zeros((N, H, W), np.uint8); ctx.chain_batch_jpeg(streams, H, W, own, p8)
    d_own = torch.zeros((N, H, W), dtype=torch.uint8, device="cuda:0")
    ctx.chain_batch_jpeg(streams, H, W, d_own.data_ptr(), p8, device=True); ctx.synchronize()
    ctx.set_gateway(1)
    assert ctx.gateway == 1
    for rep in range(2):
        routed = np.zeros_like(own); ctx.chain_batch_jpeg(streams, H, W, routed, p8)
        assert_bits_equal(routed, own, "through the gateway, repetition %d" % rep)
    d_routed = torch.zeros_like(d_own)
    ctx.chain_batch_jpeg(streams, H, W, d_routed.data_ptr(), p8, device=True); ctx.synchronize()
    assert_bits_equal(d_routed.cpu().numpy(), d_own.cpu().numpy(), "through the gateway, device destination")
    ctx.set_gateway(-1)
    ctx.close()


def test_probe_and_hostile_streams(dmc):
    img = make_image(np.random.RandomState(3), 24, 40)
    good = bytes(enc(img, 75))
    assert dmc.jpegProbe(good) == (24, 40)
    for bad in (b"", b"\xff\xd8\xff\xdb\x00\x00", good[:60], good[:len(good) // 2].replace(b"\xff\xda", b"\xff\xdb")):
        with pytest.raises(dmc.DmcError):
            dmc.jpegProbe(bad)
    # a valid header followed by garbage decodes to SOMETHING without hanging or faulting, and the context stays usable
    j = good.index(b"\xff\xda"); sos_len = int.from_bytes(good[j + 2:j + 4], "big")
    rs = np.random.RandomState(4)
    junk = [good[:j + 2 + sos_len] + bytes(rs.randint(0, 255, n).astype(np.uint8)) + b"\xff\xd9" for n in (0, 1, 50, 3000)]
    dmc.jpegDecodeGrayBatch(junk, 24, 40)
    assert_bits_equal(dmc.jpegDecodeGrayBatch([good], 24, 40)[0], cv2.imdecode(np.frombuffer(good, np.uint8), 0), "after garbage")
