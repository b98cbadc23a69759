"""Host-side mirror of the reference's filter.h / util.h operators over numpy arrays (the role cv::Mat plays in the
reference).  Same names, argument order, defaults and error behaviour:

  * a type/size violation that trips CV_Assert in the reference raises DmcError here;
  * the reference's silent no-ops ((type, method) pairs its dispatcher ignores) leave `dst` untouched here too;
  * `dst=None` plays the role of an empty Mat: it is allocated like the reference allocates it;
  * in-place calls (dst is src) are legal for every operator.

Every call is one C-ABI call into libdmc_b200.so; nothing is computed in Python.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import lib, DmcImage, DmcChainParams, DmcBrfParams, DmcError, MEM_HOST, MEM_DEVICE, FULL_KERNEL, BORDER_REPLICATE

_DEPTH = {np.dtype(np.uint8): capi.CV_8U, np.dtype(np.uint16): capi.CV_16U, np.dtype(np.int16): capi.CV_16S,
          np.dtype(np.float32): capi.CV_32F, np.dtype(np.float64): capi.CV_64F}


def _cvtype(a):
    if a.dtype not in _DEPTH:
        raise DmcError(capi.DMC_ERR_TYPE, "unsupported dtype %s" % a.dtype)
    cn = 1 if a.ndim == 2 else a.shape[2]
    return _DEPTH[a.dtype] + ((cn - 1) << 3)


def _img(a):
    """numpy array (rows x cols [x cn], last dims contiguous, row stride free) -> dmc_image"""
    if a.ndim not in (2, 3):
        raise DmcError(capi.DMC_ERR_SIZE, "image must be 2-D or 3-D")
    es = a.dtype.itemsize * (1 if a.ndim == 2 else a.shape[2])
    inner_ok = (a.strides[-1] == a.dtype.itemsize) and (a.ndim == 2 or a.strides[1] == es)
    if not inner_ok:
        raise DmcError(capi.DMC_ERR_SIZE, "pixels of a row must be contiguous")
    return DmcImage(a.ctypes.data, a.shape[0], a.shape[1], _cvtype(a), a.strides[0] if a.shape[0] > 1 else 0, MEM_HOST)


class Context:
    """One dmc_ctx: a device, a stream and scratch memory.  Not thread-safe (like a PostFilterSet instance)."""

    def __init__(self, device=0):
        h = C.c_void_p()
        rc = lib.dmc_create(int(device), C.byref(h))
        if rc != capi.DMC_OK:
            raise DmcError(rc, (lib.dmc_last_error(None) or b"").decode())
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            lib.dmc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc < 0:
            raise DmcError(rc, (lib.dmc_last_error(self.h) or b"").decode())
        return rc

    def synchronize(self):
        self.check(lib.dmc_synchronize(self.h))

    def set_stream(self, cuda_stream):
        self.check(lib.dmc_set_stream(self.h, C.c_void_p(cuda_stream)))

    def set_gateway(self, device):
        """Route this context's host traffic over another device's link (kernels reach its HBM through NVLink); -1 = own link."""
        self.check(lib.dmc_set_gateway(self.h, int(device)))

    @property
    def gateway(self):
        return int(lib.dmc_get_gateway(self.h))

    def set_lanes(self, lanes):
        self.check(lib.dmc_set_lanes(self.h, int(lanes)))

    def profile_enable(self, stage_mask):
        self.check(lib.dmc_profile_enable(self.h, int(stage_mask)))

    def profile_read(self, stage, reset=True):
        """-> (total_ms, launches, pixels) of the event-bracketed launches of `stage` since the last reset"""
        ms, n, px = C.c_double(), C.c_uint64(), C.c_uint64()
        self.check(lib.dmc_profile_read(self.h, stage, C.byref(ms), C.byref(n), C.byref(px), int(reset)))
        return ms.value, n.value, px.value

    @property
    def kernel_launches(self):
        return int(lib.dmc_kernel_launches(self.h))

    # frame batches: src/dst are device pointers (ints) or C-contiguous numpy arrays [n, rows, cols]
    def chain_batch(self, src, dst, n_frames, rows, cols, params, device=False):
        sp = C.c_void_p(src if isinstance(src, int) else src.ctypes.data)
        dp = C.c_void_p(dst if isinstance(dst, int) else dst.ctypes.data)
        return self.check(lib.dmc_chain_batch(self.h, sp, dp, n_frames, rows, cols, C.byref(params), MEM_DEVICE if device else MEM_HOST))

    def chain_batch_jpeg(self, streams, rows, cols, dst, params, device=False):
        """dmc_chain_batch_jpeg: JPEG bitstreams (list of bytes, or a (blob, offsets) pair of numpy arrays / (pointer, offsets)
        for pinned memory) -> decode -> chain, streamed; dst is a host array [n, rows, cols] or a pointer (device=True:
        device memory)."""
        blob, offsets = streams if isinstance(streams, tuple) else pack_streams(streams)
        n = len(offsets) - 1
        bp = C.c_void_p(blob if isinstance(blob, int) else blob.ctypes.data)
        dp = C.c_void_p(dst if isinstance(dst, int) else dst.ctypes.data)
        return self.check(lib.dmc_chain_batch_jpeg(self.h, bp, C.c_void_p(offsets.ctypes.data), n, rows, cols, dp, MEM_DEVICE if device else MEM_HOST, C.byref(params)))

    def chain_batch_images(self, srcs, dsts, params):
        """dmc_chain_batch_images: lists of 2-D numpy arrays (any row stride), one size; dsts are written in place."""
        n = len(srcs)
        S = (capi.DmcImage * n)(*[_img(a) for a in srcs]); D = (capi.DmcImage * n)(*[_img(a) for a in dsts])
        return self.check(lib.dmc_chain_batch_images(self.h, S, D, n, C.byref(params)))


class FrameBatchScheduler:
    """dmc_sched: persistent contexts on several GPUs of one box; chain_batch() shards a host batch over them."""

    def __init__(self, devices):
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = lib.dmc_sched_create(devs, len(devices), C.byref(h))
        if rc != capi.DMC_OK:
            raise DmcError(rc, (lib.dmc_last_error(None) or b"").decode())
        self.h = h

    def chain_batch(self, src, dst, n_frames, rows, cols, params):
        sp = C.c_void_p(src if isinstance(src, int) else src.ctypes.data)
        dp = C.c_void_p(dst if isinstance(dst, int) else dst.ctypes.data)
        rc = lib.dmc_sched_chain_batch(self.h, sp, dp, n_frames, rows, cols, C.byref(params))
        if rc < 0:
            raise DmcError(rc, (lib.dmc_sched_last_error(self.h) or b"").decode())
        return rc

    def routing(self):
        """-> (gateways per device (-1 = own link), GB/s each way with every device on its own link, GB/s each way as routed)"""
        n = lib.dmc_sched_device_count(self.h)
        g = (C.c_int * max(n, 1))(); a, b = C.c_double(), C.c_double()
        lib.dmc_sched_get_routing(self.h, g, C.byref(a), C.byref(b))
        return list(g)[:n], a.value, b.value

    def close(self):
        if getattr(self, "h", None):
            lib.dmc_sched_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def hostlink_probe(devices):
    """dmc_hostlink_probe: measures the host link of `devices` (all copying both ways at once) and proposes which devices'
    links should carry the traffic.  Call it while the devices are idle.  -> dict"""
    devs = (C.c_int * len(devices))(*devices)
    info = capi.DmcHostlinkInfo()
    rc = lib.dmc_hostlink_probe(devs, len(devices), C.byref(info))
    if rc != capi.DMC_OK:
        raise DmcError(rc, "dmc_hostlink_probe failed")
    n = info.n_devices
    return {"devices": list(info.device)[:n], "gateway": list(info.gateway)[:n], "loaded_gbs": [round(x, 2) for x in list(info.loaded_gbs)[:n]],
            "all_gbs": round(info.all_gbs, 2), "best_gbs": round(info.best_gbs, 2), "n_link": info.n_link}


def multi_chain_batch(devices, src, dst, params):
    """Frame-batch scheduler across GPUs in one process: src/dst are host arrays [n, rows, cols]; frames are sharded
    contiguously over `devices` (one host thread and context per device, no collective)."""
    n, rows, cols = src.shape
    devs = (C.c_int * len(devices))(*devices)
    err = C.create_string_buffer(512)
    rc = lib.dmc_multi_chain_batch(devs, len(devices), C.c_void_p(src.ctypes.data), C.c_void_p(dst.ctypes.data), n, rows, cols, C.byref(params), err, 512)
    if rc < 0:
        raise DmcError(rc, err.value.decode())
    return dst


def pack_streams(streams):
    """list of bytes-like JPEG streams -> (blob uint8 array, offsets uint64 array of len n+1)"""
    sizes = [len(x) for x in streams]
    offsets = np.zeros(len(streams) + 1, np.uint64); offsets[1:] = np.cumsum(sizes)
    blob = np.empty(int(offsets[-1]) + 16, np.uint8)
    for i, x in enumerate(streams):
        blob[int(offsets[i]):int(offsets[i + 1])] = np.frombuffer(x, np.uint8) if not isinstance(x, np.ndarray) else x.ravel()
    return blob, offsets


def jpegProbe(stream):
    """dmc_jpeg_probe (host only): -> (rows, cols) of a stream this library can decode; raises DmcError with the reason
    otherwise (malformed / truncated / progressive / colour ...)."""
    a = np.frombuffer(stream, np.uint8) if not isinstance(stream, np.ndarray) else np.ascontiguousarray(stream).ravel()
    r, c = C.c_int(), C.c_int(); err = C.create_string_buffer(256)
    rc = lib.dmc_jpeg_probe(C.c_void_p(a.ctypes.data if a.size else None), a.size, C.byref(r), C.byref(c), err, 256)
    if rc != capi.DMC_OK:
        raise DmcError(rc, err.value.decode())
    return r.value, c.value


def jpegDecodeGrayBatch(streams, rows, cols, dst=None, ctx=None):
    """JPEG bitstreams (list of bytes, or a (blob, offsets) pair) -> [n, rows, cols] uint8, bit-identical to
    cv::imdecode(buf, 0) as the reference calls it (main.cpp:284, :521).  dst: None (new host array), a host array,
    or a device pointer (int)."""
    ctx = ctx or default_context()
    blob, offsets = streams if isinstance(streams, tuple) else pack_streams(streams)
    n = len(offsets) - 1
    device = isinstance(dst, int)
    if dst is None:
        dst = np.empty((n, rows, cols), np.uint8)
    dp = C.c_void_p(dst if device else dst.ctypes.data)
    ctx.check(lib.dmc_jpeg_decode_gray_batch(ctx.h, C.c_void_p(blob.ctypes.data), C.c_void_p(offsets.ctypes.data), n, rows, cols, dp,
                                             MEM_DEVICE if device else MEM_HOST))
    return dst


def jpegProbeColor(stream):
    """dmc_jpeg_probe_color (host only): -> (rows, cols, components) of a stream jpegDecodeColorBatch can decode
    (components 1 or 3); raises DmcError with the reason otherwise (malformed / progressive / CMYK / RGB ...)."""
    a = np.frombuffer(stream, np.uint8) if not isinstance(stream, np.ndarray) else np.ascontiguousarray(stream).ravel()
    r, c, n = C.c_int(), C.c_int(), C.c_int(); err = C.create_string_buffer(256)
    rc = lib.dmc_jpeg_probe_color(C.c_void_p(a.ctypes.data if a.size else None), a.size, C.byref(r), C.byref(c), C.byref(n), err, 256)
    if rc != capi.DMC_OK:
        raise DmcError(rc, err.value.decode())
    return r.value, c.value, n.value


def jpegDecodeColorBatch(streams, rows, cols, dst=None, ctx=None):
    """Baseline colour (or one-component) JPEG bitstreams (list of bytes, or a (blob, offsets) pair) -> [n, rows, cols, 3]
    uint8 BGR, bit-identical to cv2.imdecode(buf, cv2.IMREAD_COLOR | cv2.IMREAD_IGNORE_ORIENTATION).  dst: None (new host
    array), a host array of that shape, or a device pointer (int) -- a device batch that renderViewBatch takes as its
    texture tuple (pointer, n, rows, cols)."""
    ctx = ctx or default_context()
    blob, offsets = streams if isinstance(streams, tuple) else pack_streams(streams)
    n = len(offsets) - 1
    device = isinstance(dst, int)
    if dst is None:
        dst = np.empty((n, max(rows, 0), max(cols, 0), 3), np.uint8)
    elif not device and (dst.dtype != np.uint8 or dst.size != n * rows * cols * 3 or not dst.flags.c_contiguous):
        raise DmcError(capi.DMC_ERR_SIZE, "jpegDecodeColorBatch: dst must be a contiguous uint8 array of n x rows x cols x 3")
    dp = C.c_void_p(dst if device else dst.ctypes.data)
    ctx.check(lib.dmc_jpeg_decode_color_batch(ctx.h, C.c_void_p(blob.ctypes.data), C.c_void_p(offsets.ctypes.data), n, rows, cols, dp,
                                              MEM_DEVICE if device else MEM_HOST))
    return dst


def _jpeg_flags(optimize):
    return capi.JPEG_OPTIMIZE_HUFFMAN if optimize else 0


def jpegEncodeBound(rows, cols, optimize=False):
    """dmc_jpeg_encode_bound_ex (host only): worst-case bytes of one rows x cols stream (optimize: with optimised Huffman
    tables); raises DmcError for sizes the encoder refuses (outside 1..65535, or a bound above 256 MB)."""
    b = C.c_uint64()
    rc = lib.dmc_jpeg_encode_bound_ex(int(rows), int(cols), _jpeg_flags(optimize), C.byref(b))
    if rc != capi.DMC_OK:
        raise DmcError(rc, (lib.dmc_last_error(None) or b"").decode())
    return int(b.value)


def _frames(frames):
    """numpy [n, rows, cols] / [rows, cols] uint8, or (device pointer, n, rows, cols) -> (pointer, n, rows, cols, mem, array)"""
    if isinstance(frames, tuple):
        ptr, n, rows, cols = frames
        return int(ptr), int(n), int(rows), int(cols), MEM_DEVICE, None
    a = np.ascontiguousarray(frames)
    if a.dtype != np.uint8 or a.ndim not in (2, 3):
        raise DmcError(capi.DMC_ERR_TYPE, "frames must be uint8 [n, rows, cols] or [rows, cols]")
    n, rows, cols = (1,) + a.shape if a.ndim == 2 else a.shape
    return a.ctypes.data, n, rows, cols, MEM_HOST, a


def jpegEncodeGrayBatch(frames, quality, ctx=None, blob=None, optimize=False):
    """Baseline JPEG encode of 8-bit frames on the GPU, byte-identical to cv2.imencode(".jpg", f, [IMWRITE_JPEG_QUALITY,
    quality]) of each frame; with optimize=True every frame gets its own optimised Huffman tables, byte-identical to
    cv2.imencode(".jpg", f, [IMWRITE_JPEG_QUALITY, quality, IMWRITE_JPEG_OPTIMIZE, 1]).  frames: uint8 numpy [n, rows, cols] (or one [rows, cols] frame), or (device pointer, n, rows,
    cols).  Returns (blob, offsets) in the layout of pack_streams: stream i is blob[offsets[i]:offsets[i+1]], ready for
    jpegDecodeGrayBatch and Context.chain_batch_jpeg.  blob=None: a new host array; blob=(device pointer, capacity): the
    streams go to device memory and (pointer, offsets) is returned."""
    ctx = ctx or default_context()
    sp, n, rows, cols, smem, keep = _frames(frames)
    offsets = np.zeros(n + 1, np.uint64)
    if blob is None:
        cap = n * jpegEncodeBound(rows, cols, optimize)
        host = np.empty(cap, np.uint8)          # pages the streams never reach are never touched
        bp, bmem = host.ctypes.data, MEM_HOST
    else:
        bp, cap = int(blob[0]), int(blob[1])
        bmem = MEM_DEVICE
    ctx.check(lib.dmc_jpeg_encode_gray_batch_ex(ctx.h, C.c_void_p(sp), smem, n, rows, cols, int(quality), _jpeg_flags(optimize), C.c_void_p(bp), bmem,
                                                cap, offsets.ctypes.data_as(C.POINTER(C.c_uint64))))
    if blob is None:
        return host[:int(offsets[-1])].copy(), offsets
    return bp, offsets


def degradeJPEG(frames, quality, dst=None, ctx=None, optimize=False):
    """The reference's degradeJPEG on the device: decoded = cv2.imdecode(cv2.imencode(f, q), 0) for every frame, and the
    stream sizes in bytes (optimize=True: the sizes of the streams with optimised Huffman tables; the decoded frames are
    the same).  frames: uint8 numpy [n, rows, cols] (or one [rows, cols] frame; nbytes is then an int), or
    (device pointer, n, rows, cols) with dst a device pointer.  Returns (decoded, nbytes)."""
    ctx = ctx or default_context()
    sp, n, rows, cols, mem, a = _frames(frames)
    if mem == MEM_DEVICE:
        if not isinstance(dst, int):
            raise DmcError(capi.DMC_ERR_ARG, "degradeJPEG: device frames need a device pointer dst")
        dp = dst
    else:
        if dst is None or dst.shape != a.shape or dst.dtype != np.uint8 or not dst.flags.c_contiguous:
            dst = np.empty(a.shape, np.uint8)
        dp = dst.ctypes.data
    nbytes = np.zeros(n, np.uint64)
    ctx.check(lib.dmc_jpeg_degrade_gray_batch_ex(ctx.h, C.c_void_p(sp), C.c_void_p(dp), n, rows, cols, int(quality), _jpeg_flags(optimize), mem,
                                                 nbytes.ctypes.data_as(C.POINTER(C.c_uint64))))
    if a is not None and a.ndim == 2:
        return dst, int(nbytes[0])
    return dst, nbytes


JPEG_SAMPLINGS = {"444": capi.DMC_JPEG_SAMPLING_444, "422": capi.DMC_JPEG_SAMPLING_422, "420": capi.DMC_JPEG_SAMPLING_420,
                  "440": capi.DMC_JPEG_SAMPLING_440, "411": capi.DMC_JPEG_SAMPLING_411}


def _sampling(sampling):
    """"444" / "422" / "420" / "440" / "411", or the value of a cv2.IMWRITE_JPEG_SAMPLING_FACTOR_* constant -> that value"""
    if isinstance(sampling, str):
        if sampling not in JPEG_SAMPLINGS:
            raise DmcError(capi.DMC_ERR_ARG, "unknown JPEG sampling %r (one of %s)" % (sampling, ", ".join(JPEG_SAMPLINGS)))
        return JPEG_SAMPLINGS[sampling]
    return int(sampling)


def _color_frames(frames):
    """numpy [n, rows, cols, 3] / [rows, cols, 3] uint8, or (device pointer, n, rows, cols) -> (pointer, n, rows, cols, mem, array)"""
    if isinstance(frames, tuple):
        ptr, n, rows, cols = frames
        return int(ptr), int(n), int(rows), int(cols), MEM_DEVICE, None
    a = np.ascontiguousarray(frames)
    if a.dtype != np.uint8 or a.ndim not in (3, 4) or a.shape[-1] != 3:
        raise DmcError(capi.DMC_ERR_TYPE, "frames must be uint8 [n, rows, cols, 3] or [rows, cols, 3]")
    n, rows, cols = (1,) + a.shape[:2] if a.ndim == 3 else a.shape[:3]
    return a.ctypes.data, n, rows, cols, MEM_HOST, a


def jpegEncodeColorBound(rows, cols, sampling="420"):
    """dmc_jpeg_encode_color_bound (host only): worst-case bytes of one rows x cols colour stream at `sampling`; raises
    DmcError for sizes or samplings the encoder refuses."""
    b = C.c_uint64()
    rc = lib.dmc_jpeg_encode_color_bound(int(rows), int(cols), _sampling(sampling), C.byref(b))
    if rc != capi.DMC_OK:
        raise DmcError(rc, (lib.dmc_last_error(None) or b"").decode())
    return int(b.value)


def jpegEncodeColorBatch(frames, quality, sampling="420", ctx=None, blob=None):
    """Baseline colour JPEG encode of 8UC3 BGR frames on the GPU, byte-identical to cv2.imencode(".jpg", f,
    [IMWRITE_JPEG_QUALITY, quality, IMWRITE_JPEG_SAMPLING_FACTOR, s]) of each frame.  sampling: "444", "422", "420"
    (cv2's default), "440", "411", or a cv2.IMWRITE_JPEG_SAMPLING_FACTOR_* value.  frames: uint8 numpy [n, rows, cols, 3]
    (or one [rows, cols, 3] frame), or (device pointer, n, rows, cols).  Returns (blob, offsets) in the layout of
    pack_streams, ready for jpegDecodeColorBatch.  blob=None: a new host array; blob=(device pointer, capacity): the
    streams go to device memory and (pointer, offsets) is returned."""
    ctx = ctx or default_context()
    sp, n, rows, cols, smem, keep = _color_frames(frames)
    s = _sampling(sampling)
    offsets = np.zeros(n + 1, np.uint64)
    if blob is None:
        cap = n * jpegEncodeColorBound(rows, cols, s)
        host = np.empty(cap, np.uint8)          # pages the streams never reach are never touched
        bp, bmem = host.ctypes.data, MEM_HOST
    else:
        bp, cap = int(blob[0]), int(blob[1])
        bmem = MEM_DEVICE
    ctx.check(lib.dmc_jpeg_encode_color_batch(ctx.h, C.c_void_p(sp), smem, n, rows, cols, int(quality), s, C.c_void_p(bp), bmem,
                                              cap, offsets.ctypes.data_as(C.POINTER(C.c_uint64))))
    if blob is None:
        return host[:int(offsets[-1])].copy(), offsets
    return bp, offsets


def degradeJPEGColor(frames, quality, sampling="420", dst=None, ctx=None):
    """A colour JPEG round trip on the device: decoded = cv2.imdecode(cv2.imencode(f, [IMWRITE_JPEG_QUALITY, quality,
    IMWRITE_JPEG_SAMPLING_FACTOR, s]), IMREAD_COLOR) for every frame, and the stream sizes in bytes; the streams never
    leave the device.  frames as for jpegEncodeColorBatch (one [rows, cols, 3] frame: nbytes is an int); device frames
    need a device pointer dst, which may equal the frames' pointer, and the result is then a texture batch that
    renderViewBatch takes as (pointer, n, rows, cols).  Returns (decoded, nbytes)."""
    ctx = ctx or default_context()
    sp, n, rows, cols, mem, a = _color_frames(frames)
    if mem == MEM_DEVICE:
        if not isinstance(dst, int):
            raise DmcError(capi.DMC_ERR_ARG, "degradeJPEGColor: device frames need a device pointer dst")
        dp = dst
    else:
        if dst is None or dst.shape != a.shape or dst.dtype != np.uint8 or not dst.flags.c_contiguous:
            dst = np.empty(a.shape, np.uint8)
        dp = dst.ctypes.data
    nbytes = np.zeros(n, np.uint64)
    ctx.check(lib.dmc_jpeg_degrade_color_batch(ctx.h, C.c_void_p(sp), C.c_void_p(dp), n, rows, cols, int(quality), _sampling(sampling), mem,
                                               nbytes.ctypes.data_as(C.POINTER(C.c_uint64))))
    if a is not None and a.ndim == 3:
        return dst, int(nbytes[0])
    return dst, nbytes


def frameSSE(a, b, ctx=None):
    """Exact per-frame sum of squared differences of two batches of 8-bit frames on the GPU (dmc_sse_gray_batch).  a, b:
    uint8 numpy [n, rows, cols] (or one [rows, cols] frame), or both (device pointer, n, rows, cols).  -> np.uint64[n]"""
    ctx = ctx or default_context()
    ap, n, rows, cols, mem, ka = _frames(a)
    bp, bn, brows, bcols, bmem, kb = _frames(b)
    if (n, rows, cols, mem) != (bn, brows, bcols, bmem):
        raise DmcError(capi.DMC_ERR_SIZE, "frameSSE: a and b must be batches of one shape in the same memory")
    sse = np.zeros(n, np.uint64)
    ctx.check(lib.dmc_sse_gray_batch(ctx.h, C.c_void_p(ap), C.c_void_p(bp), n, rows, cols, mem, sse.ctypes.data_as(C.POINTER(C.c_uint64))))
    return sse


def _ssim_frames(frames, channels):
    """numpy uint8 [n, rows, cols], [rows, cols], [n, rows, cols, 3] or [rows, cols, 3] (a trailing 3 is a colour frame: a gray
    frame needs cols >= 11), or (device pointer, n, rows, cols) with `channels` -> (pointer, n, rows, cols, channels, mem, array)"""
    if isinstance(frames, tuple):
        ptr, n, rows, cols = (int(x) for x in frames)
        return ptr, n, rows, cols, int(channels), MEM_DEVICE, None
    a = np.ascontiguousarray(frames)
    if a.dtype != np.uint8 or a.ndim not in (2, 3, 4) or (a.ndim == 4 and a.shape[-1] != 3):
        raise DmcError(capi.DMC_ERR_TYPE, "frames must be uint8 [n, rows, cols], [rows, cols], [n, rows, cols, 3] or [rows, cols, 3]")
    cn = 3 if a.ndim == 4 or (a.ndim == 3 and a.shape[-1] == 3) else 1
    shape = a.shape[:-1] if cn == 3 else a.shape
    n, rows, cols = (1,) + shape if len(shape) == 2 else shape
    return a.ctypes.data, n, rows, cols, cn, MEM_HOST, a


def frameSSIM(a, b, ctx=None, channels=1):
    """Per-frame mean structural similarity of two batches of 8-bit frames on the GPU (dmc_ssim_batch; the definition of
    Wang et al. 2004 and of skimage's structural_similarity(data_range=255, gaussian_weights=True, sigma=1.5,
    use_sample_covariance=False), channels averaged).  a, b: uint8 numpy [n, rows, cols] or [rows, cols] (gray), [n, rows, cols, 3]
    or [rows, cols, 3] (interleaved colour), or both (device pointer, n, rows, cols) with channels= 1 or 3.  Frames of at least
    11 x 11.  -> np.float64[n]"""
    ctx = ctx or default_context()
    ap, n, rows, cols, cn, mem, ka = _ssim_frames(a, channels)
    bp, bn, brows, bcols, bcn, bmem, kb = _ssim_frames(b, channels)
    if (n, rows, cols, cn, mem) != (bn, brows, bcols, bcn, bmem):
        raise DmcError(capi.DMC_ERR_SIZE, "frameSSIM: a and b must be batches of one shape in the same memory")
    out = np.zeros(n, np.float64)
    ctx.check(lib.dmc_ssim_batch(ctx.h, C.c_void_p(ap), C.c_void_p(bp), n, rows, cols, cn, mem, out.ctypes.data_as(C.POINTER(C.c_double))))
    return out


_psnr = np.vectorize(lambda sse, pixels: lib.dmc_psnr_from_sse(int(sse), int(pixels)), otypes=[np.float64])


def psnrFromSSE(sse, pixels):
    """PSNR in dB of 8-bit frames of `pixels` pixels from their exact SSE, by the formula of cv2.PSNR (dmc_psnr_from_sse);
    vectorised over both arguments."""
    r = _psnr(np.asarray(sse, np.uint64), np.asarray(pixels, np.uint64))
    return float(r) if r.ndim == 0 else r


def jpegRateDistortion(frames, qualities, params=None, optimize=False, ctx=None, brf=None, ssim=False):
    """The JPEG rate-distortion sweep on the GPU (dmc_jpeg_rd_sweep_ssim): every frame is coded at every quality as cv2.imencode
    codes it (optimize: with optimised Huffman tables), decoded, and with `params` (a chain_params(CHAIN_DISP8U, ...))
    post-filtered; with `brf` (a brf_params(...)) the decoded frames also go through boundaryReconstructionFilter.  No frame
    or stream leaves the device.  frames as for degradeJPEG.  Returns a dict of (n_q, n) arrays: bytes, sse_coded,
    psnr_coded, with params also sse_filtered, psnr_filtered, and with brf also sse_brf, psnr_brf.  ssim=True adds the
    frameSSIM of every arm against the source: ssim_coded (and ssim_filtered, ssim_brf with params, brf), float64."""
    ctx = ctx or default_context()
    sp, n, rows, cols, mem, keep = _frames(frames)
    q = np.ascontiguousarray(np.asarray(qualities).ravel(), dtype=np.int32)
    shape = (len(q), n)
    U64 = C.POINTER(C.c_uint64)
    nbytes, sc = np.zeros(shape, np.uint64), np.zeros(shape, np.uint64)
    sf = np.zeros(shape, np.uint64) if params is not None else None
    sb = np.zeros(shape, np.uint64) if brf is not None else None
    qs = {k: np.zeros(shape, np.float64) for k, on in (("ssim_coded", True), ("ssim_filtered", params is not None), ("ssim_brf", brf is not None))
          if ssim and on}
    DP = C.POINTER(C.c_double)
    ctx.check(lib.dmc_jpeg_rd_sweep_ssim(ctx.h, C.c_void_p(sp), mem, n, rows, cols, q.ctypes.data_as(C.POINTER(C.c_int)), len(q), _jpeg_flags(optimize),
                                         C.byref(params) if params is not None else None, C.byref(brf) if brf is not None else None,
                                         nbytes.ctypes.data_as(U64), sc.ctypes.data_as(U64), sf.ctypes.data_as(U64) if sf is not None else None,
                                         sb.ctypes.data_as(U64) if sb is not None else None,
                                         *[qs[k].ctypes.data_as(DP) if k in qs else None for k in ("ssim_coded", "ssim_filtered", "ssim_brf")]))
    out = {"bytes": nbytes, "sse_coded": sc, "psnr_coded": psnrFromSSE(sc, rows * cols)}
    if sf is not None:
        out["sse_filtered"] = sf
        out["psnr_filtered"] = psnrFromSSE(sf, rows * cols)
    if sb is not None:
        out["sse_brf"] = sb
        out["psnr_brf"] = psnrFromSSE(sb, rows * cols)
    out.update(qs)
    return out


def jpegViewRateDistortion(disp, texture, qualities, params, f, R, t, K, isSub=True, optimize=False, exact_divide=False, ctx=None, brf=None,
                           ssim=False):
    """The view-synthesis rate-distortion sweep on the GPU (dmc_jpeg_view_rd_sweep_ssim): coded depth scored by the views it
    renders, as pointcloudTest renders a decoded depth map.  For every frame, quality and camera (R[v], t[v], shared K) the
    reference view fillSmallHole(projectImagefromXYZ(texture, reprojectXYZ(D(disp), f), ...)), with D the unfiltered
    disp8U2depth32F, is compared with the view of D(decoded) and with the view of filterDisp8U2Depth32F(decoded, params).
    disp: frames as for degradeJPEG; texture: uint8 numpy [n, rows, cols, 3] (or one [rows, cols, 3] image), or (device
    pointer, n, rows, cols) when disp is a device tuple.  params: chain_params(CHAIN_DEPTH32F, ..., focus, baseline, amp).
    R: [n_views, 3, 3] (or one 3x3), t: [n_views, 3].  Returns a dict: bytes (n_q, n), and sse_view_coded, psnr_view_coded,
    sse_view_filtered, psnr_view_filtered (n_q, n_views, n); the PSNR is cv2.PSNR of the two 8UC3 views.  brf (a
    brf_params(...)): also sse_view_brf, psnr_view_brf, the view of D(boundaryReconstructionFilter(decoded)) against the
    same reference view.  ssim=True adds the frameSSIM of the 8UC3 views against the reference view: ssim_view_coded,
    ssim_view_filtered (and ssim_view_brf with brf), float64 (n_q, n_views, n)."""
    ctx = ctx or default_context()
    sp, n, rows, cols, mem, keep = _frames(disp)
    if isinstance(texture, tuple):
        tp, tn, trows, tcols = (int(x) for x in texture)
        tmem, tkeep = MEM_DEVICE, None
    else:
        tkeep = np.ascontiguousarray(texture)
        if tkeep.dtype != np.uint8 or tkeep.ndim not in (3, 4) or tkeep.shape[-1] != 3:
            raise DmcError(capi.DMC_ERR_TYPE, "texture must be uint8 [n, rows, cols, 3] or [rows, cols, 3]")
        tn, trows, tcols = (1,) + tkeep.shape[:2] if tkeep.ndim == 3 else tkeep.shape[:3]
        tp, tmem = tkeep.ctypes.data, MEM_HOST
    if (tn, trows, tcols, tmem) != (n, rows, cols, mem):
        raise DmcError(capi.DMC_ERR_SIZE, "jpegViewRateDistortion: disp and texture must be batches of one size in the same memory")
    q = np.ascontiguousarray(np.asarray(qualities).ravel(), dtype=np.int32)
    Rs = np.ascontiguousarray(R, np.float64).reshape(-1, 9)
    ts = np.ascontiguousarray(t, np.float64).reshape(-1, 3)
    Ks = np.ascontiguousarray(K, np.float64).reshape(9)
    if Rs.shape[0] != ts.shape[0]:
        raise DmcError(capi.DMC_ERR_ARG, "jpegViewRateDistortion: R and t must hold one camera each")
    nv = Rs.shape[0]
    U64, DP = C.POINTER(C.c_uint64), C.POINTER(C.c_double)
    nbytes = np.zeros((len(q), n), np.uint64)
    sc, sf = np.zeros((len(q), nv, n), np.uint64), np.zeros((len(q), nv, n), np.uint64)
    sb = np.zeros((len(q), nv, n), np.uint64) if brf is not None else None
    qs = {k: np.zeros((len(q), nv, n), np.float64) for k, on in (("ssim_view_coded", True), ("ssim_view_filtered", True), ("ssim_view_brf", brf is not None))
          if ssim and on}
    ctx.check(lib.dmc_jpeg_view_rd_sweep_ssim(ctx.h, C.c_void_p(sp), C.c_void_p(tp), mem, n, rows, cols, q.ctypes.data_as(C.POINTER(C.c_int)), len(q),
                                              _jpeg_flags(optimize), C.byref(params), C.byref(brf) if brf is not None else None, float(f),
                                              Rs.ctypes.data_as(DP), ts.ctypes.data_as(DP), nv, Ks.ctypes.data_as(DP), int(bool(isSub)),
                                              capi.RENDER_EXACT_DIVIDE if exact_divide else 0, nbytes.ctypes.data_as(U64), sc.ctypes.data_as(U64),
                                              sf.ctypes.data_as(U64), sb.ctypes.data_as(U64) if sb is not None else None,
                                              *[qs[k].ctypes.data_as(DP) if k in qs else None for k in ("ssim_view_coded", "ssim_view_filtered", "ssim_view_brf")]))
    px = 3 * rows * cols
    out = {"bytes": nbytes, "sse_view_coded": sc, "psnr_view_coded": psnrFromSSE(sc, px),
           "sse_view_filtered": sf, "psnr_view_filtered": psnrFromSSE(sf, px)}
    if sb is not None:
        out["sse_view_brf"] = sb
        out["psnr_view_brf"] = psnrFromSSE(sb, px)
    out.update(qs)
    return out


_default = {}


def default_context(device=0):
    if device not in _default:
        _default[device] = Context(device)
    return _default[device]


def brf_params(ksize=(13, 13), frec=1.0, color=1.0, space=1.0):
    """Parameters of boundaryReconstructionFilter(src, dest, ksize, frec, color, space) for boundaryReconstructionFilterBatch
    and the brf= arm of the sweeps.  The defaults are pointcloudTest's call (main.cpp:306-311)."""
    kw, kh = _ksize(ksize)
    return DmcBrfParams(kw, kh, float(frec), float(color), float(space))


def chain_params(chain, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method=FULL_KERNEL, focus=0.0, baseline=0.0, amp=0.0):
    return DmcChainParams(chain, median_r, gaussian_r, minmax_r, brange_r, float(brange_th), brange_method, focus, baseline, amp)


def _out(dst, src, dtype=None, shape=None):
    dtype = np.dtype(dtype or src.dtype); shape = shape or src.shape
    if dst is None or dst.shape != tuple(shape) or dst.dtype != dtype:
        return np.empty(shape, dtype)          # Mat::create on an empty / mismatching Mat
    return dst


class _PinnedOwner:
    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            lib.dmc_host_free(C.c_void_p(self.ptr))
        except Exception:
            pass


def pinned_empty(shape, dtype=np.uint8):
    """numpy array in pinned, device-mapped host memory (dmc_host_alloc): single frames of up to 2 MB are then processed in place
    over the host link, and the streaming entry points overlap their copies.  Freed with the array."""
    dtype = np.dtype(dtype); n = int(np.prod(shape)) * dtype.itemsize
    ptr = lib.dmc_host_alloc(max(n, 1))
    if not ptr:
        raise DmcError(capi.DMC_ERR_CUDA, "dmc_host_alloc failed")
    owner = _PinnedOwner(ptr)
    buf = (C.c_uint8 * max(n, 1)).from_address(ptr)
    a = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[ptr] = owner            # numpy keeps `buf` alive, not `owner`: tie the allocation to the interpreter unless released
    return a


_PINNED = {}


def pinned_free(a):
    """releases an array made by pinned_empty (optional: otherwise it lives until the interpreter exits)"""
    _PINNED.pop(a.ctypes.data, None)


def host_register(a):
    """pins and device-maps an existing contiguous numpy array (cudaHostRegister) -- see dmc_host_register"""
    rc = lib.dmc_host_register(C.c_void_p(a.ctypes.data), a.nbytes)
    if rc < 0:
        raise DmcError(rc, "dmc_host_register failed")


def host_unregister(a):
    rc = lib.dmc_host_unregister(C.c_void_p(a.ctypes.data))
    if rc < 0:
        raise DmcError(rc, "dmc_host_unregister failed")


class PostFilterSet:
    """filter.h:32-42.  Owns nothing in Python: the scratch Mats `buff`, `bufff` of the reference live in the dmc_ctx."""

    def __init__(self, ctx=None):
        self.ctx = ctx or default_context()

    def __call__(self, src, dest, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method=FULL_KERNEL):
        dest = _out(dest, src, np.uint8)
        s, d = _img(src), _img(dest)
        self.ctx.check(lib.dmc_post_filter_set(self.ctx.h, C.byref(s), C.byref(d), median_r, gaussian_r, minmax_r, brange_r, int(brange_th), brange_method))
        return dest

    def filterDisp8U2Depth32F(self, src, dest, focus, baseline, amp, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method=FULL_KERNEL):
        dest = _out(dest, src, np.float32)
        s, d = _img(src), _img(dest)
        self.ctx.check(lib.dmc_filter_disp8u_depth32f(self.ctx.h, C.byref(s), C.byref(d), focus, baseline, amp, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method))
        return dest

    def filterDisp8U2Depth16U(self, src, dest, focus, baseline, amp, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method=FULL_KERNEL):
        dest = _out(dest, src, np.uint16)
        s, d = _img(src), _img(dest)
        self.ctx.check(lib.dmc_filter_disp8u_depth16u(self.ctx.h, C.byref(s), C.byref(d), focus, baseline, amp, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method))
        return dest

    def filterDisp8U2Disp32F(self, src, dest, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method=FULL_KERNEL):
        dest = _out(dest, src, np.uint16)
        s, d = _img(src), _img(dest)
        self.ctx.check(lib.dmc_filter_disp8u_disp32f(self.ctx.h, C.byref(s), C.byref(d), median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method))
        return dest


def _ksize(k):
    return (k, k) if isinstance(k, int) else (int(k[0]), int(k[1]))     # Size(width, height)


def binalyWeightedRangeFilter(src, dst, kernelSize, threshold, method, borderType=BORDER_REPLICATE, ctx=None):
    """filter.h:29.  `dst=None`: created like `dst.create(src.size(), src.type())` (binalyWeightedRangeFilter.cpp:1108);
    for the reference's no-op (type, method) pairs a fresh dst therefore holds unspecified bytes, as in the reference."""
    ctx = ctx or default_context()
    kw, kh = _ksize(kernelSize)
    dst = _out(dst, src)
    s, d = _img(src), _img(dst)
    ctx.check(lib.dmc_bwrf(ctx.h, C.byref(s), C.byref(d), kw, kh, threshold, method, borderType))
    return dst


def jointBinalyWeightedRangeFilter(src, guide, dst, kernelSize, threshold, method=FULL_KERNEL, ctx=None):
    """Extension (no reference counterpart, SURVEY 8f-4): binalyWeightedRangeFilter on the 8UC1 image `src` with the binary
    weights taken from `guide` (8UC3 colour or 8UC1) instead of from src.  guide == src gives binalyWeightedRangeFilter."""
    ctx = ctx or default_context()
    kw, kh = _ksize(kernelSize)
    dst = _out(dst, src)
    s, g, d = _img(src), _img(guide), _img(dst)
    ctx.check(lib.dmc_joint_bwrf(ctx.h, C.byref(s), C.byref(g), C.byref(d), kw, kh, threshold, method))
    return dst


def blurRemoveMinMax(src, dest, r, ctx=None):
    """filter.h:19"""
    ctx = ctx or default_context()
    dest = _out(dest, src)
    s, d = _img(src), _img(dest)
    ctx.check(lib.dmc_blur_remove_minmax(ctx.h, C.byref(s), C.byref(d), r))
    return dest


blurRemoveMinMaxBase = blurRemoveMinMax      # filter.h:20 -- scalar twin of the same computation (minmaxFilter.cpp:7-46)


def maxFilter(src, dest, ksize, borderType=BORDER_REPLICATE, ctx=None):
    """filter.h:17"""
    ctx = ctx or default_context()
    kw, kh = _ksize(ksize)
    dest = _out(dest, src)
    s, d = _img(src), _img(dest)
    ctx.check(lib.dmc_max_filter(ctx.h, C.byref(s), C.byref(d), kw, kh, borderType))
    return dest


def minFilter(src, dest, ksize, borderType=BORDER_REPLICATE, ctx=None):
    """filter.h:18"""
    ctx = ctx or default_context()
    kw, kh = _ksize(ksize)
    dest = _out(dest, src)
    s, d = _img(src), _img(dest)
    ctx.check(lib.dmc_min_filter(ctx.h, C.byref(s), C.byref(d), kw, kh, borderType))
    return dest


def boundaryReconstructionFilter(src, dest, ksize, frec, color, space, ctx=None):
    """filter.h:45"""
    ctx = ctx or default_context()
    kw, kh = _ksize(ksize)
    dest = _out(dest, src)
    s, d = _img(src), _img(dest)
    ctx.check(lib.dmc_boundary_reconstruction(ctx.h, C.byref(s), C.byref(d), kw, kh, frec, color, space))
    return dest


def boundaryReconstructionFilterBatch(frames, dst=None, ksize=(13, 13), frec=1.0, color=1.0, space=1.0, ctx=None):
    """boundaryReconstructionFilter (filter.h:45) on a batch of frames (dmc_brf_batch): every frame of the result equals
    boundaryReconstructionFilter of that frame.  frames: numpy [n, rows, cols] (or one [rows, cols] frame) of uint8, uint16,
    int16, float32 or float64, streamed through the device; or (device pointer, n, rows, cols[, dtype]) (dtype defaults to
    uint8) with dst a device pointer, processed in stream order.  dst=None: a new host array; dst is frames: in place."""
    ctx = ctx or default_context()
    b = brf_params(ksize, frec, color, space)
    if isinstance(frames, tuple):
        ptr, n, rows, cols = (int(x) for x in frames[:4])
        dt = np.dtype(frames[4] if len(frames) > 4 else np.uint8)
        if dt not in _DEPTH:
            raise DmcError(capi.DMC_ERR_TYPE, "unsupported dtype %s" % dt)
        if not isinstance(dst, int):
            raise DmcError(capi.DMC_ERR_ARG, "boundaryReconstructionFilterBatch: device frames need a device pointer dst")
        ctx.check(lib.dmc_brf_batch(ctx.h, C.c_void_p(ptr), C.c_void_p(dst), n, rows, cols, _DEPTH[dt], C.byref(b), MEM_DEVICE))
        return dst
    a = frames if isinstance(frames, np.ndarray) and frames.flags.c_contiguous else np.ascontiguousarray(frames)
    if a.ndim not in (2, 3):
        raise DmcError(capi.DMC_ERR_SIZE, "frames must be [n, rows, cols] or [rows, cols]")
    if a.dtype not in _DEPTH:
        raise DmcError(capi.DMC_ERR_TYPE, "unsupported dtype %s" % a.dtype)
    n, rows, cols = (1,) + a.shape if a.ndim == 2 else a.shape
    if dst is None or dst.shape != a.shape or dst.dtype != a.dtype or not dst.flags.c_contiguous:
        dst = np.empty(a.shape, a.dtype)
    ctx.check(lib.dmc_brf_batch(ctx.h, C.c_void_p(a.ctypes.data), C.c_void_p(dst.ctypes.data), n, rows, cols, _DEPTH[a.dtype], C.byref(b), MEM_HOST))
    return dst


def prepareDisparityBatch(depth16, focal_baseline, a=1.0, b=0.0, passes=2, dst=None, ctx=None):
    """pointcloudTest's preparation of sensor depth on a batch (dmc_prepare_disp_batch): every frame of the result equals
    fillOcclusion(depth16U2disp8U(frame, focal_baseline, a, b), 0, FILL_DISPARITY), and with passes=2 (pointcloudTest,
    main.cpp:254-260) that filled again around a transpose; passes=1 is simpleTest's call.  depth16: uint16 numpy
    [n, rows, cols] (or one [rows, cols] frame), streamed through the device; or (device pointer, n, rows, cols) with dst a
    device pointer, processed in stream order.  dst=None: a new uint8 host array."""
    ctx = ctx or default_context()
    if isinstance(depth16, tuple):
        ptr, n, rows, cols = (int(x) for x in depth16)
        if not isinstance(dst, int):
            raise DmcError(capi.DMC_ERR_ARG, "prepareDisparityBatch: device frames need a device pointer dst")
        ctx.check(lib.dmc_prepare_disp_batch(ctx.h, C.c_void_p(ptr), C.c_void_p(dst), n, rows, cols, focal_baseline, a, b, int(passes), MEM_DEVICE))
        return dst
    s = np.ascontiguousarray(depth16)
    if s.dtype != np.uint16 or s.ndim not in (2, 3):
        raise DmcError(capi.DMC_ERR_TYPE, "prepareDisparityBatch: depth16 must be uint16 [n, rows, cols] or [rows, cols]")
    n, rows, cols = (1,) + s.shape if s.ndim == 2 else s.shape
    if dst is None or dst.shape != s.shape or dst.dtype != np.uint8 or not dst.flags.c_contiguous:
        dst = np.empty(s.shape, np.uint8)
    ctx.check(lib.dmc_prepare_disp_batch(ctx.h, C.c_void_p(s.ctypes.data), C.c_void_p(dst.ctypes.data), n, rows, cols, focal_baseline, a, b, int(passes), MEM_HOST))
    return dst


def renderViewBatch(depth, texture, f, R, t, K, isSub=True, exact_divide=False, dst=None, ctx=None):
    """pointcloudTest's views of a batch (dmc_render_view_batch): views[v, i] = fillSmallHole(projectImagefromXYZ(texture[i],
    reprojectXYZ(depth[i], f), R[v], t[v], K, isSub)), the fill in place (main.cpp:321-355).  depth: numpy [n, rows, cols]
    (or one [rows, cols] frame) of uint8, int16, uint16 or float32 (filterDisp8U2Depth32F's output as it is); texture: uint8
    [n, rows, cols, 3] (or one [rows, cols, 3] image).  Or device tuples (pointer, n, rows, cols[, dtype]) for depth (dtype
    defaults to float32) and (pointer, n, rows, cols) for texture, with dst a device pointer, processed in stream order.
    R: [n_views, 3, 3] (or one 3x3), t: [n_views, 3].  Returns uint8 [n_views, n, rows, cols, 3] (dst=None: a new host array)."""
    ctx = ctx or default_context()
    Rs = np.ascontiguousarray(R, np.float64).reshape(-1, 9)
    ts = np.ascontiguousarray(t, np.float64).reshape(-1, 3)
    Ks = np.ascontiguousarray(K, np.float64).reshape(9)
    if Rs.shape[0] != ts.shape[0]:
        raise DmcError(capi.DMC_ERR_ARG, "renderViewBatch: R and t must hold one camera each")
    nv = Rs.shape[0]
    if isinstance(depth, tuple):
        dp, n, rows, cols = (int(x) for x in depth[:4])
        dt = np.dtype(depth[4] if len(depth) > 4 else np.float32)
        if not isinstance(texture, tuple) or tuple(int(x) for x in texture[1:4]) != (n, rows, cols):
            raise DmcError(capi.DMC_ERR_SIZE, "renderViewBatch: device depth needs a device texture tuple of the same batch")
        if not isinstance(dst, int):
            raise DmcError(capi.DMC_ERR_ARG, "renderViewBatch: device frames need a device pointer dst")
        tp, mem, out = int(texture[0]), MEM_DEVICE, dst
    else:
        d, tex = np.ascontiguousarray(depth), np.ascontiguousarray(texture)
        if d.ndim not in (2, 3) or tex.dtype != np.uint8 or tex.ndim != d.ndim + 1 or tex.shape[:-1] != d.shape or tex.shape[-1] != 3:
            raise DmcError(capi.DMC_ERR_SIZE, "renderViewBatch: depth [n, rows, cols] and texture uint8 [n, rows, cols, 3] of one batch")
        dt = d.dtype
        n, rows, cols = (1,) + d.shape if d.ndim == 2 else d.shape
        dp, tp, mem = d.ctypes.data, tex.ctypes.data, MEM_HOST
        shape = (nv, n, rows, cols, 3)
        if dst is None or dst.shape != shape or dst.dtype != np.uint8 or not dst.flags.c_contiguous:
            dst = np.empty(shape, np.uint8)
        out = dst.ctypes.data
    if dt not in _DEPTH or _DEPTH[dt] == capi.CV_64F:
        raise DmcError(capi.DMC_ERR_TYPE, "renderViewBatch: depth must be uint8, int16, uint16 or float32")
    DP = C.POINTER(C.c_double)
    ctx.check(lib.dmc_render_view_batch(ctx.h, C.c_void_p(dp), _DEPTH[dt], C.c_void_p(tp), mem, n, rows, cols, float(f), Rs.ctypes.data_as(DP),
                                        ts.ctypes.data_as(DP), nv, Ks.ctypes.data_as(DP), int(bool(isSub)),
                                        capi.RENDER_EXACT_DIVIDE if exact_divide else 0, C.c_void_p(out)))
    return dst


def minmaxBoundaryReconstructionFilter(src, dest, r, ksize, frec, color, space, ctx=None):
    """Extension (filter_ext.h): blurRemoveMinMax(r) fused into boundaryReconstructionFilter, one kernel, src read once;
    bit-identical to the two reference calls.  8U / 16U / 16S, single channel."""
    ctx = ctx or default_context()
    kw, kh = _ksize(ksize)
    dest = _out(dest, src)
    s, d = _img(src), _img(dest)
    ctx.check(lib.dmc_minmax_boundary_reconstruction(ctx.h, C.byref(s), C.byref(d), r, kw, kh, frec, color, space))
    return dest


def smallGaussianBlur(src, dest, d, sigma, ctx=None):
    """filter.h:14"""
    ctx = ctx or default_context()
    dest = _out(dest, src)
    s, o = _img(src), _img(dest)
    ctx.check(lib.dmc_small_gaussian(ctx.h, C.byref(s), C.byref(o), d, sigma))
    return dest


def medianBlur(src, dst, ksize, ctx=None):
    """cv::medianBlur as the chain calls it (postFilterSet.cpp:23)"""
    ctx = ctx or default_context()
    dst = _out(dst, src)
    s, d = _img(src), _img(dst)
    ctx.check(lib.dmc_median_blur(ctx.h, C.byref(s), C.byref(d), ksize))
    return dst


def _convert(fn, src, dest, ddtype, fb, a, b, ctx, zero_new=True):
    ctx = ctx or default_context()
    if dest is None or dest.shape != src.shape or dest.dtype != np.dtype(ddtype):
        dest = np.zeros(src.shape, ddtype)     # Mat::zeros(src.size(), type) (depthmapUtil.cpp:925-926)
    s, d = _img(src), _img(dest)
    ctx.check(fn(ctx.h, C.byref(s), C.byref(d), fb, a, b))
    return dest


def disp8U2depth32F(src, dest, focal_baseline, a=1.0, b=0.0, ctx=None):
    """util.h:28"""
    return _convert(lib.dmc_disp8u2depth32f, src, dest, np.float32, focal_baseline, a, b, ctx)


def depth32F2disp8U(src, dest, focal_baseline, a=1.0, b=0.0, ctx=None):
    """util.h:25"""
    return _convert(lib.dmc_depth32f2disp8u, src, dest, np.uint8, focal_baseline, a, b, ctx)


def depth16U2disp8U(src, dest, focal_baseline, a=1.0, b=0.0, ctx=None):
    """util.h:27"""
    return _convert(lib.dmc_depth16u2disp8u, src, dest, np.uint8, focal_baseline, a, b, ctx)


def disp16S2depth16U(src, dest, focal_baseline, a=1.0, b=0.0, ctx=None):
    """util.h:26"""
    return _convert(lib.dmc_disp16s2depth16u, src, dest, np.uint16, focal_baseline, a, b, ctx)


def fillOcclusion(src, invalidvalue, disp_or_depth=capi.FILL_DEPTH, ctx=None):
    """util.h:24 -- in place"""
    ctx = ctx or default_context()
    s = _img(src)
    ctx.check(lib.dmc_fill_occlusion(ctx.h, C.byref(s), int(invalidvalue), disp_or_depth))
    return src


def transpose(src, dst=None, ctx=None):
    """cv::transpose (main.cpp:258, :260), single channel"""
    ctx = ctx or default_context()
    if dst is None or dst.shape != (src.shape[1], src.shape[0]) or dst.dtype != src.dtype:
        dst = np.empty((src.shape[1], src.shape[0]), src.dtype)
    s, d = _img(src), _img(dst)
    ctx.check(lib.dmc_transpose(ctx.h, C.byref(s), C.byref(d)))
    return dst


def reprojectXYZ(depth, xyz, f, ctx=None):
    """util.h:11 -- xyz is (rows*cols) x 1 x 3 float32"""
    ctx = ctx or default_context()
    n = depth.shape[0] * depth.shape[1]
    if xyz is None or xyz.size != n * 3 or xyz.dtype != np.float32:
        xyz = np.zeros((n, 1, 3), np.float32)          # Mat::zeros(area, 1, CV_32FC3) depthmapUtil.cpp:453
    s = _img(depth)
    x3 = xyz.reshape(n, 1, 3)
    d = _img(x3)
    ctx.check(lib.dmc_reproject_xyz(ctx.h, C.byref(s), C.byref(d), f))
    return xyz


# ---- point-cloud render (util.h:12-13, :25, :33) ------------------------------------------------------------------------
def _cam(R, t, K):
    R = np.ascontiguousarray(R, np.float64).reshape(9); t = np.ascontiguousarray(t, np.float64).reshape(3); K = np.ascontiguousarray(K, np.float64).reshape(9)
    DP = C.POINTER(C.c_double)
    return (R, t, K), (R.ctypes.data_as(DP), t.ctypes.data_as(DP), K.ctypes.data_as(DP))


def projectPointsSimple(xyz, R, t, K, dest=None, exact_divide=False, ctx=None):
    """util.h:33: xyz [n, 3] float32 -> [n, 2] float32 (the reference fills a vector<Point2f>)."""
    ctx = ctx or default_context()
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 1, 3); n = xyz.shape[0]
    dest = _out(dest, xyz, np.float32, (n, 1, 2))
    keep, cam = _cam(R, t, K)
    a, b = _img(xyz), _img(dest)
    ctx.check(lib.dmc_project_points(ctx.h, C.byref(a), cam[0], cam[1], cam[2], C.byref(b), capi.RENDER_EXACT_DIVIDE if exact_divide else 0))
    return dest.reshape(n, 2)


def projectImagefromXYZ(image, destimage, xyz, R, t, K, dist=None, mask=None, isSub=False, want_depth=False, exact_divide=False, ctx=None):
    """util.h:12-13.  `dist` and `mask` are accepted and ignored, as in the reference.  Returns destimage, or
    (destimage, depth, pt) with want_depth (the second overload's outputs)."""
    ctx = ctx or default_context()
    if image.ndim != 3 or image.shape[2] != 3 or image.dtype != np.uint8:
        raise DmcError(capi.DMC_ERR_TYPE, "projectImagefromXYZ: image must be CV_8UC3")
    H, W = image.shape[:2]
    destimage = _out(destimage, image)
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 1, 3)
    keep, cam = _cam(R, t, K)
    a, d, x = _img(image), _img(destimage), _img(xyz)
    depth = np.empty((H, W), np.float32) if want_depth else None
    pt = np.empty((H * W, 1, 2), np.float32) if want_depth else None
    zi = C.byref(_img(depth)) if want_depth else None
    pi = C.byref(_img(pt)) if want_depth else None
    ctx.check(lib.dmc_project_image_from_xyz(ctx.h, C.byref(a), C.byref(d), C.byref(x), cam[0], cam[1], cam[2], int(bool(isSub)), zi, pi,
                                             capi.RENDER_EXACT_DIVIDE if exact_divide else 0))
    return (destimage, depth, pt.reshape(-1, 2)) if want_depth else destimage


def fillSmallHole(src, dest=None, ctx=None):
    """util.h:25.  dest=None or dest is src: in place, as main.cpp:355 calls it; otherwise dest keeps its content outside the holes."""
    ctx = ctx or default_context()
    if dest is None:
        dest = src
    a, b = _img(src), _img(dest)
    ctx.check(lib.dmc_fill_small_hole(ctx.h, C.byref(a), C.byref(b)))
    return dest
