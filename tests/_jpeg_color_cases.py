"""Colour JPEG test streams shared by the CPU emulation and GPU tests of the colour decoder: images of four kinds, cv2
encodings over samplings / qualities / table kinds / restart intervals, and edited streams the decoder must refuse."""
import numpy as np

import cv2

SIZES = [(1, 1), (1, 2), (2, 1), (2, 3), (3, 3), (8, 8), (15, 17), (16, 16), (17, 23), (61, 83)]
KINDS = ("noise", "gradient", "flat", "saturated")
SAMPLINGS = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
             "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440,
             "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411}
QUALITIES = (5, 25, 50, 75, 90, 100)
TABLES = ("standard", "optimised", "restart")


def image(kind, H, W, seed=0):
    """uint8 [H, W, 3] BGR: noise, smooth gradients, one flat colour, or saturated primaries (which exercise the clamp)."""
    rs = np.random.RandomState(seed + 7919 * H + W)
    if kind == "noise":
        return rs.randint(0, 256, (H, W, 3)).astype(np.uint8)
    if kind == "gradient":
        yy, xx = np.mgrid[0:H, 0:W]
        return np.dstack([xx * 255 // max(W - 1, 1), yy * 255 // max(H - 1, 1), (xx + yy) * 127 // max(H + W - 2, 1) + 64]).astype(np.uint8)
    if kind == "flat":
        return np.full((H, W, 3), (37, 200, 90), np.uint8)
    return (rs.randint(0, 2, (H, W, 3)) * 255).astype(np.uint8)


def textured(H, W, seed=0):
    """A smooth colour gradient with +-20 of noise: photograph-like entropy."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    base = np.dstack([xx * 255 // W, yy * 255 // H, (xx + yy) * 255 // (H + W)]).astype(np.int32)
    return np.clip(base + rs.randint(-20, 21, (H, W, 3)), 0, 255).astype(np.uint8)


def encode(img, q, sampling="420", tables="standard", rst=2):
    params = [cv2.IMWRITE_JPEG_QUALITY, q]
    if img.ndim == 3:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLINGS[sampling]]
    if tables == "optimised":
        params += [cv2.IMWRITE_JPEG_OPTIMIZE, 1]
    elif tables == "restart":
        params += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    ok, buf = cv2.imencode(".jpg", img, params)
    assert ok
    return np.ascontiguousarray(buf).ravel()


def reference(stream):
    a = np.frombuffer(stream, np.uint8) if isinstance(stream, (bytes, bytearray)) else np.asarray(stream, np.uint8)
    return cv2.imdecode(a, cv2.IMREAD_COLOR | cv2.IMREAD_IGNORE_ORIENTATION)


def _segments(b):
    """(marker, start, end) of the marker segments before the first SOS (end: one past the segment)."""
    out, i = [], 2
    while i + 4 <= len(b):
        m = b[i + 1]
        n = int.from_bytes(b[i + 2:i + 4], "big")
        out.append((m, i, i + 2 + n))
        if m == 0xDA:
            break
        i += 2 + n
    return out


def without_app0(b):
    for m, s, e in _segments(b):
        if m == 0xE0:
            return b[:s] + b[e:]
    return b


def with_adobe(b, transform):
    seg = b"Adobe" + bytes([0, 100, 0, 0, 0, 0, transform])
    return b[:2] + b"\xff\xee" + (len(seg) + 2).to_bytes(2, "big") + seg + b[2:]


def with_component_ids(b, ids):
    """The frame's and the scan's component IDs replaced by `ids`."""
    b = bytearray(b)
    for m, s, e in _segments(bytes(b)):
        if m in (0xC0, 0xC1):
            for c in range(b[s + 9]):
                b[s + 10 + 3 * c] = ids[c]
        if m == 0xDA:
            for c in range(b[s + 4]):
                b[s + 5 + 2 * c] = ids[c]
    return bytes(b)


def with_sof_marker(b, marker):
    b = bytearray(b)
    for m, s, e in _segments(bytes(b)):
        if m in (0xC0, 0xC1):
            b[s + 1] = marker
    return bytes(b)


def with_precision(b, bits):
    b = bytearray(b)
    for m, s, e in _segments(bytes(b)):
        if m in (0xC0, 0xC1):
            b[s + 1] = 0xC1
            b[s + 4] = bits
    return bytes(b)


def with_first_scan_of_one_component(b):
    """The SOS rewritten to carry the first component only, as the first scan of a non-interleaved stream does."""
    for m, s, e in _segments(b):
        if m == 0xDA:
            sos = bytes([1, b[s + 5], b[s + 6], 0, 63, 0])
            return b[:s] + b"\xff\xda" + (len(sos) + 2).to_bytes(2, "big") + sos + b[e:]
    raise AssertionError("no SOS")


def with_four_components(b):
    """A SOF that declares a fourth component (CMYK / YCCK)."""
    for m, s, e in _segments(b):
        if m in (0xC0, 0xC1):
            sof = bytearray(b[s + 4:e])
            sof[5] = 4
            sof += bytes([4, 0x11, 0])
            return b[:s] + bytes([0xFF, m]) + (len(sof) + 2).to_bytes(2, "big") + bytes(sof) + b[e:]
    raise AssertionError("no SOF")


def refused_streams(img):
    """(stream, words expected in the reason) for every kind of stream the colour decoder refuses."""
    base = bytes(encode(img, 75, "420"))
    plain = without_app0(base)
    return [
        (bytes(cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1]), "progressive"),
        (with_sof_marker(base, 0xC9), "arithmetic"),
        (with_sof_marker(base, 0xC3), "lossless"),
        (with_precision(base, 12), "8-bit"),
        (with_first_scan_of_one_component(base), "non-interleaved"),
        (with_four_components(base), "CMYK"),
        (with_adobe(plain, 0), "Adobe transform 0"),
        (with_component_ids(plain, b"RGB"), "R G B"),
    ]


def accepted_variants(img):
    """Edited streams libjpeg still treats as YCbCr: JFIF wins over Adobe transform 0 and over R G B component IDs, Adobe
    transform 1 without JFIF, and no marker at all with the usual IDs."""
    base = bytes(encode(img, 75, "420"))
    plain = without_app0(base)
    return [with_adobe(base, 0), with_component_ids(base, b"RGB"), with_adobe(plain, 1), plain]
