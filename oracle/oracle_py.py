"""ctypes front-ends for the two CPU checkers -- TEST INFRASTRUCTURE ONLY.

  Port       -> oracle/libdmc_oracle.so   (plain-C restatement, oracle/dmc_oracle.c)
  Reference  -> oracle/_ref/libdmc_ref.so (unmodified reference sources through oracle/refshim)
  Shim       -> oracle/libdmc_shim.so     (oracle/refshim's cv:: stand-ins alone, no reference source)

Port and Reference expose the same numpy-level methods so a test can be parametrised over them.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module;
nothing in depthmapcompression_b200/ does.
"""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "libdmc_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libdmc_ref.so")
SHIM_SO = os.path.join(HERE, "libdmc_shim.so")

CV_8U, CV_16U, CV_16S, CV_32F, CV_64F = 0, 2, 3, 5, 6
FULL_KERNEL, FULL_KERNEL_PAIR, SEPARABLE_KERNEL = 0, 1, 2
FILL_DISPARITY, FILL_DEPTH = 0, 1

_DEPTH_OF = {np.dtype(np.uint8): CV_8U, np.dtype(np.uint16): CV_16U, np.dtype(np.int16): CV_16S,
             np.dtype(np.float32): CV_32F, np.dtype(np.float64): CV_64F}


def cvtype_of(a):
    cn = 1 if a.ndim == 2 else a.shape[2]
    return _DEPTH_OF[a.dtype] + ((cn - 1) << 3)


def build(force=False):
    """make -C oracle (the port always; the reference build only where /root/reference exists)."""
    if force or not os.path.exists(PORT_SO) or not os.path.exists(SHIM_SO) or (os.path.isdir("/root/reference") and not os.path.exists(REF_SO)):
        subprocess.check_call(["make", "-C", HERE, "all"], stdout=subprocess.DEVNULL)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _c(a, dtype=None):
    return np.ascontiguousarray(a, dtype=dtype)


class _Base:
    prefix = ""
    kind = ""

    def __init__(self, path):
        self.lib = C.CDLL(path)

    def _f(self, name):
        return getattr(self.lib, self.prefix + name)

    # ---- PostFilterSet ---------------------------------------------------------------------
    def post_filter_set(self, src, mr, gr, mmr, br, th, method=FULL_KERNEL):
        src = _c(src, np.uint8); H, W = src.shape; dst = np.zeros_like(src)
        rc = self._f("post_filter_set")(_p(src), _p(dst), H, W, mr, gr, mmr, br, int(th), method)
        assert rc >= 0, rc
        return dst

    def filter_disp8u_depth32f(self, src, focus, baseline, amp, mr, gr, mmr, br, th, method=FULL_KERNEL):
        src = _c(src, np.uint8); H, W = src.shape; dst = np.zeros((H, W), np.float32)
        rc = self._f("filter_disp8u_depth32f")(_p(src), _p(dst), H, W, C.c_double(focus), C.c_double(baseline), C.c_double(amp),
                                               mr, gr, mmr, br, C.c_float(th), method)
        assert rc >= 0, rc
        return dst

    def filter_disp8u_depth16u(self, src, focus, baseline, amp, mr, gr, mmr, br, th, method=FULL_KERNEL):
        src = _c(src, np.uint8); H, W = src.shape; dst = np.zeros((H, W), np.uint16)
        rc = self._f("filter_disp8u_depth16u")(_p(src), _p(dst), H, W, C.c_double(focus), C.c_double(baseline), C.c_double(amp),
                                               mr, gr, mmr, br, C.c_float(th), method)
        assert rc >= 0, rc
        return dst

    def filter_disp8u_disp32f(self, src, mr, gr, mmr, br, th, method=FULL_KERNEL):
        src = _c(src, np.uint8); H, W = src.shape; dst = np.zeros((H, W), np.uint16)
        rc = self._f("filter_disp8u_disp32f")(_p(src), _p(dst), H, W, mr, gr, mmr, br, C.c_float(th), method)
        assert rc >= 0, rc
        return dst

    # ---- converters ------------------------------------------------------------------------
    def _conv(self, name, src, sdt, ddt, fb, a, b, dst=None):
        src = _c(src, sdt); H, W = src.shape
        dst = np.zeros((H, W), ddt) if dst is None else _c(dst, ddt).copy()
        rc = self._f(name)(_p(src), _p(dst), H, W, C.c_float(fb), C.c_float(a), C.c_float(b))
        assert rc >= 0, rc
        return dst

    def disp8u2depth32f(self, src, fb, a=1.0, b=0.0, dst=None):
        return self._conv("disp8u2depth32f", src, np.uint8, np.float32, fb, a, b, dst)

    def depth32f2disp8u(self, src, fb, a=1.0, b=0.0):
        return self._conv("depth32f2disp8u", src, np.float32, np.uint8, fb, a, b)

    def depth16u2disp8u(self, src, fb, a=1.0, b=0.0):
        return self._conv("depth16u2disp8u", src, np.uint16, np.uint8, fb, a, b)

    def disp16s2depth16u(self, src, fb, a=1.0, b=0.0):
        return self._conv("disp16s2depth16u", src, np.int16, np.uint16, fb, a, b)

    def fill_occlusion(self, img, invalid=0, mode=FILL_DEPTH):
        img = _c(img).copy(); H, W = img.shape
        rc = self._f("fill_occlusion")(_p(img), H, W, cvtype_of(img), int(invalid), mode)
        assert rc >= 0, rc
        return img

    def reproject_xyz(self, depth, f):
        depth = _c(depth); H, W = depth.shape; xyz = np.zeros((H * W, 3), np.float32)
        rc = self._f("reproject_xyz")(_p(depth), _p(xyz), H, W, cvtype_of(depth), C.c_double(f))
        assert rc >= 0, rc
        return xyz


class Port(_Base):
    prefix = "orc_"
    kind = "port"

    def __init__(self):
        build()
        super().__init__(PORT_SO)

    def set_num_threads(self, n):
        self.lib.orc_set_num_threads(int(n))

    # ---- point-cloud render (SURVEY.md 8f-3) ------------------------------------------------
    def project_points(self, xyz, R, t, K, rcp=True):
        xyz = _c(xyz, np.float32).reshape(-1, 3); n = xyz.shape[0]; pt = np.zeros((n, 2), np.float32)
        R, t, K = _c(R, np.float64), _c(t, np.float64), _c(K, np.float64)
        assert self.lib.orc_project_points(_p(xyz), C.c_long(n), _p(R), _p(t), _p(K), _p(pt), int(bool(rcp))) == 0
        return pt

    def project_image(self, image, xyz, R, t, K, is_sub, rcp=True):
        """-> (dest 8UC3, depth 32F): the literal restatement of the reference's serial z-buffer splat."""
        image = _c(image, np.uint8); H, W = image.shape[:2]; xyz = _c(xyz, np.float32)
        R, t, K = _c(R, np.float64), _c(t, np.float64), _c(K, np.float64)
        dest = np.zeros((H, W, 3), np.uint8); depth = np.zeros((H, W), np.float32)
        fn = self.lib.orc_project_image_serial
        assert fn(_p(image), _p(xyz), H, W, _p(R), _p(t), _p(K), int(bool(is_sub)), int(bool(rcp)), _p(dest), _p(depth)) == 0
        return dest, depth

    def fill_small_hole(self, src, dst=None):
        src = _c(src, np.uint8); H, W = src.shape[:2]
        dst = src.copy() if dst is None else _c(dst, np.uint8).copy()
        assert self.lib.orc_fill_small_hole(_p(src), _p(dst), H, W) == 0
        return dst

    def median_blur(self, src, ksize):
        src = _c(src, np.uint8); H, W = src.shape; dst = np.zeros_like(src)
        assert self.lib.orc_median_blur_8u(_p(src), _p(dst), H, W, ksize) == 0
        return dst

    def gaussian_kernel32f(self, n, sigma):
        k = np.zeros(n, np.float32); self.lib.orc_gaussian_kernel32f(n, C.c_double(sigma), _p(k)); return k

    def gaussian_blur32f(self, src, d, sigma):
        src = _c(src, np.float32); H, W = src.shape; dst = np.zeros_like(src)
        assert self.lib.orc_gaussian_blur_32f(_p(src), _p(dst), H, W, d, C.c_double(sigma)) == 0
        return dst

    def small_gaussian(self, src, d, sigma):
        src = _c(src, np.uint8); H, W = src.shape; dst = np.zeros_like(src)
        assert self.lib.orc_small_gaussian_8u(_p(src), _p(dst), H, W, d, C.c_double(sigma)) == 0
        return dst

    def morph(self, src, k, is_max):
        src = _c(src); H, W = src.shape; dst = np.zeros_like(src)
        assert self.lib.orc_morph(_p(src), _p(dst), H, W, cvtype_of(src), k, k, int(is_max)) == 0
        return dst

    def bwrf(self, src, kw, kh, th, method=FULL_KERNEL, dst_init=None):
        src = _c(src); dst = np.zeros_like(src) if dst_init is None else _c(dst_init).copy()
        rc = self.lib.orc_bwrf(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), kw, kh, C.c_float(th), method)
        assert rc >= 0, rc
        return dst

    def joint_bwrf(self, src, guide, kw, kh, th):
        """extension without a reference counterpart (SURVEY 8f-4): weights from `guide`, average of the 8UC1 `src`"""
        src = _c(src, np.uint8); guide = _c(guide, np.uint8); dst = np.zeros_like(src)
        gcn = 1 if guide.ndim == 2 else guide.shape[2]
        rc = self.lib.orc_joint_bwrf(_p(src), _p(guide), _p(dst), src.shape[0], src.shape[1], gcn, kw, kh, C.c_float(th))
        assert rc >= 0, rc
        return dst

    def blur_remove_minmax(self, src, r):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.orc_blur_remove_minmax(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), r)
        assert rc >= 0, rc
        return dst

    def max_filter(self, src, kw, kh):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.orc_max_filter(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), kw, kh); assert rc >= 0
        return dst

    def min_filter(self, src, kw, kh):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.orc_min_filter(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), kw, kh); assert rc >= 0
        return dst

    def brf(self, src, kw, kh, frec, color, space):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.orc_brf(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), kw, kh,
                              C.c_float(frec), C.c_float(color), C.c_float(space))
        assert rc >= 0, rc
        return dst


class _ShimCalls:
    """The cv:: stand-ins of oracle/refshim/minicv.hpp (shim_* entry points)."""

    def median_blur(self, src, ksize):
        src = _c(src); H, W = src.shape; dst = np.zeros_like(src)
        assert self.lib.shim_median_blur(_p(src), _p(dst), H, W, cvtype_of(src), ksize) == 0
        return dst

    def gaussian_kernel32f(self, n, sigma):
        k = np.zeros(n, np.float32); self.lib.shim_gaussian_kernel32f(n, C.c_double(sigma), _p(k)); return k

    def gaussian_blur32f(self, src, d, sigma):
        src = _c(src, np.float32); H, W = src.shape; dst = np.zeros_like(src)
        assert self.lib.shim_gaussian_blur32f(_p(src), _p(dst), H, W, d, C.c_double(sigma)) == 0
        return dst

    def morph(self, src, k, is_max):
        src = _c(src); H, W = src.shape; dst = np.zeros_like(src)
        assert self.lib.shim_morph(_p(src), _p(dst), H, W, cvtype_of(src), k, int(is_max)) == 0
        return dst

    def copy_make_border(self, src, top, bottom, left, right, border):
        src = _c(src); H, W = src.shape[:2]
        dst = np.zeros((H + top + bottom, W + left + right) + src.shape[2:], src.dtype)
        assert self.lib.shim_copy_make_border(_p(src), _p(dst), H, W, cvtype_of(src), top, bottom, left, right, border) == 0
        return dst

    def convert_to(self, src, ddtype):
        src = _c(src); dst = np.zeros(src.shape, ddtype)
        dt = _DEPTH_OF[np.dtype(ddtype)] + (cvtype_of(src) & ~7)
        assert self.lib.shim_convert_to(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), dt) == 0
        return dst


class Reference(_Base, _ShimCalls):
    prefix = "ref_"
    kind = "reference"

    def __init__(self):
        build()
        if not os.path.exists(REF_SO):
            raise FileNotFoundError(REF_SO)
        super().__init__(REF_SO)

    @staticmethod
    def available():
        return os.path.exists(REF_SO) or os.path.isdir("/root/reference")

    def set_num_threads(self, n):
        self.lib.ref_set_num_threads(int(n))

    # ---- point-cloud render: the reference itself (_mm_rcp_ps projection, serial z-buffer) ----
    def project_points(self, xyz, R, t, K):
        xyz = _c(xyz, np.float32).reshape(-1, 3); n = xyz.shape[0]; pt = np.zeros((n, 2), np.float32)
        R, t, K = _c(R, np.float64), _c(t, np.float64), _c(K, np.float64)
        assert self.lib.ref_project_points(_p(xyz), n, _p(R), _p(t), _p(K), _p(pt)) == 0
        return pt

    def project_image(self, image, xyz, R, t, K, is_sub):
        image = _c(image, np.uint8); H, W = image.shape[:2]; xyz = _c(xyz, np.float32)
        R, t, K = _c(R, np.float64), _c(t, np.float64), _c(K, np.float64)
        dest = np.zeros((H, W, 3), np.uint8); depth = np.zeros((H, W), np.float32)
        assert self.lib.ref_project_image_from_xyz(_p(image), _p(xyz), H, W, _p(R), _p(t), _p(K), int(bool(is_sub)), _p(dest), _p(depth)) == 0
        return dest, depth

    def fill_small_hole(self, src, dst=None):
        src = _c(src, np.uint8); H, W = src.shape[:2]
        out = src.copy() if dst is None else _c(dst, np.uint8).copy()
        assert self.lib.ref_fill_small_hole(_p(src), _p(out), H, W, int(dst is None)) == 0
        return out

    def small_gaussian(self, src, d, sigma):
        src = _c(src); H, W = src.shape; dst = np.zeros_like(src)
        assert self.lib.ref_small_gaussian(_p(src), _p(dst), H, W, cvtype_of(src), d, C.c_double(sigma)) == 0
        return dst

    def bwrf(self, src, kw, kh, th, method=FULL_KERNEL, dst_init=None, inplace=False):
        src = _c(src); dst = np.zeros_like(src) if dst_init is None else _c(dst_init).copy()
        rc = self.lib.ref_bwrf(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), kw, kh, C.c_float(th), method, int(inplace))
        assert rc >= 0, rc
        return dst

    def blur_remove_minmax(self, src, r, inplace=False):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.ref_blur_remove_minmax(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), r, int(inplace))
        assert rc >= 0, rc
        return dst

    def blur_remove_minmax_base(self, src, r):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.ref_blur_remove_minmax_base(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), r); assert rc >= 0
        return dst

    def max_filter(self, src, kw, kh):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.ref_max_filter(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), kw, kh); assert rc >= 0
        return dst

    def min_filter(self, src, kw, kh):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.ref_min_filter(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), kw, kh); assert rc >= 0
        return dst

    def brf(self, src, kw, kh, frec, color, space, inplace=False):
        src = _c(src); dst = np.zeros_like(src)
        rc = self.lib.ref_brf(_p(src), _p(dst), src.shape[0], src.shape[1], cvtype_of(src), kw, kh,
                              C.c_float(frec), C.c_float(color), C.c_float(space), int(inplace))
        assert rc >= 0, rc
        return dst


class Shim(_ShimCalls):
    """The stand-ins alone (oracle/libdmc_shim.so): built from oracle/refshim without the reference sources."""

    def __init__(self):
        build()
        self.lib = C.CDLL(SHIM_SO)


def synth_disp(H, W, seed, shift=(0, 0)):
    """Deterministic piecewise-smooth disparity map (SURVEY.md 8d): smooth base + 16 rectangles, in [1,255]."""
    rs = np.random.RandomState(seed)
    x = np.arange(W, dtype=np.float64)[None, :]; y = np.arange(H, dtype=np.float64)[:, None]
    img = 90 + 40 * np.sin(x / (W / 6.0)) + 30 * np.cos(y / (H / 5.0))
    for _ in range(16):
        w = rs.randint(max(1, W // 24), max(2, W // 6) + 1); h = rs.randint(max(1, H // 24), max(2, H // 4) + 1)
        v = rs.randint(30, 250); x0 = (rs.randint(0, W) + shift[0]) % W; y0 = (rs.randint(0, H) + shift[1]) % H
        img[y0:y0 + h, x0:x0 + w] = v
    return np.clip(np.rint(img), 1, 255).astype(np.uint8)


def degrade_blocks(img, seed, amp=6):
    """Cheap deterministic stand-in for codec distortion (no encoder on the GPU box): 8x8 block-wise
    quantisation noise + ringing-like +-amp noise near edges."""
    rs = np.random.RandomState(seed)
    H, W = img.shape
    noise = rs.randint(-amp, amp + 1, size=(H, W)).astype(np.int16)
    blk = rs.randint(-2, 3, size=((H + 7) // 8, (W + 7) // 8)).astype(np.int16)
    blk = np.kron(blk, np.ones((8, 8), np.int16))[:H, :W]
    gx = np.abs(np.diff(img.astype(np.int16), axis=1, prepend=img[:, :1].astype(np.int16)))
    gy = np.abs(np.diff(img.astype(np.int16), axis=0, prepend=img[:1, :].astype(np.int16)))
    edge = ((gx + gy) > 8)
    k = np.ones((5, 5), np.uint8)
    try:
        import cv2
        edge = cv2.dilate(edge.astype(np.uint8), k) > 0
    except Exception:
        pass
    out = img.astype(np.int16) + blk + np.where(edge, noise, noise // 3)
    return np.clip(out, 1, 255).astype(np.uint8)
