"""ctypes binding of include/dmc_c.h (libdmc_b200.so).  Thin: every function here is one C-ABI call.

The library is CUDA-only.  Importing this module never falls back to anything: a missing .so raises at import
time, a missing GPU raises at Context() creation.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdmc_b200.so")

DMC_OK, DMC_UNSUPPORTED = 0, 1
DMC_ERR_TYPE, DMC_ERR_SIZE, DMC_ERR_CUDA, DMC_ERR_ARG = -1, -2, -3, -4
MEM_HOST, MEM_DEVICE = 0, 1
JPEG_OPTIMIZE_HUFFMAN = 1
DMC_JPEG_SAMPLING_444, DMC_JPEG_SAMPLING_422, DMC_JPEG_SAMPLING_420, DMC_JPEG_SAMPLING_440, DMC_JPEG_SAMPLING_411 = 0x111111, 0x211111, 0x221111, 0x121111, 0x411111
CV_8U, CV_16U, CV_16S, CV_32F, CV_64F = 0, 2, 3, 5, 6
FULL_KERNEL, FULL_KERNEL_PAIR, SEPARABLE_KERNEL = 0, 1, 2       # filter.h:23-28
FILL_DISPARITY, FILL_DEPTH = 0, 1                               # util.h:19-23
BORDER_REPLICATE = 1
CHAIN_DISP8U, CHAIN_DEPTH32F, CHAIN_DEPTH16U, CHAIN_DISP32F = 0, 1, 2, 3
STAGE_MEDIAN, STAGE_GAUSS, STAGE_MINMAX, STAGE_RANGE = 0, 1, 2, 3
STAGE_NAMES = ["median", "gauss", "minmax", "range"]

EXPORTS = [
    "dmc_version", "dmc_device_count", "dmc_create", "dmc_destroy", "dmc_last_error", "dmc_set_stream", "dmc_get_stream",
    "dmc_synchronize", "dmc_kernel_launches", "dmc_host_alloc", "dmc_host_free", "dmc_host_register", "dmc_host_unregister", "dmc_profile_enable", "dmc_profile_read", "dmc_set_lanes",
    "dmc_post_filter_set", "dmc_filter_disp8u_depth32f", "dmc_filter_disp8u_depth16u", "dmc_filter_disp8u_disp32f",
    "dmc_chain_batch", "dmc_chain_batch_images", "dmc_multi_chain_batch", "dmc_sched_create", "dmc_sched_destroy", "dmc_sched_device_count", "dmc_sched_last_error", "dmc_sched_chain_batch", "dmc_shard_frames", "dmc_jpeg_decode_gray_batch",
    "dmc_bwrf", "dmc_joint_bwrf", "dmc_blur_remove_minmax", "dmc_max_filter", "dmc_min_filter", "dmc_boundary_reconstruction", "dmc_minmax_boundary_reconstruction",
    "dmc_small_gaussian", "dmc_median_blur",
    "dmc_disp8u2depth32f", "dmc_depth32f2disp8u", "dmc_depth16u2disp8u", "dmc_disp16s2depth16u",
    "dmc_fill_occlusion", "dmc_reproject_xyz", "dmc_transpose",
    "dmc_chain_batch_jpeg", "dmc_jpeg_probe", "dmc_jpeg_decode_color_batch", "dmc_jpeg_probe_color", "dmc_jpeg_encode_bound", "dmc_jpeg_encode_gray_batch", "dmc_jpeg_degrade_gray_batch", "dmc_jpeg_encode_bound_ex", "dmc_jpeg_encode_gray_batch_ex", "dmc_jpeg_degrade_gray_batch_ex", "dmc_jpeg_encode_color_bound", "dmc_jpeg_encode_color_batch", "dmc_jpeg_degrade_color_batch", "dmc_split_bgr_line_interleave", "dmc_project_points", "dmc_project_image_from_xyz", "dmc_fill_small_hole", "dmc_hostlink_probe", "dmc_release_device", "dmc_set_gateway", "dmc_get_gateway", "dmc_sched_get_routing",
    "dmc_sse_gray_batch", "dmc_psnr_from_sse", "dmc_jpeg_rd_sweep", "dmc_jpeg_view_rd_sweep",
    "dmc_brf_batch", "dmc_jpeg_rd_sweep_ex", "dmc_jpeg_view_rd_sweep_ex",
    "dmc_prepare_disp_batch", "dmc_render_view_batch",
    "dmc_ssim_batch", "dmc_jpeg_rd_sweep_ssim", "dmc_jpeg_view_rd_sweep_ssim",
]
MAX_DEVICES = 16
RENDER_EXACT_DIVIDE = 1


class DmcImage(C.Structure):
    _fields_ = [("data", C.c_void_p), ("rows", C.c_int), ("cols", C.c_int), ("cvtype", C.c_int),
                ("step", C.c_size_t), ("mem", C.c_int)]


class DmcChainParams(C.Structure):
    _fields_ = [("chain", C.c_int), ("median_r", C.c_int), ("gaussian_r", C.c_int), ("minmax_r", C.c_int),
                ("brange_r", C.c_int), ("brange_th", C.c_float), ("brange_method", C.c_int),
                ("focus", C.c_double), ("baseline", C.c_double), ("amp", C.c_double)]


class DmcBrfParams(C.Structure):
    _fields_ = [("kernel_w", C.c_int), ("kernel_h", C.c_int), ("frec", C.c_float), ("color", C.c_float), ("space", C.c_float)]


class DmcHostlinkInfo(C.Structure):
    _fields_ = [("n_devices", C.c_int), ("device", C.c_int * 16), ("gateway", C.c_int * 16), ("loaded_gbs", C.c_double * 16),
                ("all_gbs", C.c_double), ("best_gbs", C.c_double), ("n_link", C.c_int)]


class DmcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libdmc_b200 error %d: %s" % (code, msg))
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: build it with `python build_native.py` "
                          "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    P, I, F, D = C.c_void_p, C.c_int, C.c_float, C.c_double
    IMG = C.POINTER(DmcImage)
    sig = {
        "dmc_version": (I, []), "dmc_device_count": (I, []),
        "dmc_create": (I, [I, C.POINTER(P)]), "dmc_destroy": (None, [P]), "dmc_last_error": (C.c_char_p, [P]),
        "dmc_set_stream": (I, [P, P]), "dmc_get_stream": (P, [P]), "dmc_synchronize": (I, [P]),
        "dmc_kernel_launches": (C.c_uint64, [P]), "dmc_host_alloc": (P, [C.c_size_t]), "dmc_host_free": (None, [P]), "dmc_host_register": (I, [P, C.c_size_t]), "dmc_host_unregister": (I, [P]),
        "dmc_profile_enable": (I, [P, I]), "dmc_set_lanes": (I, [P, I]),
        "dmc_profile_read": (I, [P, I, C.POINTER(D), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), I]),
        "dmc_post_filter_set": (I, [P, IMG, IMG, I, I, I, I, I, I]),
        "dmc_filter_disp8u_depth32f": (I, [P, IMG, IMG, D, D, D, I, I, I, I, F, I]),
        "dmc_filter_disp8u_depth16u": (I, [P, IMG, IMG, D, D, D, I, I, I, I, F, I]),
        "dmc_filter_disp8u_disp32f": (I, [P, IMG, IMG, I, I, I, I, F, I]),
        "dmc_chain_batch": (I, [P, P, P, I, I, I, C.POINTER(DmcChainParams), I]),
        "dmc_chain_batch_images": (I, [P, C.POINTER(DmcImage), C.POINTER(DmcImage), I, C.POINTER(DmcChainParams)]),
        "dmc_shard_frames": (I, [I, I, I, C.POINTER(I), C.POINTER(I)]),
        "dmc_jpeg_decode_gray_batch": (I, [P, P, P, I, I, I, P, I]),
        "dmc_chain_batch_jpeg": (I, [P, P, P, I, I, I, P, I, C.POINTER(DmcChainParams)]),
        "dmc_jpeg_probe": (I, [P, C.c_size_t, C.POINTER(I), C.POINTER(I), C.c_char_p, C.c_size_t]),
        "dmc_jpeg_decode_color_batch": (I, [P, P, P, I, I, I, P, I]),
        "dmc_jpeg_probe_color": (I, [P, C.c_size_t, C.POINTER(I), C.POINTER(I), C.POINTER(I), C.c_char_p, C.c_size_t]),
        "dmc_jpeg_encode_bound": (I, [I, I, C.POINTER(C.c_uint64)]),
        "dmc_jpeg_encode_gray_batch": (I, [P, P, I, I, I, I, I, P, I, C.c_uint64, C.POINTER(C.c_uint64)]),
        "dmc_jpeg_degrade_gray_batch": (I, [P, P, P, I, I, I, I, I, C.POINTER(C.c_uint64)]),
        "dmc_jpeg_encode_bound_ex": (I, [I, I, I, C.POINTER(C.c_uint64)]),
        "dmc_jpeg_encode_gray_batch_ex": (I, [P, P, I, I, I, I, I, I, P, I, C.c_uint64, C.POINTER(C.c_uint64)]),
        "dmc_jpeg_degrade_gray_batch_ex": (I, [P, P, P, I, I, I, I, I, I, C.POINTER(C.c_uint64)]),
        "dmc_jpeg_encode_color_bound": (I, [I, I, I, C.POINTER(C.c_uint64)]),
        "dmc_jpeg_encode_color_batch": (I, [P, P, I, I, I, I, I, I, P, I, C.c_uint64, C.POINTER(C.c_uint64)]),
        "dmc_jpeg_degrade_color_batch": (I, [P, P, P, I, I, I, I, I, I, C.POINTER(C.c_uint64)]),
        "dmc_sse_gray_batch": (I, [P, P, P, I, I, I, I, C.POINTER(C.c_uint64)]),
        "dmc_psnr_from_sse": (D, [C.c_uint64, C.c_uint64]),
        "dmc_jpeg_rd_sweep": (I, [P, P, I, I, I, I, C.POINTER(I), I, I, C.POINTER(DmcChainParams), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "dmc_jpeg_view_rd_sweep": (I, [P, P, P, I, I, I, I, C.POINTER(I), I, I, C.POINTER(DmcChainParams), D, C.POINTER(D), C.POINTER(D), I, C.POINTER(D), I, I,
                                       C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "dmc_brf_batch": (I, [P, P, P, I, I, I, I, C.POINTER(DmcBrfParams), I]),
        "dmc_jpeg_rd_sweep_ex": (I, [P, P, I, I, I, I, C.POINTER(I), I, I, C.POINTER(DmcChainParams), C.POINTER(DmcBrfParams),
                                     C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "dmc_jpeg_view_rd_sweep_ex": (I, [P, P, P, I, I, I, I, C.POINTER(I), I, I, C.POINTER(DmcChainParams), C.POINTER(DmcBrfParams), D, C.POINTER(D),
                                          C.POINTER(D), I, C.POINTER(D), I, I, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                          C.POINTER(C.c_uint64)]),
        "dmc_ssim_batch": (I, [P, P, P, I, I, I, I, I, C.POINTER(D)]),
        "dmc_jpeg_rd_sweep_ssim": (I, [P, P, I, I, I, I, C.POINTER(I), I, I, C.POINTER(DmcChainParams), C.POINTER(DmcBrfParams),
                                       C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                       C.POINTER(D), C.POINTER(D), C.POINTER(D)]),
        "dmc_jpeg_view_rd_sweep_ssim": (I, [P, P, P, I, I, I, I, C.POINTER(I), I, I, C.POINTER(DmcChainParams), C.POINTER(DmcBrfParams), D, C.POINTER(D),
                                            C.POINTER(D), I, C.POINTER(D), I, I, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                            C.POINTER(C.c_uint64), C.POINTER(D), C.POINTER(D), C.POINTER(D)]),
        "dmc_sched_create": (I, [C.POINTER(I), I, C.POINTER(P)]), "dmc_sched_destroy": (None, [P]), "dmc_sched_device_count": (I, [P]),
        "dmc_sched_last_error": (C.c_char_p, [P]), "dmc_sched_chain_batch": (I, [P, P, P, I, I, I, C.POINTER(DmcChainParams)]),
        "dmc_multi_chain_batch": (I, [C.POINTER(I), I, P, P, I, I, I, C.POINTER(DmcChainParams), C.c_char_p, C.c_size_t]),
        "dmc_bwrf": (I, [P, IMG, IMG, I, I, F, I, I]),
        "dmc_joint_bwrf": (I, [P, IMG, IMG, IMG, I, I, F, I]),
        "dmc_blur_remove_minmax": (I, [P, IMG, IMG, I]),
        "dmc_max_filter": (I, [P, IMG, IMG, I, I, I]), "dmc_min_filter": (I, [P, IMG, IMG, I, I, I]),
        "dmc_boundary_reconstruction": (I, [P, IMG, IMG, I, I, F, F, F]),
        "dmc_minmax_boundary_reconstruction": (I, [P, IMG, IMG, I, I, I, F, F, F]),
        "dmc_small_gaussian": (I, [P, IMG, IMG, I, D]), "dmc_median_blur": (I, [P, IMG, IMG, I]),
        "dmc_disp8u2depth32f": (I, [P, IMG, IMG, F, F, F]), "dmc_depth32f2disp8u": (I, [P, IMG, IMG, F, F, F]),
        "dmc_depth16u2disp8u": (I, [P, IMG, IMG, F, F, F]), "dmc_disp16s2depth16u": (I, [P, IMG, IMG, F, F, F]),
        "dmc_project_points": (I, [P, IMG, C.POINTER(D), C.POINTER(D), C.POINTER(D), IMG, I]),
        "dmc_project_image_from_xyz": (I, [P, IMG, IMG, IMG, C.POINTER(D), C.POINTER(D), C.POINTER(D), I, IMG, IMG, I]),
        "dmc_fill_small_hole": (I, [P, IMG, IMG]), "dmc_split_bgr_line_interleave": (I, [P, IMG, IMG]),
        "dmc_hostlink_probe": (I, [C.POINTER(I), I, C.POINTER(DmcHostlinkInfo)]), "dmc_release_device": (I, [I]), "dmc_set_gateway": (I, [P, I]), "dmc_get_gateway": (I, [P]),
        "dmc_sched_get_routing": (I, [P, C.POINTER(I), C.POINTER(D), C.POINTER(D)]),
        "dmc_prepare_disp_batch": (I, [P, P, P, I, I, I, F, F, F, I, I]),
        "dmc_render_view_batch": (I, [P, P, I, P, I, I, I, I, D, C.POINTER(D), C.POINTER(D), I, C.POINTER(D), I, I, P]),
        "dmc_fill_occlusion": (I, [P, IMG, I, I]), "dmc_reproject_xyz": (I, [P, IMG, IMG, D]), "dmc_transpose": (I, [P, IMG, IMG]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def shard_frames(n_frames, rank, world):
    b, c = C.c_int(), C.c_int()
    rc = lib.dmc_shard_frames(n_frames, rank, world, C.byref(b), C.byref(c))
    if rc != DMC_OK:
        raise DmcError(rc, "dmc_shard_frames: bad arguments")
    return b.value, c.value
