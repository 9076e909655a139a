"""ctypes binding of libstitch_b200.so (include/stitch_b200.h).

There is no CPU fallback: if the CUDA library is missing or no sm_100 device is usable, importing the
binding works but the first call raises.  The library is built in-tree by `make -C stitching_b200/csrc`
(or `__graft_entry__.build()`).
"""
import ctypes as C
import os

from .stitching_error import StitchingError

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libstitch_b200.so")

SB_OK = 0
WARP_TYPES = {  # warper.py:10-27 -> sb_warp_type
    "spherical": 0, "cylindrical": 1, "plane": 2, "affine": 3, "fisheye": 4, "stereographic": 5,
    "compressedPlaneA2B1": 6, "compressedPlaneA1.5B1": 7, "compressedPlanePortraitA2B1": 8, "compressedPlanePortraitA1.5B1": 9,
    "paniniA2B1": 10, "paniniA1.5B1": 11, "paniniPortraitA2B1": 12, "paniniPortraitA1.5B1": 13,
    "mercator": 14, "transverseMercator": 15,
}
BLEND_KINDS = {"no": 0, "feather": 1, "multiband": 2}
PIX_FMTS = {"bgr": 0, "nv12": 1, "i420": 2}  # sb_pix_fmt

c_float_p = C.POINTER(C.c_float)
c_int_p = C.POINTER(C.c_int)
c_u8_p = C.POINTER(C.c_uint8)
c_s16_p = C.POINTER(C.c_int16)


class Rig(C.Structure):
    _fields_ = [
        ("n_images", C.c_int),
        ("warp_type", C.c_int),
        ("scale", C.c_float),
        ("blend_kind", C.c_int),
        ("blend_strength", C.c_float),
        ("src_w", c_int_p),
        ("src_h", c_int_p),
        ("K", c_float_p),
        ("R", c_float_p),
        ("mask_mode", C.c_int),
    ]


# every symbol include/stitch_b200.h declares: (name, restype, argtypes)
SIGNATURES = [
    ("sb_last_error", C.c_char_p, []),
    ("sb_version", C.c_char_p, []),
    ("sb_init", C.c_int, [C.c_int]),
    ("sb_device_info", C.c_int, [C.c_char_p, C.c_size_t, c_int_p, c_int_p, c_int_p]),
    ("sb_launch_count", C.c_ulonglong, []),
    ("sb_warp_roi", C.c_int, [C.c_int, C.c_float, c_float_p, c_float_p, C.c_int, C.c_int, c_int_p]),
    ("sb_warp", C.c_int, [C.c_int, C.c_float, c_float_p, c_float_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t,
                          C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, c_int_p]),
    ("sb_warp_keep", C.c_int, [C.c_int, C.c_float, c_float_p, c_float_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t,
                               C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, c_int_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    ("sb_devimg_release", None, [C.c_void_p]),
    ("sb_devimg_info", C.c_int, [C.c_void_p, c_int_p, c_int_p, c_int_p]),
    ("sb_gain_apply_dev", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int,
                                    C.c_int, C.c_void_p]),
    ("sb_blender_feed_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t,
                                      C.c_int, C.c_int, C.c_int, C.c_int]),
    ("sb_blender_create", C.c_void_p, [C.c_int, C.c_int, C.c_float]),
    ("sb_blender_destroy", None, [C.c_void_p]),
    ("sb_blender_prepare", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    ("sb_blender_num_bands", C.c_int, [C.c_void_p]),
    ("sb_blender_feed", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_int,
                                  C.c_int, C.c_int]),
    ("sb_blender_blend", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
    ("sb_compositor_create", C.c_void_p, [C.POINTER(Rig)]),
    ("sb_compositor_destroy", None, [C.c_void_p]),
    ("sb_compositor_geometry", C.c_int, [C.c_void_p, c_int_p, c_int_p, c_int_p]),
    ("sb_compositor_model_bytes", C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int]),
    ("sb_compositor_upload", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int]),
    ("sb_compositor_upload_frame", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int]),
    ("sb_compositor_download_frame", C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_void_p, C.c_size_t]),
    ("sb_compositor_submit_frames", C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int,
                                              C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_void_p, C.c_size_t,
                                              C.POINTER(C.c_ulonglong)]),
    ("sb_cvt_yuv420_to_bgr", C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    ("sb_cvt_bgr_to_yuv420", C.c_int, [C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    ("sb_compositor_set_mask", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    ("sb_compositor_set_seam_mask", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int]),
    ("sb_compositor_set_gain", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("sb_resize_exact", C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int]),
    ("sb_gain_apply", C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("sb_seam_resize", C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    ("sb_compositor_shard_axis", C.c_int, [C.c_void_p]),
    ("sb_compositor_run", C.c_int, [C.c_void_p]),
    ("sb_compositor_download", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
    ("sb_compositor_download_warped", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
    ("sb_compositor_sync", C.c_int, [C.c_void_p]),
    ("sb_compositor_submit", C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_void_p, C.c_size_t,
                                       C.c_void_p, C.c_size_t, C.POINTER(C.c_ulonglong)]),
    ("sb_compositor_wait", C.c_int, [C.c_void_p, C.c_ulonglong]),
    ("sb_compositor_time", C.c_int, [C.c_void_p, C.c_int, C.c_int, c_float_p]),
    ("sb_compositor_time_multi", C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, c_float_p]),
    ("sb_compositor_stage_times", C.c_int, [C.c_void_p, C.POINTER(C.c_char_p), c_float_p, C.c_int]),
    ("sb_compositor_create_sharded", C.c_void_p, [C.POINTER(Rig), C.c_int, C.c_int]),
    ("sb_compositor_shard_info", C.c_int, [C.c_void_p, c_int_p, c_int_p, c_int_p]),
    ("sb_compositor_shard_phase", C.c_int, [C.c_void_p, C.c_int]),
    ("sb_compositor_shard_slab", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    ("sb_device_copy", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    ("sb_selftest_division", C.c_int, [C.c_ulonglong, C.c_ulonglong, C.c_int, C.POINTER(C.c_ulonglong)]),
    ("sb_timelapse_frame", C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.POINTER(C.c_int), C.c_void_p, C.c_size_t]),
    ("sb_host_alloc", C.c_void_p, [C.c_size_t]),
    ("sb_host_free", None, [C.c_void_p]),
    ("sb_comm_unique_id", C.c_int, [c_u8_p]),
    ("sb_comm_init", C.c_int, [c_u8_p, C.c_int, C.c_int]),
    ("sb_comm_destroy", C.c_int, []),
]

_lib = None


def bind(path):
    """dlopen `path` and attach the prototypes of every exported entry."""
    L = C.CDLL(path)
    for name, res, args in SIGNATURES:
        fn = getattr(L, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    return L


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise StitchingError(
                f"{LIB_PATH} is missing: build it with `make -C stitching_b200/csrc` "
                "(stitching_b200 has no CPU fallback)"
            )
        _lib = bind(LIB_PATH)
    return _lib


def check(rc, what=""):
    if rc != SB_OK:
        msg = lib().sb_last_error().decode(errors="replace")
        raise StitchingError(f"libstitch_b200 {what} failed ({rc}): {msg}")
