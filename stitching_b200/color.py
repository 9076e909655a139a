"""BGR <-> YUV 4:2:0 on the device (sb_cvt_* in the C ABI), bit-exact to cv.cvtColor.

A YUV 4:2:0 frame is cv2's single-array layout: a uint8 (h * 3/2, w) array holding the h rows of Y, then
  "nv12": h/2 rows of interleaved U V (what NVDEC writes and NVENC reads),
  "i420": the h/2 x w/2 U plane, then the V plane, each packed contiguously (ffmpeg's yuv420p).
yuv420_to_bgr == cv.cvtColor(frame, COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) and bgr_to_yuv420(img, "i420") ==
cv.cvtColor(img, COLOR_BGR2YUV_I420); cv2 has no BGR -> NV12 code, so "nv12" is that result with U and V interleaved.
Widths and heights are even, as cv2 requires.
"""
import ctypes as C

import numpy as np

from . import _lib
from .stitching_error import StitchingError

FORMATS = ("bgr", "nv12", "i420")


def fmt_code(fmt):
    if fmt not in _lib.PIX_FMTS:
        raise StitchingError(f"unknown pixel format {fmt!r} (one of {', '.join(FORMATS)})")
    return _lib.PIX_FMTS[fmt]


def frame_shape(w, h, fmt):
    """Array shape of a w x h frame in `fmt`."""
    fmt_code(fmt)
    return (h, w, 3) if fmt == "bgr" else (h * 3 // 2, w)


def planes(arr, w, h, fmt, writable=False):
    """(plane pointers, plane pitches, array the pointers point into) of a w x h frame held in `arr` (C arrays of three
    entries each, the layout of the sb_pix_fmt entries).  Input frames that are not laid out as the entries need are
    copied; output frames (writable) must already be."""
    code = fmt_code(fmt)
    arr = np.asarray(arr) if not writable else arr
    shape = frame_shape(w, h, fmt)
    if not isinstance(arr, np.ndarray) or arr.dtype != np.uint8 or arr.shape != shape:
        raise StitchingError(f"expected a uint8 {fmt} frame of shape {shape}")
    if code == 0:
        dense = arr.strides[1:] == (3, 1)
    elif code == 1:
        dense = arr.strides[1] == 1
    else:
        dense = arr.flags.c_contiguous  # the U and V planes are packed into the rows after Y
    if not dense:
        if writable:
            raise StitchingError(f"the {fmt} output frame must be laid out like a C-contiguous array")
        arr = np.ascontiguousarray(arr)
    base, pitch = arr.ctypes.data, arr.strides[0]
    ptrs = (C.c_void_p * 3)()
    pitches = (C.c_size_t * 3)()
    ptrs[0], pitches[0] = base, pitch
    if code == 1:
        ptrs[1], pitches[1] = base + h * pitch, pitch
    elif code == 2:
        ptrs[1], pitches[1] = base + h * w, w // 2
        ptrs[2], pitches[2] = base + h * w + (w // 2) * (h // 2), w // 2
    return ptrs, pitches, arr


def yuv420_to_bgr(frame, fmt):
    """cv.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420) on the device: (h * 3/2, w) uint8 -> (h, w, 3) uint8."""
    if fmt not in ("nv12", "i420"):
        raise StitchingError(f"{fmt!r} is not a YUV 4:2:0 format")
    frame = np.asarray(frame)
    if frame.ndim != 2 or frame.shape[0] % 3:
        raise StitchingError("expected a 2-d (h * 3/2, w) uint8 YUV frame")
    w, h = frame.shape[1], frame.shape[0] // 3 * 2
    ptrs, pitches, frame = planes(frame, w, h, fmt)
    out = np.empty((h, w, 3), np.uint8)
    _lib.check(_lib.lib().sb_cvt_yuv420_to_bgr(fmt_code(fmt), ptrs, pitches, w, h, out.ctypes.data_as(C.c_void_p), out.strides[0]),
               "sb_cvt_yuv420_to_bgr")
    return out


def bgr_to_yuv420(img, fmt):
    """cv.cvtColor(img, COLOR_BGR2YUV_I420) on the device, chroma interleaved for "nv12": (h, w, 3) -> (h * 3/2, w)."""
    if fmt not in ("nv12", "i420"):
        raise StitchingError(f"{fmt!r} is not a YUV 4:2:0 format")
    img = np.asarray(img)
    if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3:
        raise StitchingError("expected a uint8 h x w x 3 image")
    if img.strides[1:] != (3, 1):
        img = np.ascontiguousarray(img)
    h, w = img.shape[:2]
    out = np.empty((h * 3 // 2, w), np.uint8)
    ptrs, pitches, _ = planes(out, w, h, fmt, writable=True)
    _lib.check(_lib.lib().sb_cvt_bgr_to_yuv420(fmt_code(fmt), img.ctypes.data_as(C.c_void_p), img.strides[0], w, h, ptrs, pitches),
               "sb_cvt_bgr_to_yuv420")
    return out
