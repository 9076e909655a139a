"""Independent restatement of cv.cvtColor between BGR and YUV 4:2:0 (the checker of stitching_b200/csrc/sb_yuv.cu).

OpenCV's fixed-point closed forms, written out per pixel in int64 numpy (no shared code with the kernels):
  COLOR_YUV2BGR_NV12 / _I420   y = max(0, Y - 16) * 1220542, u = U - 128, v = V - 128, H = 1 << 19
                               R = sat8((y + H + 1673527 v) >> 20)
                               G = sat8((y + H - 852492 v - 409993 u) >> 20)
                               B = sat8((y + H + 2116026 u) >> 20)
                               each 2 x 2 block of Y pixels shares one (U, V)
  COLOR_BGR2YUV_I420           Y = sat8((269484 R + 528482 G + 102760 B + H + (16 << 20)) >> 20) for every pixel
                               U = sat8((-155188 R - 305135 G + 460324 B + H + (128 << 20)) >> 20)
                               V = sat8((460324 R - 385875 G - 74448 B + H + (128 << 20)) >> 20)
                               from the TOP-LEFT pixel of each 2 x 2 block (no averaging)
Frames are cv2's single-array layout, uint8 (h * 3/2, w): Y rows, then interleaved UV rows (NV12) or the U plane followed
by the V plane, each h/2 x w/2 and packed contiguously (I420).  NV12 output is the I420 result with U and V interleaved
(cv2 has no BGR -> NV12 code).  Odd widths or heights raise ValueError, as cv2 rejects them.
"""
import numpy as np

H = 1 << 19


def _sat8(v):
    return np.clip(v, 0, 255).astype(np.uint8)


def _check_size(w, h):
    if w <= 0 or h <= 0 or w % 2 or h % 2:
        raise ValueError(f"YUV 4:2:0 needs an even width and height, got {w}x{h}")


def split(frame, fmt):
    """(Y, U, V) planes of a (h * 3/2, w) frame: Y h x w, U and V h/2 x w/2."""
    frame = np.asarray(frame, np.uint8)
    if frame.ndim != 2 or frame.shape[0] % 3:
        raise ValueError(f"expected a (h * 3/2, w) frame, got {frame.shape}")
    h, w = frame.shape[0] // 3 * 2, frame.shape[1]
    _check_size(w, h)
    y = frame[:h]
    if fmt == "nv12":
        uv = frame[h:].reshape(h // 2, w // 2, 2)
        return y, uv[..., 0], uv[..., 1]
    if fmt == "i420":
        chroma = frame[h:].reshape(-1)
        q = (h // 2) * (w // 2)
        return y, chroma[:q].reshape(h // 2, w // 2), chroma[q:].reshape(h // 2, w // 2)
    raise ValueError(f"unknown YUV format {fmt!r}")


def join(y, u, v, fmt):
    """The (h * 3/2, w) frame of planes Y (h x w), U and V (h/2 x w/2)."""
    h, w = y.shape
    if fmt == "nv12":
        chroma = np.stack([u, v], axis=-1).reshape(h // 2, w)
    elif fmt == "i420":
        chroma = np.concatenate([u.reshape(-1), v.reshape(-1)]).reshape(h // 2, w)
    else:
        raise ValueError(f"unknown YUV format {fmt!r}")
    return np.ascontiguousarray(np.concatenate([y, chroma], axis=0), np.uint8)


def yuv420_to_bgr(frame, fmt):
    """cv.cvtColor(frame, COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420): (h * 3/2, w) -> (h, w, 3)."""
    Y, U, V = split(frame, fmt)
    y = np.maximum(Y.astype(np.int64) - 16, 0) * 1220542
    u = np.repeat(np.repeat(U.astype(np.int64) - 128, 2, axis=0), 2, axis=1)
    v = np.repeat(np.repeat(V.astype(np.int64) - 128, 2, axis=0), 2, axis=1)
    r = _sat8((y + H + 1673527 * v) >> 20)
    g = _sat8((y + H - 852492 * v - 409993 * u) >> 20)
    b = _sat8((y + H + 2116026 * u) >> 20)
    return np.stack([b, g, r], axis=-1)


def bgr_to_yuv420(img, fmt):
    """cv.cvtColor(img, COLOR_BGR2YUV_I420), chroma interleaved for "nv12": (h, w, 3) -> (h * 3/2, w)."""
    img = np.asarray(img, np.uint8)
    if img.ndim != 3 or img.shape[2] != 3:
        raise ValueError(f"expected an h x w x 3 image, got {img.shape}")
    h, w = img.shape[:2]
    _check_size(w, h)
    b, g, r = (img[..., k].astype(np.int64) for k in range(3))
    Y = _sat8((269484 * r + 528482 * g + 102760 * b + H + (16 << 20)) >> 20)
    b0, g0, r0 = b[::2, ::2], g[::2, ::2], r[::2, ::2]
    U = _sat8((-155188 * r0 - 305135 * g0 + 460324 * b0 + H + (128 << 20)) >> 20)
    V = _sat8((460324 * r0 - 385875 * g0 - 74448 * b0 + H + (128 << 20)) >> 20)
    return join(Y, U, V, fmt)


def exhaustive_frame(fmt):
    """One 4096 x 4096 frame holding every (Y, U, V) triple exactly once: block k of the 2^22 2 x 2 blocks (row-major) has
    (U, V) = (k & 255, (k >> 8) & 255) and the four Y values 4 (k >> 16) + 0..3."""
    n = 4096
    k = np.arange((n // 2) * (n // 2), dtype=np.int64).reshape(n // 2, n // 2)
    U, V = (k & 255).astype(np.uint8), ((k >> 8) & 255).astype(np.uint8)
    y0 = 4 * (k >> 16)
    Y = np.empty((n, n), np.uint8)
    Y[0::2, 0::2], Y[0::2, 1::2], Y[1::2, 0::2], Y[1::2, 1::2] = y0, y0 + 1, y0 + 2, y0 + 3
    return join(Y, U, V, fmt)
