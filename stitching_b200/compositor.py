"""Fused warp + blend on one B200 with every intermediate resident in HBM (sb_compositor_* in the C ABI).

Equivalent to running, for a fixed rig, stitcher.py:178-189 (Warper.warp_images / create_and_warp_masks /
warp_rois at final resolution) and stitcher.py:241-259 (Blender.prepare / feed / blend) -- with the warped
validity mask as blend mask (seam finder "no") -- but with one host->device copy of the sources and one
device->host copy of the panorama.
"""
import ctypes as C
from statistics import median

import numpy as np

from . import _lib, color
from .stitching_error import StitchingError
from .warper import Warper


def time_multi(compositors, iters):
    """Device time (ms) of `iters` steps dealt round-robin to several compositors of the same rig (batches in flight)."""
    n = len(compositors)
    arr = (C.c_void_p * n)(*[c._c for c in compositors])
    ms = C.c_float()
    _lib.check(_lib.lib().sb_compositor_time_multi(arr, n, int(iters), C.byref(ms)), "sb_compositor_time_multi")
    return ms.value


class Compositor:
    def __init__(self, cameras, sizes, warper_type="spherical", blender_type="multiband", blend_strength=5, scale=None,
                 aspect=1, rank=0, world=1):
        """cameras: objects with .focal, .K(), .R (cv.detail.CameraParams or rigs.Camera); sizes: [(w, h)].

        world > 1: one panorama over `world` GPUs, one process per GPU.  Every rank passes ALL cameras; rank r owns
        images [r*n/world, (r+1)*n/world) -- `self.first`, `self.count` -- uploads only those and gets the column
        strip `self.strip` = (lo, hi) of the panorama back (stitching_b200.dist.init_comm must have run)."""
        n = len(cameras)
        if n == 0 or len(sizes) != n:
            raise StitchingError("Compositor needs one size per camera")
        if warper_type not in _lib.WARP_TYPES:
            raise StitchingError(f"warper type '{warper_type}' is not on the B200 path")
        if blender_type not in _lib.BLEND_KINDS:
            raise StitchingError(f"unknown blender type '{blender_type}'")
        self.n = n
        self.sizes = [(int(w), int(h)) for w, h in sizes]
        if scale is None:
            scale = median([cam.focal for cam in cameras])  # Warper.set_scale
        self.scale = scale * aspect
        self._K = np.ascontiguousarray(np.stack([Warper.get_K(c, aspect) for c in cameras]).astype(np.float32))
        self._R = np.ascontiguousarray(np.stack([np.asarray(c.R, np.float32) for c in cameras]))
        self._w = (C.c_int * n)(*[s[0] for s in self.sizes])
        self._h = (C.c_int * n)(*[s[1] for s in self.sizes])
        rig = _lib.Rig(n, _lib.WARP_TYPES[warper_type], np.float32(self.scale), _lib.BLEND_KINDS[blender_type],
                       np.float32(blend_strength), self._w, self._h, self._K.ctypes.data_as(_lib.c_float_p),
                       self._R.ctypes.data_as(_lib.c_float_p), 0)
        L = _lib.lib()
        self.rank, self.world = int(rank), int(world)
        if self.world > 1:
            self._c = L.sb_compositor_create_sharded(C.byref(rig), self.rank, self.world)
        else:
            self._c = L.sb_compositor_create(C.byref(rig))
        if not self._c:
            _lib.check(-1, "sb_compositor_create")
        rects = (C.c_int * (4 * n))()
        roi = (C.c_int * 4)()
        nb = C.c_int()
        _lib.check(L.sb_compositor_geometry(self._c, rects, roi, C.byref(nb)), "sb_compositor_geometry")
        self.rects = [tuple(rects[4 * i: 4 * i + 4]) for i in range(n)]
        self.roi = tuple(roi)
        self.num_bands = nb.value
        self._pinned = []
        first, count, strip = C.c_int(), C.c_int(), (C.c_int * 2)()
        _lib.check(L.sb_compositor_shard_info(self._c, C.byref(first), C.byref(count), strip), "sb_compositor_shard_info")
        self.first, self.count, self.strip = first.value, count.value, (strip[0], strip[1])
        self.strip_axis = int(L.sb_compositor_shard_axis(self._c))  # 0: self.strip are columns of the panorama, 1: rows

    # -- data movement ---------------------------------------------------------------------------
    def upload(self, images, pinned=False, fmt="bgr"):
        """images: the frames of THIS rank's block, in order (all n frames when world == 1).

        fmt "nv12" / "i420": YUV 4:2:0 frames as (h * 3/2, w) uint8 arrays (stitching_b200.color), converted to BGR on the
        device exactly as cv.cvtColor does (single-GPU compositors, even frame sizes)."""
        L = _lib.lib()
        if len(images) != self.count:
            raise StitchingError(f"expected {self.count} images (block {self.first}..{self.first + self.count - 1}), got {len(images)}")
        if fmt != "bgr":
            code = color.fmt_code(fmt)
            for i, img in enumerate(images, start=self.first):
                ptrs, pitches, _keep = color.planes(img, self.sizes[i][0], self.sizes[i][1], fmt)
                _lib.check(L.sb_compositor_upload_frame(self._c, i, code, ptrs, pitches, int(pinned)), "sb_compositor_upload_frame")
            return
        for i, img in enumerate(images, start=self.first):
            img = np.asarray(img)
            if img.dtype != np.uint8 or img.shape != (self.sizes[i][1], self.sizes[i][0], 3):
                raise StitchingError(f"image {i}: expected uint8 {self.sizes[i][1]}x{self.sizes[i][0]}x3")
            if img.strides[2] != 1 or img.strides[1] != 3:
                img = np.ascontiguousarray(img)
            _lib.check(L.sb_compositor_upload(self._c, i, img.ctypes.data_as(C.c_void_p), img.strides[0], int(pinned)),
                       "sb_compositor_upload")

    def set_mask(self, i, mask):
        """Blend mask of image i in warped coordinates (uint8 h' x w', e.g. SeamFinder.resize's output); replaces the
        warped validity mask as blend weight from the next run on."""
        if hasattr(mask, "get") and not isinstance(mask, np.ndarray):
            mask = mask.get()
        mask = np.ascontiguousarray(mask, np.uint8)
        if mask.shape != (self.rects[i][3], self.rects[i][2]):
            raise StitchingError(f"mask {i}: expected {self.rects[i][3]}x{self.rects[i][2]}")
        _lib.check(_lib.lib().sb_compositor_set_mask(self._c, i, mask.ctypes.data_as(C.c_void_p), mask.strides[0]),
                   "sb_compositor_set_mask")

    def set_gain(self, i, gain):
        """Exposure gain of image i (one entry of a fed cv.detail compensator's getMatGains(): float32 map of 1 or 3
        channels, float64 scalar or vector; None removes it): ExposureErrorCompensator.apply (stitcher.py:219-221)
        fused into the warp kernel's epilogue from the next run on."""
        from .exposure_error_compensator import gain_arguments

        gmap, gw, gh, gc, gscalar = gain_arguments(gain)
        _lib.check(_lib.lib().sb_compositor_set_gain(self._c, i, gmap.ctypes.data_as(C.c_void_p) if gmap is not None else None, gw, gh, gc,
                                                     gscalar.ctypes.data_as(C.c_void_p) if gscalar is not None else None),
                   "sb_compositor_set_gain")

    def set_seam_mask(self, i, seam_mask):
        """Blend mask of image i from its LOW-resolution seam mask (what SeamFinder.find returns): SeamFinder.resize
        (seam_finder.py:38-43) runs on the device -- dilate, resize to the warped size, AND with the warped mask."""
        if hasattr(seam_mask, "get") and not isinstance(seam_mask, np.ndarray):
            seam_mask = seam_mask.get()
        seam_mask = np.ascontiguousarray(seam_mask, np.uint8)
        if seam_mask.ndim != 2:
            raise StitchingError(f"seam mask {i}: expected a 2-d uint8 array")
        _lib.check(_lib.lib().sb_compositor_set_seam_mask(self._c, i, seam_mask.ctypes.data_as(C.c_void_p), seam_mask.strides[0],
                                                          seam_mask.shape[1], seam_mask.shape[0]), "sb_compositor_set_seam_mask")

    def run(self):
        _lib.check(_lib.lib().sb_compositor_run(self._c), "sb_compositor_run")

    def sync(self):
        _lib.check(_lib.lib().sb_compositor_sync(self._c), "sb_compositor_sync")

    def download(self, out=None, out_mask=None, fmt="bgr"):
        """(pano, mask); with world > 1 the columns (strip_axis 0) or rows (strip_axis 1) self.strip[0]:self.strip[1].

        fmt "nv12" / "i420": the panorama as a (h * 3/2, w) YUV 4:2:0 array, cv.cvtColor(pano, COLOR_BGR2YUV_I420) of the BGR
        panorama (U and V interleaved for nv12), converted on the device (single-GPU compositors, even panorama sizes)."""
        h, w = self.roi[3], self.roi[2]
        if self.strip_axis == 0:
            w = self.strip[1] - self.strip[0]
        else:
            h = self.strip[1] - self.strip[0]
        if fmt != "bgr":
            pano = np.empty(color.frame_shape(w, h, fmt), np.uint8) if out is None else out
            mask = np.empty((h, w), np.uint8) if out_mask is None else out_mask
            ptrs, pitches, _ = color.planes(pano, w, h, fmt, writable=True)
            _lib.check(_lib.lib().sb_compositor_download_frame(self._c, color.fmt_code(fmt), ptrs, pitches,
                                                               mask.ctypes.data_as(C.c_void_p), mask.strides[0]),
                       "sb_compositor_download_frame")
            return pano, mask
        pano = np.empty((h, w, 3), np.uint8) if out is None else out
        mask = np.empty((h, w), np.uint8) if out_mask is None else out_mask
        _lib.check(_lib.lib().sb_compositor_download(self._c, pano.ctypes.data_as(C.c_void_p), pano.strides[0],
                                                     mask.ctypes.data_as(C.c_void_p), mask.strides[0]),
                   "sb_compositor_download")
        return pano, mask

    def download_warped(self, i):
        _, _, w, h = self.rects[i]
        img = np.empty((h, w, 3), np.uint8)
        mask = np.empty((h, w), np.uint8)
        _lib.check(_lib.lib().sb_compositor_download_warped(self._c, i, img.ctypes.data_as(C.c_void_p), w * 3,
                                                            mask.ctypes.data_as(C.c_void_p), w),
                   "sb_compositor_download_warped")
        return img, mask

    # -- sharded composite: transport hooks (sb_compositor_run moves the slabs with NCCL itself) ---------
    def shard_phase(self, phase):
        """0: local kernels up to the filled send slabs; 1: finish after the receive slabs were filled."""
        _lib.check(_lib.lib().sb_compositor_shard_phase(self._c, int(phase)), "sb_compositor_shard_phase")

    def shard_slab(self, peer, outgoing):
        """(device pointer, bytes) of the slab sent to (outgoing=True) or received from `peer`; bytes may be 0."""
        p, n = C.c_void_p(), C.c_size_t()
        _lib.check(_lib.lib().sb_compositor_shard_slab(self._c, int(peer), int(bool(outgoing)), C.byref(p), C.byref(n)),
                   "sb_compositor_shard_slab")
        return p.value, n.value

    def submit(self, images, out, out_mask, in_fmt="bgr", out_fmt="bgr"):
        """Pipelined step: enqueue upload of `images`, warp + blend, download into `out` / `out_mask`; returns a
        ticket for wait().  At most three tickets in flight; host arrays should live in pinned memory
        (`pinned_empty`) and must stay untouched until wait(ticket) returns.

        in_fmt / out_fmt "nv12" / "i420": sources and / or panorama as (h * 3/2, w) YUV 4:2:0 arrays (see upload and
        download); with YUV formats `out` and `out_mask` may be None (that output is not copied back)."""
        if in_fmt != "bgr" or out_fmt != "bgr":
            return self._submit_frames(images, out, out_mask, in_fmt, out_fmt)
        n = self.n
        ptrs = (C.c_void_p * n)()
        pitches = (C.c_size_t * n)()
        for i, img in enumerate(images):
            if img.dtype != np.uint8 or img.shape != (self.sizes[i][1], self.sizes[i][0], 3) or img.strides[1:] != (3, 1):
                raise StitchingError(f"image {i}: expected a uint8 {self.sizes[i][1]}x{self.sizes[i][0]}x3 array with packed pixels")
            ptrs[i] = img.ctypes.data
            pitches[i] = img.strides[0]
        ticket = C.c_ulonglong()
        _lib.check(_lib.lib().sb_compositor_submit(self._c, ptrs, pitches, out.ctypes.data_as(C.c_void_p), out.strides[0],
                                                   out_mask.ctypes.data_as(C.c_void_p), out_mask.strides[0], C.byref(ticket)),
                   "sb_compositor_submit")
        return ticket.value

    def _submit_frames(self, images, out, out_mask, in_fmt, out_fmt):
        n = self.n
        if len(images) != n:
            raise StitchingError(f"expected {n} images, got {len(images)}")
        in_code, out_code = color.fmt_code(in_fmt), color.fmt_code(out_fmt)
        ptrs = (C.c_void_p * (3 * n))()
        pitches = (C.c_size_t * (3 * n))()
        for i, img in enumerate(images):
            if not isinstance(img, np.ndarray):
                raise StitchingError(f"image {i}: expected a uint8 ndarray")
            p, q, arr = color.planes(img, self.sizes[i][0], self.sizes[i][1], in_fmt)
            if arr is not img:  # a copy would not outlive this call: the caller's array must already have the layout
                raise StitchingError(f"image {i}: the {in_fmt} frame must be laid out like a C-contiguous array")
            ptrs[3 * i: 3 * i + 3] = list(p)
            pitches[3 * i: 3 * i + 3] = list(q)
        _, _, pw, ph = self.roi
        out_ptrs, out_pitches = (C.c_void_p * 3)(), (C.c_size_t * 3)()
        if out is not None:
            out_ptrs, out_pitches, _ = color.planes(out, pw, ph, out_fmt, writable=True)
        ticket = C.c_ulonglong()
        _lib.check(_lib.lib().sb_compositor_submit_frames(self._c, in_code, ptrs, pitches, out_code, out_ptrs, out_pitches,
                                                          None if out_mask is None else out_mask.ctypes.data_as(C.c_void_p),
                                                          0 if out_mask is None else out_mask.strides[0], C.byref(ticket)),
                   "sb_compositor_submit_frames")
        return ticket.value

    def wait(self, ticket):
        _lib.check(_lib.lib().sb_compositor_wait(self._c, C.c_ulonglong(ticket)), "sb_compositor_wait")

    def pinned_empty(self, shape):
        """uint8 ndarray in page-locked host memory (freed with the compositor)."""
        nbytes = int(np.prod(shape))
        p = _lib.lib().sb_host_alloc(nbytes)
        if not p:
            _lib.check(-5, "sb_host_alloc")
        self._pinned.append(p)
        return np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p)).reshape(shape)

    def composite(self, images, in_fmt="bgr", out_fmt="bgr"):
        """One call: upload, warp + blend, download.  Returns (uint8 pano, uint8 mask) like Blender.blend(); the pixel
        formats are those of upload and download."""
        self.upload(images, fmt=in_fmt)
        self.run()
        return self.download(fmt=out_fmt)

    # -- measurement -------------------------------------------------------------------------------
    def time(self, iters, flush_l2=False):
        """Device time of `iters` runs, CUDA events on the compositor stream.

        Returns (total_ms, [(launch name, ms per run)]) with one entry per kernel launch, in launch order."""
        ms = C.c_float()
        _lib.check(_lib.lib().sb_compositor_time(self._c, int(iters), int(flush_l2), C.byref(ms)), "sb_compositor_time")
        cap = 64
        names = (C.c_char_p * cap)()
        vals = (C.c_float * cap)()
        k = _lib.lib().sb_compositor_stage_times(self._c, names, vals, cap)
        return ms.value, [(names[i].decode(), vals[i]) for i in range(k)]

    def model_bytes(self):
        """Compulsory HBM traffic of one run: (total bytes, [bytes per launch, in launch order])."""
        cap = 64
        tot = C.c_double()
        per = (C.c_double * cap)()
        k = _lib.lib().sb_compositor_model_bytes(self._c, C.byref(tot), per, cap)
        if k < 0:
            _lib.check(k, "sb_compositor_model_bytes")
        return tot.value, [per[i] for i in range(k)]

    def close(self):
        if getattr(self, "_c", None):
            _lib.lib().sb_compositor_destroy(self._c)  # synchronises all its streams first
            self._c = None
            for p in self._pinned:
                _lib.lib().sb_host_free(p)
            self._pinned = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
