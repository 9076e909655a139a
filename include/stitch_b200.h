/*
 * stitch_b200.h -- C ABI of libstitch_b200.so: the B200-native (sm_100a) compositing hot path of
 * OpenStitching/stitching, i.e. what stitching/warper.py and stitching/blender.py reach in OpenCV.
 *
 * Conventions
 *   - plain C, no exceptions cross the boundary; every int-returning entry returns SB_OK (0) or a
 *     negative sb_status, and sb_last_error() gives the text for the calling thread.
 *   - host pointers belong to the caller for the duration of a call; nothing is retained after
 *     return except inside opaque handles.  Device memory is owned by the library.
 *   - images are uint8 HxWx3 interleaved with a row pitch in BYTES; masks are uint8 HxW.
 *   - K and R are row-major float32 3x3 (warper.py:84-94 get_K, camera.R).
 *   - there is NO CPU fallback: without a usable sm_100 device every compute entry fails with
 *     SB_ERR_NO_DEVICE.
 *
 * Each entry cites the reference interface it replaces (file:line in OpenStitching/stitching v0.7.0).
 */
#ifndef STITCH_B200_H
#define STITCH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB_API __attribute__((visibility("default")))

typedef enum {
    SB_OK = 0,
    SB_ERR_INVALID = -1,   /* bad argument (what cv2 would assert on) */
    SB_ERR_NO_DEVICE = -2, /* no CUDA device / not sm_100 */
    SB_ERR_CUDA = -3,      /* CUDA runtime failure, see sb_last_error */
    SB_ERR_STATE = -4,     /* call order violation (feed before prepare, blend twice, ...) */
    SB_ERR_NOMEM = -5,
    SB_ERR_COMM = -6       /* NCCL failure */
} sb_status;

/* warper.py:10-27 WARP_TYPE_CHOICES; the four projections on the hot path */
/* warper.py:10-27 WARP_TYPE_CHOICES.  0-3: the projection runs on the device from separable trig tables (mercator, 14,
 * too); 4-15: mapBackward is not separable and has to match glibc's sinf / atan2f / tanf ... bit for bit, so the float
 * maps are built by the library's host code (libm, all cores) and the device does the resampling (sb_geometry.cpp). */
typedef enum {
    SB_WARP_SPHERICAL = 0, SB_WARP_CYLINDRICAL = 1, SB_WARP_PLANE = 2, SB_WARP_AFFINE = 3,
    SB_WARP_FISHEYE = 4, SB_WARP_STEREOGRAPHIC = 5,
    SB_WARP_COMPRESSED_PLANE_A2_B1 = 6, SB_WARP_COMPRESSED_PLANE_A1_5_B1 = 7,
    SB_WARP_COMPRESSED_PLANE_PORTRAIT_A2_B1 = 8, SB_WARP_COMPRESSED_PLANE_PORTRAIT_A1_5_B1 = 9,
    SB_WARP_PANINI_A2_B1 = 10, SB_WARP_PANINI_A1_5_B1 = 11, SB_WARP_PANINI_PORTRAIT_A2_B1 = 12, SB_WARP_PANINI_PORTRAIT_A1_5_B1 = 13,
    SB_WARP_MERCATOR = 14, SB_WARP_TRANSVERSE_MERCATOR = 15
} sb_warp_type;
/* blender.py:8-12 BLENDER_CHOICES */
typedef enum { SB_BLEND_NO = 0, SB_BLEND_FEATHER = 1, SB_BLEND_MULTIBAND = 2 } sb_blend_kind;

SB_API const char *sb_last_error(void);
SB_API const char *sb_version(void);

/* Select the CUDA device of this process (one process per GPU).  Must be called before any other
 * compute entry; calling it again with the same ordinal is a no-op. */
SB_API int sb_init(int device_ordinal);
/* name, SM count, compute capability of the selected device (any pointer may be NULL) */
SB_API int sb_device_info(char *name, size_t name_len, int *sm_count, int *cc_major, int *cc_minor);
/* number of kernels this library has launched so far in this process (bench.py "gpu_launches") */
SB_API unsigned long long sb_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Warper  (stitching/warper.py)
 * ------------------------------------------------------------------------------------------- */

/* warper.py:79-82  Warper.warp_roi -> cv.PyRotationWarper.warpRoi.
 * Host-only (libm) -- out_rect = {tl.x, tl.y, width, height}. */
SB_API int sb_warp_roi(int warp_type, float scale, const float K[9], const float R[9], int src_w, int src_h,
                       int out_rect[4]);

/* exposure_error_compensator.py:43-45 ExposureErrorCompensator.apply(index, corner, image, mask) -> cv.detail
 * {Gain,Channels,BlocksGain,BlocksChannels}Compensator::apply, in place on a uint8 h x w x 3 host image, with the
 * compensator's gain for that image (getMatGains()[index]):
 *   gain_map    float32 gh x gw x gc, gc = 1 (gain_blocks) or 3 (channel_blocks): resized to w x h as cv::resize
 *               (INTER_LINEAR) does in the reference's wheel, then saturate(cvRound(float(value) * gain));
 *   gain_scalar three doubles (gain: the value three times; channel): saturate(cvRound(double(value) * gain)).
 * Exactly one of the two is non-NULL; both NULL is the identity (compensator "no"). */
SB_API int sb_gain_apply(uint8_t *img, size_t pitch, int w, int h, const float *gain_map, int gw, int gh, int gc,
                         const double *gain_scalar);

/* images.py:120-123 Images.resize_img_by_scaler -> cv.resize(img, (dw, dh), interpolation=cv.INTER_LINEAR_EXACT) on a
 * uint8 image of 1 or 3 channels with host buffers (the step that produces the MEDIUM / LOW / FINAL resolution inputs
 * of the pipeline; OpenCV's bit-exact fixed-point bilinear, any scale). */
SB_API int sb_resize_exact(const uint8_t *src, size_t src_pitch, int sw, int sh, int channels, uint8_t *dst, size_t dst_pitch,
                           int dw, int dh);

/* seam_finder.py:38-43 SeamFinder.resize(seam_mask, mask) with host buffers:
 *   dst = cv.bitwise_and(cv.resize(cv.dilate(seam_mask, None), (w, h), 0, 0, cv.INTER_LINEAR_EXACT), mask)
 * (the positional arguments of that cv.resize call select its default INTER_LINEAR; reproduced bit for bit).
 * seam: uint8 sh x sw; mask, dst: uint8 h x w. */
SB_API int sb_seam_resize(const uint8_t *seam, size_t seam_pitch, int sw, int sh, const uint8_t *mask, size_t mask_pitch,
                          int w, int h, uint8_t *dst, size_t dst_pitch);

/* ---------------------------------------------------------------------------------------------
 * Pixel formats of frames going in and out of the compositor.  A YUV 4:2:0 frame (BT.601, limited range, what cameras,
 * NVDEC / NVENC and ffmpeg's yuv420p carry) is given as up to three planes with a row pitch in bytes each:
 *   SB_PIX_BGR   planes[0] = uint8 h x w x 3 (planes[1], planes[2] unused)
 *   SB_PIX_NV12  planes[0] = Y, h rows of w bytes; planes[1] = interleaved U V, h/2 rows of w bytes
 *   SB_PIX_I420  planes[0] = Y; planes[1] = U and planes[2] = V, h/2 rows of w/2 bytes each
 * A YUV input frame means cv.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420) followed by the BGR pipeline; a YUV panorama
 * means cv.cvtColor(pano, COLOR_BGR2YUV_I420) of the BGR panorama, with U and V interleaved for NV12.  Both are bit-exact
 * to OpenCV.  As in OpenCV, YUV frames have even widths and heights (SB_ERR_INVALID otherwise).
 * ------------------------------------------------------------------------------------------- */
typedef enum { SB_PIX_BGR = 0, SB_PIX_NV12 = 1, SB_PIX_I420 = 2 } sb_pix_fmt;

/* cv.cvtColor(COLOR_YUV2BGR_NV12 / _I420) with host buffers: fmt is SB_PIX_NV12 or SB_PIX_I420, dst uint8 h x w x 3 */
SB_API int sb_cvt_yuv420_to_bgr(int fmt, const uint8_t *const planes[3], const size_t pitches[3], int w, int h, uint8_t *dst,
                                size_t dst_pitch);
/* cv.cvtColor(COLOR_BGR2YUV_I420) with host buffers, chroma interleaved for SB_PIX_NV12 */
SB_API int sb_cvt_bgr_to_yuv420(int fmt, const uint8_t *src, size_t src_pitch, int w, int h, uint8_t *const planes[3],
                                const size_t pitches[3]);

/* warper.py:43-52 Warper.warp_image   -> PyRotationWarper.warp(INTER_LINEAR, BORDER_REFLECT)
 * warper.py:58-68 create_and_warp_mask -> PyRotationWarper.warp(INTER_NEAREST, BORDER_CONSTANT) on a 255 mask
 * Both outputs come from ONE kernel pass.  dst_img / dst_mask may each be NULL; their extents must be
 * out_rect[3] rows x out_rect[2] columns as given by sb_warp_roi for the same arguments.
 * src may be NULL when dst_img is NULL (mask only needs the source size). */
SB_API int sb_warp(int warp_type, float scale, const float K[9], const float R[9], const uint8_t *src, int src_w,
                   int src_h, size_t src_pitch, uint8_t *dst_img, size_t dst_pitch, uint8_t *dst_mask,
                   size_t mask_pitch, int out_rect[4]);

/* Device-resident twins (SURVEY.md 8b "device-handle variants"): stitcher.py hands every warped FINAL-resolution image
 * from Warper.warp_image (:185-189) through cropping (cropper.py:150-151, slicing) and ExposureErrorCompensator.apply
 * (:219-221) to Blender.feed (:254).  sb_warp_keep is sb_warp that additionally keeps what it computed in device memory
 * and hands out a handle; the *_dev entries below take a rectangle of such a handle instead of a host buffer, so the
 * image crosses PCIe once in each direction instead of three times.  A handle is dense uint8, h x w x channels. */
typedef struct sb_devimg sb_devimg;
SB_API int sb_warp_keep(int warp_type, float scale, const float K[9], const float R[9], const uint8_t *src, int src_w,
                        int src_h, size_t src_pitch, uint8_t *dst_img, size_t dst_pitch, uint8_t *dst_mask,
                        size_t mask_pitch, int out_rect[4], sb_devimg **keep_img, sb_devimg **keep_mask);
SB_API void sb_devimg_release(sb_devimg *d);
SB_API int sb_devimg_info(const sb_devimg *d, int *w, int *h, int *channels);
/* sb_gain_apply on the rectangle (x, y, w, h) of a 3-channel handle: the device copy is updated in place and the result
 * is also written to `host` (the reference's apply modifies its argument in place and returns it) */
SB_API int sb_gain_apply_dev(sb_devimg *img, int x, int y, int w, int h, uint8_t *host, size_t host_pitch, const float *gain_map,
                             int gw, int gh, int gc, const double *gain_scalar);

/* ---------------------------------------------------------------------------------------------
 * Blender  (stitching/blender.py)
 * ------------------------------------------------------------------------------------------- */
typedef struct sb_blender sb_blender;

/* blender.py:27-36: kind + setNumBands(num_bands) / setSharpness(sharpness) */
SB_API sb_blender *sb_blender_create(int kind, int num_bands, float sharpness);
SB_API void sb_blender_destroy(sb_blender *b);
/* blender.py:38 blender.prepare(dst_roi): dst_roi = cv.detail.resultRoi(corners, sizes) (blender.py:24) */
SB_API int sb_blender_prepare(sb_blender *b, int x, int y, int w, int h);
/* effective number of bands after MultiBandBlender::prepare's clipping (valid after prepare) */
SB_API int sb_blender_num_bands(const sb_blender *b);
/* blender.py:40-41 Blender.feed(img, mask, corner).  img is uint8 HxWx3 (img_is_s16 = 0) or int16 HxWx3
 * (img_is_s16 = 1, pitch still in bytes); mask uint8 HxW with gray values 0..255.
 * The feed is recorded and uploaded; arithmetic is deferred to sb_blender_blend, which applies the
 * feeds in call order (results are identical to eager accumulation). */
SB_API int sb_blender_feed(sb_blender *b, const void *img, int img_is_s16, size_t img_pitch, const uint8_t *mask,
                           size_t mask_pitch, int w, int h, int tl_x, int tl_y);
/* the same feed with the uint8 image taken from the rectangle (ix, iy, w, h) of a device twin and the mask either from the
 * rectangle (mx, my, w, h) of a 1-channel twin (mask_dev != NULL) or from the host (mask_host) */
SB_API int sb_blender_feed_dev(sb_blender *b, const sb_devimg *img, int ix, int iy, const sb_devimg *mask_dev, int mx, int my,
                               const uint8_t *mask_host, size_t mask_pitch, int w, int h, int tl_x, int tl_y);

/* blender.py:43-48 Blender.blend(): ::blend + cv.convertScaleAbs.  dst is uint8 HxWx3 of the prepared
 * roi size, dst_mask uint8 HxW; dst_s16 (nullable) additionally receives the int16 result before
 * convertScaleAbs (pitch in bytes).  The blender returns to the un-prepared state. */
SB_API int sb_blender_blend(sb_blender *b, uint8_t *dst, size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch,
                            int16_t *dst_s16, size_t s16_pitch);

/* ---------------------------------------------------------------------------------------------
 * Timelapser  (stitching/timelapser.py) -- the other consumer of warped frames (stitcher.py:249-252)
 * ------------------------------------------------------------------------------------------- */
/* timelapser.py:40-52 Timelapser.process_frame + get_frame -> cv.detail.Timelapser(AS_IS | CROP).process / getDst +
 * cv.convertScaleAbs: the uint8 frame of the prepared roi (`roi` = x, y, w, h: cv.detail.resultRoi of the warped rects for
 * "as_is", resultRoiIntersection for "crop", timelapser.py:36-37 initialize) that is zero except for ONE warped image
 * pasted at its corner (tlx, tly); pixels outside the roi are dropped, values shown as min(|v|, 255).
 * The image comes from the host (`img`: uint8 x3, or int16 x3 when is_s16, pitch in bytes) or, when `dev` is given, from
 * the rectangle (dev_x, dev_y, w, h) of a warped image that still lies in device memory (sb_warp_keep). */
SB_API int sb_timelapse_frame(const void *img, int is_s16, size_t pitch, const sb_devimg *dev, int dev_x, int dev_y, int w, int h,
                              int tlx, int tly, const int roi[4], uint8_t *dst, size_t dst_pitch);


/* ---------------------------------------------------------------------------------------------
 * Fused compositor: warp + blend with every intermediate resident in HBM.
 * The call sequence replaces stitcher.py:178-189 (warp_final_resolution) + :241-259 (prepare / feed /
 * blend) for a fixed rig; one compositor = one rig geometry (plan), run once per batch of frames.
 * ------------------------------------------------------------------------------------------- */
typedef struct sb_compositor sb_compositor;

typedef struct {
    int n_images;
    int warp_type;        /* sb_warp_type */
    float scale;          /* Warper.scale * aspect (warper.py:44) */
    int blend_kind;       /* sb_blend_kind */
    float blend_strength; /* blender.py:14 DEFAULT_BLEND_STRENGTH = 5; num_bands / sharpness derived as blender.py:25-36 */
    const int *src_w;     /* [n] */
    const int *src_h;     /* [n] */
    const float *K;       /* [n][9] */
    const float *R;       /* [n][9] */
    int mask_mode;        /* 0: blend mask = warped validity mask (seam finder "no"); 1: masks supplied via sb_compositor_set_mask */
} sb_rig;

SB_API sb_compositor *sb_compositor_create(const sb_rig *rig);
SB_API void sb_compositor_destroy(sb_compositor *c);
/* geometry of the plan: per image warped rect {x,y,w,h} (== sb_warp_roi) and the pano roi {x,y,w,h} */
SB_API int sb_compositor_geometry(const sb_compositor *c, int *rects /*[n][4]*/, int pano_roi[4], int *num_bands);
/* compulsory HBM traffic of one run (DESIGN.md byte model) for the roofline: total, and per kernel launch in
 * launch order (same order as sb_compositor_stage_times).  Returns the number of launches (or < 0). */
SB_API int sb_compositor_model_bytes(const sb_compositor *c, double *total_bytes, double *per_launch, int cap);
/* host -> device copy of source image i (uint8 HxWx3); asynchronous on the compositor stream when
 * `pinned` != 0 (caller guarantees page-locked memory and keeps it alive until sync) */
SB_API int sb_compositor_upload(sb_compositor *c, int i, const uint8_t *src, size_t pitch, int pinned);
/* the same for a frame in any sb_pix_fmt (sb_compositor_upload is this with SB_PIX_BGR); a YUV frame is converted on the
 * device.  YUV frames need a single-GPU compositor (SB_ERR_STATE on a sharded one). */
SB_API int sb_compositor_upload_frame(sb_compositor *c, int i, int fmt, const uint8_t *const planes[3], const size_t pitches[3],
                                      int pinned);
/* optional per-image blend mask in warped coordinates (mask_mode 1), uint8 h' x w' */
SB_API int sb_compositor_set_mask(sb_compositor *c, int i, const uint8_t *mask, size_t pitch);
/* the same from the LOW-resolution seam mask of image i (uint8 sh x sw, what SeamFinder.find returns): the device
 * performs SeamFinder.resize (seam_finder.py:38-43, called at stitcher.py:223-225) -- cv.dilate 3x3, cv.resize to the
 * warped size, AND with the warped mask -- and uses the result as blend mask from the next run on */
SB_API int sb_compositor_set_seam_mask(sb_compositor *c, int i, const uint8_t *seam, size_t seam_pitch, int sw, int sh);
/* exposure compensation of image i, fused into the warp: what ExposureErrorCompensator.apply(i, corner, warped, mask)
 * (exposure_error_compensator.py:43-45, stitcher.py:219-221) does to the warped image, with the compensator's gain for
 * image i -- cv.detail ...Compensator.getMatGains()[i] -- passed as in sb_gain_apply.  Both NULL: no compensation. */
SB_API int sb_compositor_set_gain(sb_compositor *c, int i, const float *gain_map, int gw, int gh, int gc, const double *gain_scalar);
/* enqueue warp + blend on the compositor stream (no host sync) */
SB_API int sb_compositor_run(sb_compositor *c);
/* device -> host copy of the panorama (uint8 HxWx3 + uint8 mask); synchronises */
SB_API int sb_compositor_download(sb_compositor *c, uint8_t *dst, size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch);
/* the same with the panorama in any sb_pix_fmt (sb_compositor_download is this with SB_PIX_BGR); planes == NULL or
 * planes[0] == NULL skips the panorama, dst_mask == NULL the mask.  A YUV panorama needs an even panorama size and a
 * single-GPU compositor (SB_ERR_STATE on a sharded one). */
SB_API int sb_compositor_download_frame(sb_compositor *c, int fmt, uint8_t *const planes[3], const size_t pitches[3], uint8_t *dst_mask,
                                        size_t mask_pitch);
/* Pipelined end-to-end step (throughput path): enqueue H2D of the n sources, warp + blend, and D2H of the
 * panorama on separate streams chained by events, and return a ticket.  Three buffer sets are kept, so at most
 * three tickets may be in flight: the copies of one step overlap the kernels of its neighbours.  Host buffers
 * should be page-locked (sb_host_alloc) and must stay valid until sb_compositor_wait(ticket) returns. */
SB_API int sb_compositor_submit(sb_compositor *c, const uint8_t *const *srcs, const size_t *pitches, uint8_t *dst,
                                size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch, unsigned long long *ticket);
/* the same with sources and panorama in any sb_pix_fmt (sb_compositor_submit is this with SB_PIX_BGR both ways): planes /
 * pitches hold three entries per source image (planes[3 i + k]), out_planes == NULL or out_planes[0] == NULL skips the
 * panorama.  The YUV copies share the copy streams with the BGR ones; the conversions run on the device. */
SB_API int sb_compositor_submit_frames(sb_compositor *c, int in_fmt, const uint8_t *const *planes, const size_t *pitches, int out_fmt,
                                       uint8_t *const out_planes[3], const size_t out_pitches[3], uint8_t *dst_mask, size_t mask_pitch,
                                       unsigned long long *ticket);
SB_API int sb_compositor_wait(sb_compositor *c, unsigned long long ticket);
/* device -> host copy of warped image i / its mask (for parity tests of the fused path) */
SB_API int sb_compositor_download_warped(sb_compositor *c, int i, uint8_t *dst, size_t dst_pitch, uint8_t *dst_mask,
                                         size_t mask_pitch);
SB_API int sb_compositor_sync(sb_compositor *c);
/* time `iters` back-to-back runs with CUDA events on the compositor stream; flush_l2 != 0 writes a
 * buffer larger than L2 between runs (outside the timed intervals).  ms_total = sum of the intervals. */
SB_API int sb_compositor_time(sb_compositor *c, int iters, int flush_l2, float *ms_total);
/* throughput with several batches in flight: `iters` steps dealt round-robin to n (<= 8) compositors of the same rig,
 * each on its own stream; ms_total = device time from the common start event to the last stream's end event */
SB_API int sb_compositor_time_multi(sb_compositor *const *cs, int n, int iters, float *ms_total);
/* device time of every kernel launch of the last sb_compositor_time call, averaged per run, in launch order:
 * names[] receives up to `cap` strings owned by the compositor, ms[] the matching times.  Returns count. */
SB_API int sb_compositor_stage_times(sb_compositor *c, const char **names, float *ms, int cap);

/* page-locked host memory for the e2e path */
SB_API void *sb_host_alloc(size_t bytes);
SB_API void sb_host_free(void *p);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU (one process per GPU): images are sharded over ranks, each rank composites its shard
 * and the per-band accumulators of overlapping footprints are exchanged with NCCL.
 * ------------------------------------------------------------------------------------------- */
/* One panorama over `world` GPUs.  Every rank passes the SAME rig (all n images); rank r warps and builds pyramids
 * for images [r*n/world, (r+1)*n/world) only (upload just those) and owns one column strip of the panorama.
 * sb_compositor_run = local kernels + one grouped NCCL send/recv of the per-band partial sums where padded
 * footprints cross strip boundaries + normalise/collapse of the own strip.  Requires sb_comm_init, the
 * multiband blender with >= 1 band and image blocks ordered left to right.  download() returns the strip. */
SB_API sb_compositor *sb_compositor_create_sharded(const sb_rig *rig, int rank, int world);
/* first image / number of images of this rank and its output columns [strip[0], strip[1]) in pano-roi coordinates */
SB_API int sb_compositor_shard_info(const sb_compositor *c, int *first_image, int *n_local, int strip[2]);
/* 0: `strip` above are columns of the panorama (multiband always; feather when the image blocks lie side by side);
 * 1: rows (feather with image blocks stacked vertically, e.g. the rows of BASELINE configs[4]'s 4x4 grid) */
SB_API int sb_compositor_shard_axis(const sb_compositor *c);
/* transport hooks: phase 0 = local kernels up to the filled send slabs, phase 1 = finish after the receive slabs
 * were filled; sb_compositor_shard_slab exposes the device buffers (outgoing != 0: send slab to `peer`) */
SB_API int sb_compositor_shard_phase(sb_compositor *c, int phase);
SB_API int sb_compositor_shard_slab(sb_compositor *c, int peer, int outgoing, void **dev_ptr, size_t *bytes);
/* plain device-to-device copy on the library's default stream, synchronous (utility for the hooks above) */
SB_API int sb_device_copy(void *dst, const void *src, size_t bytes);

/* Device self test of the shared-reciprocal division the warp (mode 0) and collapse (mode 1) kernels use in place of
 * one IEEE division per quotient: n pseudo-random operand pairs from the ranges those kernels guarantee, compared bit
 * for bit with the IEEE division on the device; *mismatches must come back 0. */
SB_API int sb_selftest_division(unsigned long long n, unsigned long long seed, int mode, unsigned long long *mismatches);

#define SB_COMM_ID_BYTES 128
SB_API int sb_comm_unique_id(uint8_t id[SB_COMM_ID_BYTES]);
SB_API int sb_comm_init(const uint8_t id[SB_COMM_ID_BYTES], int rank, int world);
SB_API int sb_comm_destroy(void);

#ifdef __cplusplus
}
#endif
#endif /* STITCH_B200_H */
