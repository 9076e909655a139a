// sb_internal.h -- shared declarations of libstitch_b200.so (not part of the public C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/stitch_b200.h"

#define SB_MAX_BANDS 16
#define SB_MAX_IMAGES 256
#define SB_SRC_PAD 16  // spare bytes after a source image: the warp kernel reads aligned 8-byte words

namespace sb {

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);
#define SB_CUDA(call)                                                         \
    do {                                                                      \
        cudaError_t e__ = (call);                                             \
        if (e__ != cudaSuccess) return sb::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)
#define SB_TRY(call)            \
    do {                        \
        int r__ = (call);       \
        if (r__ != SB_OK) return r__; \
    } while (0)

int ensure_device();  // SB_OK when sb_init succeeded (or lazily selects device 0)
int sm_count();
void count_launch(unsigned n = 1);
void adjust_launch_count(long long delta);  // graph capture records launches that do not execute; replays execute them
cudaStream_t default_stream();

// stream-ordered device allocation (cudaMallocAsync pool with a high release threshold)
int dev_alloc(void **p, size_t bytes, cudaStream_t s);
void dev_free(void *p, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
// geometry (host, libm): sb_geometry.cpp
// ---------------------------------------------------------------------------------------------
struct Projector {
    int type;  // SB_WARP_* (affine folded into plane; the A/B variants folded into their class, parameters in a, b)
    float scale;
    float a, b;  // compressedPlane / panini parameters
    float k[9], rinv[9], r_kinv[9], k_rinv[9], t[3];
};
void projector_setup(Projector &p, int warp_type, float scale, const float *K, const float *R);
void projector_roi(const Projector &p, int src_w, int src_h, int rect[4]);
// Separable backward-map tables: for output column u (absolute, tl.x + i) and row v
//   x_ = rowA[v] * colX[u];  y_ = rowY[v];  z_ = rowA[v] * colZ[u]
// (multiplication by an exact 1.0f keeps cylindrical / plane bit-identical to the unfactored form)
void projector_tables(const Projector &p, const int rect[4], float *colX, float *colZ, float *rowA, float *rowY);
// projections whose mapBackward is not separable: the float maps of RotationWarperBase::buildMaps over `rect`
// (rect[3] rows of rect[2] floats each), computed with libm on all host cores
bool projector_needs_maps(const Projector &p);
void projector_maps(const Projector &p, const int rect[4], float *xmap, float *ymap);

// ---------------------------------------------------------------------------------------------
// device-side descriptors
// ---------------------------------------------------------------------------------------------
struct WarpJob {
    const uint8_t *src;  // u8x3 interleaved
    int sw, sh;
    long long spitch;    // bytes
    const uint32_t *src4;  // optional: the same image as r | g<<8 | b<<16 (byte 3 zero), sw pixels per row (compositor: repacked at upload)
    uint8_t *dst_rgb;    // u8x3 interleaved or null
    long long dst_pitch;
    uint8_t *dst_mask;   // u8 or null
    long long mask_pitch;
    uint32_t *dst_rgbm;  // packed r | g<<8 | b<<16 | mask<<24, or null
    long long rgbm_pitch;  // elements
    int blend_mask_and;         // 1: the stored weight byte is blend_mask & validity (sb_compositor_set_seam_mask)
    const uint8_t *blend_mask;  // optional blend mask (seam mask AND validity, stitcher.py:223-239) stored in the
    long long blend_mask_pitch; // mask byte of dst_rgbm instead of the validity mask
    int dw, dh;
    const float *colX, *colZ, *rowA, *rowY;
    const float *xmap, *ymap;  // non-null: backward map given per pixel (dw floats per row), the tables are unused
    float k[9];
    int always_divide;  // plane / affine: x/z, y/z unconditionally
    float xin_hi, yin_hi;  // 32 (sw-1) - 0.5, 32 (sh-1) - 0.5: upper limits of x*32, y*32 for a footprint inside the image
    // exposure compensation of the warped image (ExposureErrorCompensator.apply, stitcher.py:219-221), fused into the
    // warp's epilogue.  gain_mode 0: none; 1: float32 gain map (gain_gc = 1 or 3 channels) resized to dw x dh through
    // the per-axis taps below (resize_f32_taps); 2: scalar gains as three 256-entry tables (gain_lut[c * 256 + value])
    int gain_mode, gain_gw, gain_gc, gain_pad;
    const float *gain_map;
    const int *gain_tx, *gain_ty;    // [i0 | i1], dw / dh entries each
    const float *gain_fx, *gain_fy;  // fractions
    const uint8_t *gain_lut;
};

// floats in the device tables of a w x h warp: colX, colZ (each padded to a multiple of 4), rowA, rowY
inline size_t warp_table_floats(int w, int h) { return (size_t)2 * ((w + 3) & ~3) + (size_t)2 * h; }

// one pyramid level of one fed image: planar int16 x3 + float32 weights
// Two colour layouts.  An image fed as bytes (RGBM) keeps every Gaussian level inside 0..255 (the 5x5 weights sum
// to 256), so its levels are stored as LANE PAIRS: q[y*pitch + x] = (r | b << 16, g), 8 bytes per pixel -- red and
// blue travel as two 16-bit lanes of one word through every filter (no lane ever carries: 256*255+128 < 2^16).
// A generic int16 feed (arbitrary values) keeps planar int16 and is served by the simple kernels only.
struct Level {
    uint2 *q;          // [h][pitch] lane pairs, or null
    int16_t *g;        // [3][h][pitch] planar, or null
    float *w;          // [h][pitch]
    int w_px, h_px;    // level size
    int pitch;         // elements, for q / g rows and w rows
    long long plane;   // elements between colour planes of g
};

#define SB_DT_CHUNKS 32    // row chunks per column in the parallel column pass of the L1 distance transform
struct FeedImage {
    // level 0 (one of the two layouts)
    const uint32_t *rgbm;  // packed u8x3 + mask
    long long rgbm_pitch;  // elements
    const int16_t *s16;    // interleaved int16x3 (generic feed) or null
    long long s16_pitch;   // elements (int16)
    const uint8_t *mask;   // with s16 layout
    long long mask_pitch;
    int w, h;              // fed image size
    int left, top;         // image origin inside its padded rect
    int px, py;            // padded rect origin relative to the padded pano (level 0)
    int pw, ph;            // padded rect size (multiples of 2^nb)
    int dx, dy;            // feather / no: image origin relative to the pano roi
    const float *fw;       // feather weight map [h][w] (dense)
    int *dts;              // feather: scratch of the distance transform's column pass, [2][SB_DT_CHUNKS][w] ints
    Level lv[SB_MAX_BANDS + 1];  // lv[0] unused
};

// Compact per-(image, level) descriptors for the fast kernels: everything a kernel needs for one level in a
// few 16-byte words, prebuilt on the host (the generic FeedImage stays the source of truth for the simple ones).
struct alignas(16) ColDesc {       // collapse of level l
    int ox, oy, w_l, h_l;          // padded rect of the image at level l, pano level coordinates
    const uint32_t *rgbm;          // level 0: packed fed image
    union {
        const uint2 *q;            // kind 0, level l >= 1: colour lane pairs
        const int16_t *g;          // kind 1: the slab's three int16 planes of partial sums
    };
    const float *w;                // weights (kind 1: weight sums)
    const uint2 *uq;               // level l+1 colour lane pairs (null at the top level)
    int rgbm_pitch, iw, ih, left;  // level 0: image size and origin inside the padded rect
    int top, pitch, plane, upitch; // level l / l+1 pitches, in elements; plane: stride of a slab's planes
    int pad0, kind, pad1, pad2;    // kind 0: a fed image; 1: a slab of partial sums
};
struct alignas(16) PyrDesc {       // pyrDown of level l -> l+1
    int sw, sh, dpitch, pad3;      // source level size; destination pitch (elements)
    const uint32_t *rgbm;          // level 0 source
    const uint2 *sq;               // level >= 1 source lane pairs
    const float *swt;
    uint2 *dq;
    float *dwt;
    int rgbm_pitch, iw;
    int ih, left, top, spitch;
    int pad0, pad1, pad2, pad4;
};

// Per-(level, image) descriptor of the tile kernels (sb_collapse_tile.cu), next to the item's ColDesc: the rect that
// decides whether the item touches a tile (= the extent of its level-l source) and the origins of its staged windows.
struct alignas(16) TileDesc {
    int x0, y0, w, h;           // level 0: the fed IMAGE inside its padded rect (weights are 0 outside); levels >= 1: the padded rect
    int ox, oy, uw, uh;         // padded rect origin at this level; size of the next coarser level (source of the pyrUp)
};
// window shapes of the tile kernels (one CTA = TILE_W x TILE_H pixels of a level, one thread per 2x2 quad)
#define SB_TILE_W 64
#define SB_TILE_H 16
#define SB_TILE_UPW (SB_TILE_W / 2 + 2)   // 34: the 3x3 neighbourhoods of the tile's quads at the coarser level
#define SB_TILE_UPH (SB_TILE_H / 2 + 2)   // 10

struct PanoLevel {
    int16_t *c;  // collapsed planar int16 x3 [3][h][pitch]
    int w_px, h_px, pitch;
    long long plane;
};

struct PanoOut {
    uint8_t *rgb; long long rgb_pitch;     // final uint8 HxWx3 (nullable)
    uint8_t *mask; long long mask_pitch;   // final uint8 mask (nullable)
    int16_t *s16; long long s16_pitch;     // final int16 HxWx3 before convertScaleAbs (nullable); pitch in elements
    int w, h;                              // unpadded roi size
};

// one launch of the fast per-level multiband kernel (sb_collapse_fast.cu), passed by value
#define SB_MAX_ITEMS 320  // fed images + slabs of other ranks
struct CollapseArgs {
    const ColDesc *col;       // items of this level in feed order (device)
    int n;
    PanoLevel up, cur;        // C_{l+1} (source of the pyrUp) and C_l (destination)
    int rx0, ry0, rw, rh;     // region of the level covered by this launch (even-aligned below the top level)
    int partial;              // 1: write the partial sums (acc, wsum) of the items to the slab below instead of finishing
    int16_t *slab_acc;        //    int16 x3 planes, origin = (rx0, ry0)
    float *slab_w;
    int slab_pitch, slab_plane;
    PanoOut out;              // level 0: final outputs; the buffer covers pano columns [out_x0, out_x0 + out.w)
    int out_x0, out_lo, out_hi;  // only columns [out_lo, out_hi) are stored (a strip's margin is not output)
    const TileDesc *tile;     // tile kernels: items of this level, same order as col (null: not available for this launch)
    int has_slabs;            // some items are slabs of partial sums (ColDesc kind 1): the tile kernels' slab instantiation
};
// the shared-memory tile version of the per-level kernel for the plain single-GPU roles; returns SB_ERR_STATE when the launch
// does not qualify (the caller then uses launch_collapse_fast)
int launch_collapse_tile(const CollapseArgs &A, int l, int nb, cudaStream_t s);
bool collapse_tile_enabled();
int launch_collapse_fast(const CollapseArgs &A, int l, int nb, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
// kernel launchers
// ---------------------------------------------------------------------------------------------
// jobs are HOST structs: they are passed by value in the kernel parameter block, SB_WARP_BATCH images per launch
#define SB_WARP_BATCH 32
int launch_warp(const WarpJob *jobs_host, int n_jobs, cudaStream_t s);
int warp_maps_upload(const Projector &p, const int rect[4], float *maps_dev, WarpJob *job, cudaStream_t s);  // sb_api.cpp
// u8x3 contiguous (w * h pixels) -> r | g<<8 | b<<16 words (the compositor's source layout for the warp kernel)
int launch_repack_rgbx(const uint8_t *rgb, uint32_t *dst, long long pixels, cudaStream_t s);
int launch_pack_rgbm(const uint8_t *rgb, long long rgb_pitch, const uint8_t *mask, long long mask_pitch, uint32_t *dst,
                     long long dst_pitch, int w, int h, cudaStream_t s);
// true when launch_warp(jobs, n_jobs) serves job i with a kernel that reads WarpJob::src4 and never WarpJob::src
bool warp_reads_src4_only(const WarpJob *jobs, int n_jobs, int i);
// YUV 4:2:0 planes (sb_yuv.cu): NV12 has Y and the interleaved UV plane in `u` (v unused), I420 has Y, U and V.  Pitches
// are in bytes and even.
struct YuvPlanes {
    const uint8_t *y, *u, *v;
    long long ypitch, upitch, vpitch;
};
struct YuvOut {
    uint8_t *y, *u, *v;
    long long ypitch, upitch, vpitch;
};
// cv.cvtColor(COLOR_YUV2BGR_NV12 / _I420) of an even w x h frame into the packed 3-byte source (bgr != null) or the
// word-per-pixel source of the warp kernel (bgrx != null, pitch in words)
int launch_yuv420_to_src(int fmt, const YuvPlanes &in, int w, int h, uint8_t *bgr, long long bgr_pitch, uint32_t *bgrx,
                         long long bgrx_pitch, cudaStream_t s);
// cv.cvtColor(COLOR_BGR2YUV_I420) of an even w x h uint8 BGR image, chroma interleaved for NV12
int launch_bgr_to_yuv420(int fmt, const uint8_t *bgr, long long bgr_pitch, int w, int h, const YuvOut &out, cudaStream_t s);
// level `l` -> `l+1` of images [first, first+count)
// `pyr` / `col`: the compact descriptors of level l for the same images (device pointers, `count` / `n` entries)
// binary_masks: the caller guarantees that every mask byte of these images is 0 or 255 (used for l <= 2; sb_pyrdown_fast.cu)
int launch_pyrdown(const FeedImage *imgs_dev, const FeedImage *imgs_host, const PyrDesc *pyr, int first, int count, int l,
                   int max_w, int max_h, cudaStream_t s, bool binary_masks = false);
// SB_KERNELS=simple selects the one-thread-per-pixel gather kernels everywhere (debugging / A-B parity)
bool use_simple_kernels();
// multiband: accumulate + normalise + collapse level l (top-down); at l == 0 writes the final outputs
struct TileDesc;
int launch_collapse(const FeedImage *imgs_dev, const FeedImage *imgs_host, const ColDesc *col, int n, const PanoLevel *pano_dev,
                    const PanoLevel *pano_host, int l, int nb, int lw, int lh, PanoOut out, cudaStream_t s,
                    const TileDesc *tile = nullptr);
// feather: distance-transform weight maps, then one fused accumulate/normalise pass; NO blender
// levels T .. nb in one launch (sb_tail.cu); SB_ERR_STATE: not available (emulation build), launch per level instead
int launch_tail(const FeedImage *imgs_dev, const PanoLevel *pano_dev, int first, int count, int n, int T, int nb, int wp, int hp, const PanoOut &out,
                unsigned *state, cudaStream_t s);
int launch_feather_weights(const FeedImage *imgs_dev, const FeedImage *imgs_host, int n, float sharpness, cudaStream_t s);
int launch_simple_blend(const FeedImage *imgs_dev, int n, int feather, PanoOut out, cudaStream_t s);
// sharded feather blend: a slab of partial sums (acc int16 x3 planes with wrap-around, wsum float32) over a rectangle of
// the pano roi, and one launch over a region: the slabs of lower ranks, images [i0, i1), the slabs of higher ranks, in that
// order; `partial`: write the sums as a slab instead of normalising
struct FeatherSlab {
    int x0, y0, w, h, pitch, plane;
    const int16_t *acc;
    const float *wsum;
};
struct FeatherRegionArgs {
    const FeedImage *imgs;
    int i0, i1;
    const FeatherSlab *slabs;
    int n_before, n_after;
    int rx0, ry0, rw, rh;    // region, pano-roi coordinates
    int partial;
    int16_t *slab_acc;       // partial: origin = (rx0, ry0)
    float *slab_w;
    int slab_pitch, slab_plane;
    PanoOut out;             // !partial: the buffer's origin is pano pixel (out_x0, out_y0)
    int out_x0, out_y0;
};
int launch_feather_region(const FeatherRegionArgs &A, cudaStream_t s);
int launch_flush_l2(void *buf, size_t bytes, cudaStream_t s);
int launch_wait_flags(const unsigned *flags, unsigned mask, unsigned value, cudaStream_t s);  // lanes with a mask bit wait for flags[lane] >= value
// ExposureErrorCompensator.apply: taps of the float32 bilinear resize of a gain map (sb_geometry.cpp), the 256-entry
// table of a scalar gain, and the host-buffer entry's kernel (sb_warp.cu)
void resize_f32_taps(int n_src, int n_dst, int *i0i1, float *fr);  // i0i1: 2 * n_dst ints
void gain_scalar_lut(const double gain[3], uint8_t lut[768]);
// rows copy; a fully contiguous image goes as ONE linear transfer (the DMA engines reach PCIe line rate with those)
static inline cudaError_t sb_copy2d(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width, size_t height,
                                    cudaMemcpyKind kind, cudaStream_t s)
{
    if (dpitch == width && spitch == width) return cudaMemcpyAsync(dst, src, width * height, kind, s);
    return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, kind, s);
}

// YUV 4:2:0 frames (sb_pix_fmt): plane k's bytes per row and rows, and its offset / pitch in the dense layout -- cv2's
// single (h * 3/2) x w array: Y, then UV (NV12) or U then V (I420), rows without padding
inline int yuv_nplanes(int fmt) { return fmt == SB_PIX_NV12 ? 2 : 3; }
inline size_t yuv_row_bytes(int fmt, int k, int w) { return k == 0 || fmt == SB_PIX_NV12 ? (size_t)w : (size_t)w / 2; }
inline int yuv_rows(int k, int h) { return k == 0 ? h : h / 2; }
inline size_t yuv_bytes(int w, int h) { return (size_t)w * h / 2 * 3; }
inline size_t yuv_dense_offset(int fmt, int k, int w, int h)
{
    return k == 0 ? 0 : (size_t)w * h + (k == 2 ? yuv_row_bytes(fmt, 1, w) * (size_t)(h / 2) : 0);
}
// every plane the format uses is given, with a pitch that holds its row
inline bool yuv_planes_ok(int fmt, const uint8_t *const planes[3], const size_t pitches[3], int w)
{
    if (!planes || !pitches) return false;
    for (int k = 0; k < yuv_nplanes(fmt); ++k)
        if (!planes[k] || pitches[k] < yuv_row_bytes(fmt, k, w)) return false;
    return true;
}
inline YuvPlanes yuv_dense_planes(int fmt, const uint8_t *buf, int w, int h)
{
    YuvPlanes p;
    p.y = buf;
    p.ypitch = w;
    p.u = buf + yuv_dense_offset(fmt, 1, w, h);
    p.upitch = (long long)yuv_row_bytes(fmt, 1, w);
    p.v = fmt == SB_PIX_NV12 ? nullptr : buf + yuv_dense_offset(fmt, 2, w, h);
    p.vpitch = fmt == SB_PIX_NV12 ? 0 : (long long)yuv_row_bytes(fmt, 2, w);
    return p;
}
inline YuvOut yuv_dense_out(int fmt, uint8_t *buf, int w, int h)
{
    const YuvPlanes p = yuv_dense_planes(fmt, buf, w, h);
    return YuvOut{const_cast<uint8_t *>(p.y), const_cast<uint8_t *>(p.u), const_cast<uint8_t *>(p.v), p.ypitch, p.upitch, p.vpitch};
}
// the planes of a frame between host buffers and a dense device buffer `dev`: one copy per plane, or ONE copy when the host
// planes lie densely in one buffer as well (the DMA engines reach PCIe line rate with long linear transfers)
static inline cudaError_t yuv_copy(uint8_t *dev, const uint8_t *const host[3], const size_t pitches[3], int fmt, int w, int h,
                                   cudaMemcpyKind kind, cudaStream_t s)
{
    const int np = yuv_nplanes(fmt);
    bool dense = true;
    for (int k = 0; k < np; ++k)
        dense = dense && pitches[k] == yuv_row_bytes(fmt, k, w) && host[k] == host[0] + yuv_dense_offset(fmt, k, w, h);
    if (dense) {
        const bool up = kind == cudaMemcpyHostToDevice;
        return cudaMemcpyAsync(up ? (void *)dev : (void *)host[0], up ? (const void *)host[0] : (const void *)dev, yuv_bytes(w, h), kind, s);
    }
    for (int k = 0; k < np; ++k) {
        uint8_t *d = dev + yuv_dense_offset(fmt, k, w, h);
        const size_t row = yuv_row_bytes(fmt, k, w);
        const cudaError_t e = kind == cudaMemcpyHostToDevice
                                  ? sb_copy2d(d, row, host[k], pitches[k], row, yuv_rows(k, h), kind, s)
                                  : sb_copy2d((void *)host[k], pitches[k], d, row, row, yuv_rows(k, h), kind, s);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// Timelapser frame: src8 (uint8 x3, pitch in bytes) or src16 (int16 x3, pitch in ELEMENTS) pasted at (dx, dy) of a cw x ch canvas
int launch_timelapse_frame(const uint8_t *src8, const int16_t *src16, long long spitch, int sw, int sh, int dx, int dy, uint8_t *dst,
                           long long dpitch, int cw, int ch, cudaStream_t s);
int launch_gain_apply(uint8_t *img, long long pitch, int w, int h, const WarpJob &gain_fields, cudaStream_t s);
// device copies of one image's gain (map + taps for a w x h target, or the scalar tables) and the WarpJob fields for them
struct GainData {
    float *map = nullptr, *fx = nullptr, *fy = nullptr;
    int *tx = nullptr, *ty = nullptr;
    uint8_t *lut = nullptr;
};
int gain_upload(WarpJob *job, GainData *gd, int w, int h, const float *gain_map, int gw, int gh, int gc, const double *gain_scalar,
                cudaStream_t s);  // synchronises s
void gain_free(GainData *gd, cudaStream_t s);
// Images.resize_img_by_scaler: cv.resize(uint8, INTER_LINEAR_EXACT) (sb_seam.cu, sb_geometry.cpp)
void resize_exact_taps(int n_src, int n_dst, int *t);  // t: 3 * n_dst ints
int launch_resize_exact(const uint8_t *src, long long spitch, int cn, const int *tx, const int *ty, uint8_t *dst, long long dpitch, int w,
                        int h, cudaStream_t s);
// SeamFinder.resize (sb_seam.cu, sb_geometry.cpp)
void resize_linear_taps(int n_src, int n_dst, bool columns, int *t);  // t: 4 * n_dst ints
int launch_seam_resize(const uint8_t *seam, int sw, int sh, uint8_t *scratch, const int *tx, const int *ty, const uint8_t *mask,
                       long long mask_pitch, uint8_t *dst, long long dst_pitch, int w, int h, cudaStream_t s);
// device version of SeamFinder.resize for host or device `mask` / `dst` buffers already on the device: uploads the seam
// mask, builds the taps, runs the two kernels (synchronises `s`)
int seam_resize_device(const uint8_t *seam_host, size_t seam_pitch, int sw, int sh, const uint8_t *mask_dev, long long mask_pitch,
                       uint8_t *dst_dev, long long dst_pitch, int w, int h, cudaStream_t s);
int launch_selftest_division(unsigned long long n, unsigned long long seed, int mode, unsigned long long *bad_dev, cudaStream_t s);

}  // namespace sb
