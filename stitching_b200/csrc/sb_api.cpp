// sb_api.cpp -- the C ABI (include/stitch_b200.h): Warper and Blender entry points with host buffers.
#include <algorithm>
#include <cstring>
#include <mutex>
#include <memory>
#include <vector>

#include "sb_plan.h"

using namespace sb;

namespace {

bool valid_warp_type(int t) { return t >= SB_WARP_SPHERICAL && t <= SB_WARP_TRANSVERSE_MERCATOR; }

// temp device buffers freed in stream order when the scope ends
struct Scratch {
    cudaStream_t s;
    std::vector<void *> ptrs;
    explicit Scratch(cudaStream_t st) : s(st) {}
    ~Scratch()
    {
        for (void *p : ptrs) dev_free(p, s);
    }
    template <typename T>
    int get(T **p, size_t count)
    {
        void *q = nullptr;
        int r = dev_alloc(&q, count * sizeof(T), s);
        if (r == SB_OK) ptrs.push_back(q);
        *p = (T *)q;
        return r;
    }
};

}  // namespace

namespace sb {
// shared with the compositor: builds the device tables + job for one image; tables go into `tab` (4 arrays)
int make_warp_job(const Projector &p, const int rect[4], int src_w, int src_h, float *tab_dev, WarpJob *job, cudaStream_t s,
                  std::vector<float> &host_tab)
{
    const int w = rect[2], h = rect[3];
    const int wp = (w + 3) & ~3;
    host_tab.assign(warp_table_floats(w, h), 0.f);
    float *colX = host_tab.data(), *colZ = colX + wp, *rowA = colZ + wp, *rowY = rowA + h;
    if (!projector_needs_maps(p)) projector_tables(p, rect, colX, colZ, rowA, rowY);  // (else: warp_maps_upload)
    SB_CUDA(cudaMemcpyAsync(tab_dev, host_tab.data(), host_tab.size() * sizeof(float), cudaMemcpyHostToDevice, s));
    std::memset(job, 0, sizeof *job);
    job->sw = src_w;
    job->sh = src_h;
    job->dw = w;
    job->dh = h;
    job->colX = tab_dev;
    job->colZ = tab_dev + wp;
    job->rowA = tab_dev + 2 * wp;
    job->rowY = tab_dev + 2 * wp + h;
    std::memcpy(job->k, p.k_rinv, sizeof job->k);
    job->always_divide = p.type == SB_WARP_PLANE;
    job->xmap = job->ymap = nullptr;
    job->xin_hi = 32.f * (float)(src_w - 1) - 0.5f;
    job->yin_hi = 32.f * (float)(src_h - 1) - 0.5f;
    return SB_OK;
}
// projections that are not separable: the float maps of buildMaps, built on the host (libm, all cores) and uploaded;
// `maps_dev` holds xmap then ymap (w * h floats each)
int warp_maps_upload(const Projector &p, const int rect[4], float *maps_dev, WarpJob *job, cudaStream_t s)
{
    const size_t n = (size_t)rect[2] * rect[3];
    std::vector<float> host(2 * n);
    projector_maps(p, rect, host.data(), host.data() + n);
    SB_CUDA(cudaMemcpyAsync(maps_dev, host.data(), 2 * n * sizeof(float), cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaStreamSynchronize(s));  // `host` is a local
    job->xmap = maps_dev;
    job->ymap = maps_dev + n;
    return SB_OK;
}
}  // namespace sb

struct sb_devimg {
    uint8_t *p;
    int w, h, ch;
};

// The reference asks for the same roi several times per image -- warp_roi, then warp (image), then warp (mask), each of
// which runs detectResultRoi again (warper.py:43-82) -- and for eleven of the projections that is a pass over EVERY source
// pixel.  The result depends on nothing but the arguments, so the last few are remembered (host memory, a few hundred bytes).
namespace {
struct RoiKey {
    int type, w, h;
    float scale, K[9], R[9];
};
struct RoiEntry {
    RoiKey key;
    int rect[4];
};
std::mutex g_roi_mutex;
std::vector<RoiEntry> g_roi_cache;  // most recent last
constexpr size_t ROI_CACHE_ENTRIES = 64;

void cached_roi(const Projector &p, int warp_type, float scale, const float K[9], const float R[9], int src_w, int src_h, int rect[4])
{
    RoiKey key;
    std::memset(&key, 0, sizeof key);
    key.type = warp_type;
    key.w = src_w;
    key.h = src_h;
    key.scale = scale;
    std::memcpy(key.K, K, sizeof key.K);
    std::memcpy(key.R, R, sizeof key.R);
    {
        std::lock_guard<std::mutex> lock(g_roi_mutex);
        for (size_t i = g_roi_cache.size(); i-- > 0;)
            if (!std::memcmp(&g_roi_cache[i].key, &key, sizeof key)) {  // bit patterns: -0.0f and NaNs simply miss
                std::memcpy(rect, g_roi_cache[i].rect, sizeof g_roi_cache[i].rect);
                return;
            }
    }
    projector_roi(p, src_w, src_h, rect);
    RoiEntry e;
    e.key = key;
    std::memcpy(e.rect, rect, sizeof e.rect);
    std::lock_guard<std::mutex> lock(g_roi_mutex);
    if (g_roi_cache.size() >= ROI_CACHE_ENTRIES) g_roi_cache.erase(g_roi_cache.begin());
    g_roi_cache.push_back(e);
}
}  // namespace

extern "C" {

int sb_warp_roi(int warp_type, float scale, const float K[9], const float R[9], int src_w, int src_h, int out_rect[4])
{
    if (!valid_warp_type(warp_type) || !K || !R || !out_rect || src_w <= 0 || src_h <= 0) {
        set_error("sb_warp_roi: invalid argument");
        return SB_ERR_INVALID;
    }
    Projector p;
    projector_setup(p, warp_type, scale, K, R);
    cached_roi(p, warp_type, scale, K, R, src_w, src_h, out_rect);
    return SB_OK;
}

static int warp_impl(int warp_type, float scale, const float K[9], const float R[9], const uint8_t *src, int src_w, int src_h,
                     size_t src_pitch, uint8_t *dst_img, size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch, int out_rect[4],
                     sb_devimg **keep_img, sb_devimg **keep_mask)
{
    if (keep_img) *keep_img = nullptr;
    if (keep_mask) *keep_mask = nullptr;
    if (!valid_warp_type(warp_type) || !K || !R || !out_rect || src_w <= 0 || src_h <= 0 || (dst_img && !src) ||
        (src && src_pitch < (size_t)src_w * 3)) {
        set_error("sb_warp: invalid argument");
        return SB_ERR_INVALID;
    }
    Projector p;
    projector_setup(p, warp_type, scale, K, R);
    int rect[4];
    cached_roi(p, warp_type, scale, K, R, src_w, src_h, rect);
    std::memcpy(out_rect, rect, sizeof rect);
    if (!dst_img && !dst_mask) return SB_OK;
    const int w = rect[2], h = rect[3];
    if (w <= 0 || h <= 0 || (long long)w * h > (1ll << 31)) {
        set_error("sb_warp: degenerate result roi %dx%d", w, h);
        return SB_ERR_INVALID;
    }
    if ((dst_img && dst_pitch < (size_t)w * 3) || (dst_mask && mask_pitch < (size_t)w)) {
        set_error("sb_warp: destination pitch too small for roi width %d", w);
        return SB_ERR_INVALID;
    }
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    Scratch tmp(s);
    float *tab = nullptr;
    uint8_t *d_src = nullptr, *d_img = nullptr, *d_mask = nullptr;
    SB_TRY(tmp.get(&tab, warp_table_floats(w, h)));
    std::vector<float> host_tab;
    WarpJob job;
    SB_TRY(make_warp_job(p, rect, src_w, src_h, tab, &job, s, host_tab));
    if (projector_needs_maps(p)) {
        float *maps = nullptr;
        SB_TRY(tmp.get(&maps, (size_t)2 * w * h));
        SB_TRY(warp_maps_upload(p, rect, maps, &job, s));
    }
    const bool keep_i = dst_img && keep_img, keep_m = dst_mask && keep_mask;
    if (dst_img) {
        SB_TRY(tmp.get(&d_src, (size_t)src_w * 3 * src_h + SB_SRC_PAD));
        if (keep_i)
            SB_TRY(dev_alloc((void **)&d_img, (size_t)w * 3 * h, s));  // survives the call inside the handle
        else
            SB_TRY(tmp.get(&d_img, (size_t)w * 3 * h));
        SB_CUDA(sb_copy2d(d_src, (size_t)src_w * 3, src, src_pitch, (size_t)src_w * 3, src_h, cudaMemcpyHostToDevice, s));
        job.src = d_src;
        job.spitch = (long long)src_w * 3;
        job.dst_rgb = d_img;
        job.dst_pitch = (long long)w * 3;
    }
    if (dst_mask) {
        if (keep_m)
            SB_TRY(dev_alloc((void **)&d_mask, (size_t)w * h, s));
        else
            SB_TRY(tmp.get(&d_mask, (size_t)w * h));
        job.dst_mask = d_mask;
        job.mask_pitch = w;
    }
    int rc = launch_warp(&job, 1, s);
    if (rc == SB_OK && dst_img && sb_copy2d(dst_img, dst_pitch, d_img, (size_t)w * 3, (size_t)w * 3, h, cudaMemcpyDeviceToHost, s) != cudaSuccess)
        rc = cuda_fail(cudaGetLastError(), "cudaMemcpy2DAsync", __FILE__, __LINE__);
    if (rc == SB_OK && dst_mask && sb_copy2d(dst_mask, mask_pitch, d_mask, w, w, h, cudaMemcpyDeviceToHost, s) != cudaSuccess)
        rc = cuda_fail(cudaGetLastError(), "cudaMemcpy2DAsync", __FILE__, __LINE__);
    if (cudaStreamSynchronize(s) != cudaSuccess && rc == SB_OK) rc = cuda_fail(cudaGetLastError(), "cudaStreamSynchronize", __FILE__, __LINE__);
    if (rc != SB_OK) {
        if (keep_i) dev_free(d_img, s);
        if (keep_m) dev_free(d_mask, s);
        return rc;
    }
    if (keep_i) *keep_img = new sb_devimg{d_img, w, h, 3};
    if (keep_m) *keep_mask = new sb_devimg{d_mask, w, h, 1};
    return SB_OK;
}

int sb_warp(int warp_type, float scale, const float K[9], const float R[9], const uint8_t *src, int src_w, int src_h,
            size_t src_pitch, uint8_t *dst_img, size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch, int out_rect[4])
{
    return warp_impl(warp_type, scale, K, R, src, src_w, src_h, src_pitch, dst_img, dst_pitch, dst_mask, mask_pitch, out_rect, nullptr, nullptr);
}

int sb_warp_keep(int warp_type, float scale, const float K[9], const float R[9], const uint8_t *src, int src_w, int src_h,
                 size_t src_pitch, uint8_t *dst_img, size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch, int out_rect[4],
                 sb_devimg **keep_img, sb_devimg **keep_mask)
{
    return warp_impl(warp_type, scale, K, R, src, src_w, src_h, src_pitch, dst_img, dst_pitch, dst_mask, mask_pitch, out_rect, keep_img, keep_mask);
}

void sb_devimg_release(sb_devimg *d)
{
    if (!d) return;
    dev_free(d->p, default_stream());
    delete d;
}

int sb_devimg_info(const sb_devimg *d, int *w, int *h, int *channels)
{
    if (!d) {
        set_error("sb_devimg_info: null handle");
        return SB_ERR_INVALID;
    }
    if (w) *w = d->w;
    if (h) *h = d->h;
    if (channels) *channels = d->ch;
    return SB_OK;
}

}  // extern "C"

namespace sb {
// SeamFinder.resize on the device: seam mask from the host, `mask_dev` / `dst_dev` on the device (mask_dev may be null)
int seam_resize_device(const uint8_t *seam_host, size_t seam_pitch, int sw, int sh, const uint8_t *mask_dev, long long mask_pitch,
                       uint8_t *dst_dev, long long dst_pitch, int w, int h, cudaStream_t s)
{
    Scratch tmp(s);
    uint8_t *d_seam = nullptr, *d_dil = nullptr;
    int *d_tx = nullptr, *d_ty = nullptr;
    SB_TRY(tmp.get(&d_seam, (size_t)sw * sh));
    SB_TRY(tmp.get(&d_dil, (size_t)sw * sh));
    SB_TRY(tmp.get(&d_tx, (size_t)4 * w));
    SB_TRY(tmp.get(&d_ty, (size_t)4 * h));
    std::vector<int> tx((size_t)4 * w), ty((size_t)4 * h);
    resize_linear_taps(sw, w, true, tx.data());
    resize_linear_taps(sh, h, false, ty.data());
    SB_CUDA(sb_copy2d(d_seam, sw, seam_host, seam_pitch, sw, sh, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_tx, tx.data(), tx.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_ty, ty.data(), ty.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    SB_TRY(launch_seam_resize(d_seam, sw, sh, d_dil, d_tx, d_ty, mask_dev, mask_pitch, dst_dev, dst_pitch, w, h, s));
    SB_CUDA(cudaStreamSynchronize(s));  // the tap vectors and the scratch buffers go out of scope
    return SB_OK;
}
}  // namespace sb

namespace sb {
void gain_free(GainData *gd, cudaStream_t s)
{
    dev_free(gd->map, s);
    dev_free(gd->fx, s);
    dev_free(gd->fy, s);
    dev_free(gd->tx, s);
    dev_free(gd->ty, s);
    dev_free(gd->lut, s);
    *gd = GainData{};
}

// ExposureErrorCompensator.apply's per-image data on the device: either the float32 gain map (gc = 1 or 3 channels) with
// the resize taps for a w x h image, or the three 256-entry tables of scalar gains
int gain_upload(WarpJob *job, GainData *gd, int w, int h, const float *gain_map, int gw, int gh, int gc, const double *gain_scalar,
                cudaStream_t s)
{
    gain_free(gd, s);
    job->gain_mode = 0;
    if (gain_scalar) {
        uint8_t lut[768];
        gain_scalar_lut(gain_scalar, lut);
        SB_TRY(dev_alloc((void **)&gd->lut, sizeof lut, s));
        SB_CUDA(cudaMemcpyAsync(gd->lut, lut, sizeof lut, cudaMemcpyHostToDevice, s));
        SB_CUDA(cudaStreamSynchronize(s));
        job->gain_lut = gd->lut;
        job->gain_mode = 2;
        return SB_OK;
    }
    if (!gain_map) return SB_OK;  // no gain: compensator "no"
    std::vector<int> tx((size_t)2 * w), ty((size_t)2 * h);
    std::vector<float> fx((size_t)w), fy((size_t)h);
    resize_f32_taps(gw, w, tx.data(), fx.data());
    resize_f32_taps(gh, h, ty.data(), fy.data());
    SB_TRY(dev_alloc((void **)&gd->map, sizeof(float) * (size_t)gw * gh * gc, s));
    SB_TRY(dev_alloc((void **)&gd->tx, sizeof(int) * tx.size(), s));
    SB_TRY(dev_alloc((void **)&gd->ty, sizeof(int) * ty.size(), s));
    SB_TRY(dev_alloc((void **)&gd->fx, sizeof(float) * fx.size(), s));
    SB_TRY(dev_alloc((void **)&gd->fy, sizeof(float) * fy.size(), s));
    SB_CUDA(cudaMemcpyAsync(gd->map, gain_map, sizeof(float) * (size_t)gw * gh * gc, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(gd->tx, tx.data(), sizeof(int) * tx.size(), cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(gd->ty, ty.data(), sizeof(int) * ty.size(), cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(gd->fx, fx.data(), sizeof(float) * fx.size(), cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(gd->fy, fy.data(), sizeof(float) * fy.size(), cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaStreamSynchronize(s));
    job->gain_map = gd->map;
    job->gain_tx = gd->tx;
    job->gain_ty = gd->ty;
    job->gain_fx = gd->fx;
    job->gain_fy = gd->fy;
    job->gain_gw = gw;
    job->gain_gc = gc;
    job->gain_mode = 1;
    return SB_OK;
}
}  // namespace sb

static bool valid_gain_args(const float *gain_map, int gw, int gh, int gc, const double *gain_scalar)
{
    if (gain_map && gain_scalar) return false;
    if (gain_map && (gw <= 0 || gh <= 0 || (gc != 1 && gc != 3))) return false;
    return true;
}

extern "C" {

int sb_gain_apply(uint8_t *img, size_t pitch, int w, int h, const float *gain_map, int gw, int gh, int gc, const double *gain_scalar)
{
    if (!img || w <= 0 || h <= 0 || pitch < (size_t)w * 3 || !valid_gain_args(gain_map, gw, gh, gc, gain_scalar)) {
        set_error("sb_gain_apply: invalid argument");
        return SB_ERR_INVALID;
    }
    if (!gain_map && !gain_scalar) return SB_OK;  // compensator "no": identity
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    Scratch tmp(s);
    uint8_t *d_img = nullptr;
    SB_TRY(tmp.get(&d_img, (size_t)w * 3 * h));
    SB_CUDA(sb_copy2d(d_img, (size_t)w * 3, img, pitch, (size_t)w * 3, h, cudaMemcpyHostToDevice, s));
    WarpJob job;
    std::memset(&job, 0, sizeof job);
    GainData gd;
    int rc = gain_upload(&job, &gd, w, h, gain_map, gw, gh, gc, gain_scalar, s);
    if (rc == SB_OK) rc = launch_gain_apply(d_img, (long long)w * 3, w, h, job, s);
    if (rc == SB_OK && sb_copy2d(img, pitch, d_img, (size_t)w * 3, (size_t)w * 3, h, cudaMemcpyDeviceToHost, s) != cudaSuccess)
        rc = SB_ERR_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess && rc == SB_OK) rc = SB_ERR_CUDA;
    gain_free(&gd, s);
    return rc;
}

int sb_gain_apply_dev(sb_devimg *img, int x, int y, int w, int h, uint8_t *host, size_t host_pitch, const float *gain_map, int gw, int gh,
                      int gc, const double *gain_scalar)
{
    if (!img || img->ch != 3 || x < 0 || y < 0 || w <= 0 || h <= 0 || x + w > img->w || y + h > img->h || (host && host_pitch < (size_t)w * 3) ||
        !valid_gain_args(gain_map, gw, gh, gc, gain_scalar)) {
        set_error("sb_gain_apply_dev: invalid argument");
        return SB_ERR_INVALID;
    }
    if (!gain_map && !gain_scalar) return SB_OK;  // compensator "no": identity (host and device copies stay as they are)
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    uint8_t *view = img->p + ((size_t)y * img->w + x) * 3;
    const long long pitch = (long long)img->w * 3;
    WarpJob job;
    std::memset(&job, 0, sizeof job);
    GainData gd;
    int rc = gain_upload(&job, &gd, w, h, gain_map, gw, gh, gc, gain_scalar, s);
    if (rc == SB_OK) rc = launch_gain_apply(view, pitch, w, h, job, s);
    if (rc == SB_OK && host && sb_copy2d(host, host_pitch, view, (size_t)pitch, (size_t)w * 3, h, cudaMemcpyDeviceToHost, s) != cudaSuccess)
        rc = SB_ERR_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess && rc == SB_OK) rc = SB_ERR_CUDA;
    gain_free(&gd, s);
    if (rc == SB_ERR_CUDA) set_error("sb_gain_apply_dev: CUDA failure");
    return rc;
}

int sb_timelapse_frame(const void *img, int is_s16, size_t pitch, const sb_devimg *dev, int dev_x, int dev_y, int w, int h, int tlx, int tly,
                       const int roi[4], uint8_t *dst, size_t dst_pitch)
{
    const size_t px = is_s16 ? 6 : 3;
    if ((!img && !dev) || !roi || !dst || w <= 0 || h <= 0 || roi[2] <= 0 || roi[3] <= 0 || dst_pitch < (size_t)roi[2] * 3 ||
        (long long)roi[2] * roi[3] > (1ll << 31) || (!dev && pitch < (size_t)w * px) ||
        (dev && (dev->ch != 3 || dev_x < 0 || dev_y < 0 || dev_x + w > dev->w || dev_y + h > dev->h))) {
        set_error("sb_timelapse_frame: invalid argument");
        return SB_ERR_INVALID;
    }
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    Scratch tmp(s);
    const int cw = roi[2], ch = roi[3];
    uint8_t *d_dst = nullptr, *d_src = nullptr;
    SB_TRY(tmp.get(&d_dst, (size_t)cw * 3 * ch));
    const uint8_t *src8 = nullptr;
    const int16_t *src16 = nullptr;
    long long spitch = 0;
    if (dev) {
        src8 = dev->p + ((size_t)dev_y * dev->w + dev_x) * 3;
        spitch = (long long)dev->w * 3;
    } else {
        // only the rows / columns that land on the canvas travel
        SB_TRY(tmp.get(&d_src, (size_t)w * px * h));
        SB_CUDA(sb_copy2d(d_src, (size_t)w * px, img, pitch, (size_t)w * px, h, cudaMemcpyHostToDevice, s));
        if (is_s16) {
            src16 = reinterpret_cast<const int16_t *>(d_src);
            spitch = (long long)w * 3;
        } else {
            src8 = d_src;
            spitch = (long long)w * 3;
        }
    }
    SB_TRY(launch_timelapse_frame(src8, src16, spitch, w, h, tlx - roi[0], tly - roi[1], d_dst, (long long)cw * 3, cw, ch, s));
    SB_CUDA(sb_copy2d(dst, dst_pitch, d_dst, (size_t)cw * 3, (size_t)cw * 3, ch, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));
    return SB_OK;
}

int sb_resize_exact(const uint8_t *src, size_t src_pitch, int sw, int sh, int channels, uint8_t *dst, size_t dst_pitch, int dw, int dh)
{
    if (!src || !dst || sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || (channels != 1 && channels != 3) ||
        src_pitch < (size_t)sw * channels || dst_pitch < (size_t)dw * channels || (long long)sw * sh * channels > (1ll << 31) ||
        (long long)dw * dh * channels > (1ll << 31)) {
        set_error("sb_resize_exact: invalid argument");
        return SB_ERR_INVALID;
    }
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    Scratch tmp(s);
    uint8_t *d_src = nullptr, *d_dst = nullptr;
    int *d_tx = nullptr, *d_ty = nullptr;
    const size_t srow = (size_t)sw * channels, drow = (size_t)dw * channels;
    SB_TRY(tmp.get(&d_src, srow * sh));
    SB_TRY(tmp.get(&d_dst, drow * dh));
    SB_TRY(tmp.get(&d_tx, (size_t)3 * dw));
    SB_TRY(tmp.get(&d_ty, (size_t)3 * dh));
    std::vector<int> tx((size_t)3 * dw), ty((size_t)3 * dh);
    resize_exact_taps(sw, dw, tx.data());
    resize_exact_taps(sh, dh, ty.data());
    SB_CUDA(sb_copy2d(d_src, srow, src, src_pitch, srow, sh, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_tx, tx.data(), tx.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_ty, ty.data(), ty.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    SB_TRY(launch_resize_exact(d_src, (long long)srow, channels, d_tx, d_ty, d_dst, (long long)drow, dw, dh, s));
    SB_CUDA(sb_copy2d(dst, dst_pitch, d_dst, drow, drow, dh, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));
    return SB_OK;
}

int sb_seam_resize(const uint8_t *seam, size_t seam_pitch, int sw, int sh, const uint8_t *mask, size_t mask_pitch, int w, int h,
                   uint8_t *dst, size_t dst_pitch)
{
    if (!seam || !mask || !dst || sw <= 0 || sh <= 0 || w <= 0 || h <= 0 || seam_pitch < (size_t)sw || mask_pitch < (size_t)w ||
        dst_pitch < (size_t)w || (long long)w * h > (1ll << 31) || (long long)sw * sh > (1ll << 31)) {
        set_error("sb_seam_resize: invalid argument");
        return SB_ERR_INVALID;
    }
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    Scratch tmp(s);
    uint8_t *d_mask = nullptr, *d_dst = nullptr;
    SB_TRY(tmp.get(&d_mask, (size_t)w * h));
    SB_TRY(tmp.get(&d_dst, (size_t)w * h));
    SB_CUDA(sb_copy2d(d_mask, w, mask, mask_pitch, w, h, cudaMemcpyHostToDevice, s));
    SB_TRY(seam_resize_device(seam, seam_pitch, sw, sh, d_mask, w, d_dst, w, w, h, s));
    SB_CUDA(sb_copy2d(dst, dst_pitch, d_dst, w, w, h, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));
    return SB_OK;
}

// -------------------------------------------------------------------------------------------------
// cv.cvtColor between BGR and YUV 4:2:0 (sb_yuv.cu) with host buffers
// -------------------------------------------------------------------------------------------------
static int check_yuv_size(const char *who, int fmt, int w, int h)
{
    if (fmt != SB_PIX_NV12 && fmt != SB_PIX_I420) {
        set_error("%s: format %d is not a YUV 4:2:0 format (SB_PIX_NV12, SB_PIX_I420)", who, fmt);
        return SB_ERR_INVALID;
    }
    if (w <= 0 || h <= 0 || (w | h) & 1 || (long long)w * h > (1ll << 31)) {
        set_error("%s: a YUV 4:2:0 frame needs an even width and height, got %dx%d", who, w, h);
        return SB_ERR_INVALID;
    }
    return SB_OK;
}

int sb_cvt_yuv420_to_bgr(int fmt, const uint8_t *const planes[3], const size_t pitches[3], int w, int h, uint8_t *dst, size_t dst_pitch)
{
    SB_TRY(check_yuv_size("sb_cvt_yuv420_to_bgr", fmt, w, h));
    if (!yuv_planes_ok(fmt, planes, pitches, w) || !dst || dst_pitch < (size_t)w * 3) {
        set_error("sb_cvt_yuv420_to_bgr: missing plane or short pitch");
        return SB_ERR_INVALID;
    }
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    Scratch tmp(s);
    uint8_t *d_yuv = nullptr, *d_bgr = nullptr;
    SB_TRY(tmp.get(&d_yuv, yuv_bytes(w, h)));
    SB_TRY(tmp.get(&d_bgr, (size_t)w * 3 * h));
    SB_CUDA(yuv_copy(d_yuv, planes, pitches, fmt, w, h, cudaMemcpyHostToDevice, s));
    SB_TRY(launch_yuv420_to_src(fmt, yuv_dense_planes(fmt, d_yuv, w, h), w, h, d_bgr, (long long)w * 3, nullptr, 0, s));
    SB_CUDA(sb_copy2d(dst, dst_pitch, d_bgr, (size_t)w * 3, (size_t)w * 3, h, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));
    return SB_OK;
}

int sb_cvt_bgr_to_yuv420(int fmt, const uint8_t *src, size_t src_pitch, int w, int h, uint8_t *const planes[3], const size_t pitches[3])
{
    SB_TRY(check_yuv_size("sb_cvt_bgr_to_yuv420", fmt, w, h));
    if (!yuv_planes_ok(fmt, planes, pitches, w) || !src || src_pitch < (size_t)w * 3) {
        set_error("sb_cvt_bgr_to_yuv420: missing plane or short pitch");
        return SB_ERR_INVALID;
    }
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    Scratch tmp(s);
    uint8_t *d_yuv = nullptr, *d_bgr = nullptr;
    SB_TRY(tmp.get(&d_yuv, yuv_bytes(w, h)));
    SB_TRY(tmp.get(&d_bgr, (size_t)w * 3 * h));
    SB_CUDA(sb_copy2d(d_bgr, (size_t)w * 3, src, src_pitch, (size_t)w * 3, h, cudaMemcpyHostToDevice, s));
    SB_TRY(launch_bgr_to_yuv420(fmt, d_bgr, (long long)w * 3, w, h, yuv_dense_out(fmt, d_yuv, w, h), s));
    SB_CUDA(yuv_copy(d_yuv, planes, pitches, fmt, w, h, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));
    return SB_OK;
}

// -------------------------------------------------------------------------------------------------
// Blender
// -------------------------------------------------------------------------------------------------
struct sb_blender {
    int kind;
    int num_bands;
    float sharpness;
    bool prepared = false;
    BlendPlan plan;
    std::vector<void *> level0;  // device buffers of the recorded feeds
};

sb_blender *sb_blender_create(int kind, int num_bands, float sharpness)
{
    if (kind < SB_BLEND_NO || kind > SB_BLEND_MULTIBAND) {
        set_error("sb_blender_create: unknown kind %d", kind);
        return nullptr;
    }
    sb_blender *b = new sb_blender;
    b->kind = kind;
    b->num_bands = num_bands;
    b->sharpness = sharpness;
    return b;
}

static void blender_drop_feeds(sb_blender *b)
{
    cudaStream_t s = default_stream();
    for (void *p : b->level0) dev_free(p, s);
    b->level0.clear();
    b->plan.release(s);
    b->plan.imgs.clear();
}

void sb_blender_destroy(sb_blender *b)
{
    if (!b) return;
    blender_drop_feeds(b);
    delete b;
}

int sb_blender_prepare(sb_blender *b, int x, int y, int w, int h)
{
    if (!b) {
        set_error("sb_blender_prepare: null handle");
        return SB_ERR_INVALID;
    }
    blender_drop_feeds(b);
    b->prepared = false;
    SB_TRY(b->plan.set_geometry(b->kind, b->num_bands, b->sharpness, Rect{x, y, w, h}));
    b->prepared = true;
    return SB_OK;
}

int sb_blender_num_bands(const sb_blender *b) { return b ? b->plan.nb : -1; }

// one recorded feed: geometry first (host only, so that an out-of-roi feed fails before any device work), then the level-0
// data on the device.  The image comes from the host (img) or from a device rectangle (dimg, dimg_pitch); likewise the mask.
static int blender_feed_impl(sb_blender *b, const void *img, int img_is_s16, size_t img_pitch, const uint8_t *dimg, size_t dimg_pitch,
                             const uint8_t *mask, size_t mask_pitch, const uint8_t *dmask, size_t dmask_pitch, int w, int h, int tl_x, int tl_y)
{
    FeedDesc f;
    std::memset(&f, 0, sizeof f);
    f.w = w; f.h = h; f.tlx = tl_x; f.tly = tl_y;
    SB_TRY(b->plan.add_feed(f));
    FeedImage &im = b->plan.imgs.back();
    const size_t px_bytes = img_is_s16 ? 6 : 3;
    auto upload = [&]() -> int {
        SB_TRY(ensure_device());
        cudaStream_t s = default_stream();
        const uint8_t *m_ptr = dmask;
        size_t m_pitch = dmask_pitch;
        if (!dmask) {
            uint8_t *d_mask = nullptr;
            SB_TRY(dev_alloc((void **)&d_mask, (size_t)w * h, s));
            b->level0.push_back(d_mask);
            SB_CUDA(sb_copy2d(d_mask, w, mask, mask_pitch, w, h, cudaMemcpyHostToDevice, s));
            m_ptr = d_mask;
            m_pitch = (size_t)w;
        }
        const uint8_t *i_ptr = dimg;
        size_t i_pitch = dimg_pitch;
        if (!dimg) {
            void *d_img = nullptr;
            SB_TRY(dev_alloc(&d_img, (size_t)w * h * px_bytes, s));
            b->level0.push_back(d_img);
            SB_CUDA(sb_copy2d(d_img, (size_t)w * px_bytes, img, img_pitch, (size_t)w * px_bytes, h, cudaMemcpyHostToDevice, s));
            i_ptr = (const uint8_t *)d_img;
            i_pitch = (size_t)w * px_bytes;
        }
        if (img_is_s16) {
            if (dmask) {  // the generic layout keeps a pointer to the mask: it has to outlive this call
                uint8_t *d_mask = nullptr;
                SB_TRY(dev_alloc((void **)&d_mask, (size_t)w * h, s));
                b->level0.push_back(d_mask);
                SB_CUDA(sb_copy2d(d_mask, w, dmask, dmask_pitch, w, h, cudaMemcpyDeviceToDevice, s));
                m_ptr = d_mask;
                m_pitch = (size_t)w;
            }
            im.s16 = (const int16_t *)i_ptr;
            im.s16_pitch = (long long)w * 3;
            im.mask = m_ptr;
            im.mask_pitch = (long long)m_pitch;
        } else {
            uint32_t *d_rgbm = nullptr;
            const int rp = (w + 3) & ~3;  // 16-byte rows: the tile kernels stage windows of this buffer with 16-byte copies
            SB_TRY(dev_alloc((void **)&d_rgbm, (size_t)rp * h * 4, s));
            b->level0.push_back(d_rgbm);
            if (rp != w) SB_CUDA(cudaMemsetAsync(d_rgbm, 0, (size_t)rp * h * 4, s));  // zero row padding = weight 0
            SB_TRY(launch_pack_rgbm(i_ptr, (long long)i_pitch, m_ptr, (long long)m_pitch, d_rgbm, rp, w, h, s));
            im.rgbm = d_rgbm;
            im.rgbm_pitch = rp;
        }
        // the caller's buffers (and device twins) may change as soon as we return
        SB_CUDA(cudaStreamSynchronize(s));
        return SB_OK;
    };
    const int rc = upload();
    if (rc != SB_OK) b->plan.imgs.pop_back();
    return rc;
}

int sb_blender_feed(sb_blender *b, const void *img, int img_is_s16, size_t img_pitch, const uint8_t *mask, size_t mask_pitch,
                    int w, int h, int tl_x, int tl_y)
{
    if (!b || !img || !mask || w <= 0 || h <= 0) {
        set_error("sb_blender_feed: invalid argument");
        return SB_ERR_INVALID;
    }
    if (!b->prepared) {
        set_error("sb_blender_feed: prepare() has not been called");
        return SB_ERR_STATE;
    }
    const size_t px_bytes = img_is_s16 ? 6 : 3;
    if (img_pitch < (size_t)w * px_bytes || mask_pitch < (size_t)w) {
        set_error("sb_blender_feed: pitch smaller than a row");
        return SB_ERR_INVALID;
    }
    return blender_feed_impl(b, img, img_is_s16, img_pitch, nullptr, 0, mask, mask_pitch, nullptr, 0, w, h, tl_x, tl_y);
}

int sb_blender_feed_dev(sb_blender *b, const sb_devimg *img, int ix, int iy, const sb_devimg *mask_dev, int mx, int my,
                        const uint8_t *mask_host, size_t mask_pitch, int w, int h, int tl_x, int tl_y)
{
    if (!b || !img || img->ch != 3 || w <= 0 || h <= 0 || ix < 0 || iy < 0 || ix + w > img->w || iy + h > img->h ||
        (!mask_dev && (!mask_host || mask_pitch < (size_t)w)) ||
        (mask_dev && (mask_dev->ch != 1 || mx < 0 || my < 0 || mx + w > mask_dev->w || my + h > mask_dev->h))) {
        set_error("sb_blender_feed_dev: invalid argument");
        return SB_ERR_INVALID;
    }
    if (!b->prepared) {
        set_error("sb_blender_feed_dev: prepare() has not been called");
        return SB_ERR_STATE;
    }
    const uint8_t *dimg = img->p + ((size_t)iy * img->w + ix) * 3;
    const uint8_t *dmask = mask_dev ? mask_dev->p + (size_t)my * mask_dev->w + mx : nullptr;
    return blender_feed_impl(b, nullptr, 0, 0, dimg, (size_t)img->w * 3, mask_host, mask_pitch, dmask, mask_dev ? (size_t)mask_dev->w : 0, w, h, tl_x,
                             tl_y);
}

int sb_blender_blend(sb_blender *b, uint8_t *dst, size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch, int16_t *dst_s16,
                     size_t s16_pitch)
{
    if (!b) {
        set_error("sb_blender_blend: null handle");
        return SB_ERR_INVALID;
    }
    if (!b->prepared) {
        set_error("sb_blender_blend: prepare() has not been called (or blend() was already called)");
        return SB_ERR_STATE;
    }
    const int w = b->plan.roi.w, h = b->plan.roi.h;
    if ((dst && dst_pitch < (size_t)w * 3) || (dst_mask && mask_pitch < (size_t)w) || (dst_s16 && s16_pitch < (size_t)w * 6)) {
        set_error("sb_blender_blend: destination pitch too small for roi width %d", w);
        return SB_ERR_INVALID;
    }
    SB_TRY(ensure_device());
    cudaStream_t s = default_stream();
    Scratch tmp(s);
    PanoOut out;
    std::memset(&out, 0, sizeof out);
    out.w = w;
    out.h = h;
    if (dst) {
        SB_TRY(tmp.get(&out.rgb, (size_t)w * 3 * h));
        out.rgb_pitch = (long long)w * 3;
    }
    if (dst_mask) {
        SB_TRY(tmp.get(&out.mask, (size_t)w * h));
        out.mask_pitch = w;
    }
    if (dst_s16) {
        SB_TRY(tmp.get(&out.s16, (size_t)w * 3 * h));
        out.s16_pitch = (long long)w * 3;
    }
    int rc = b->plan.allocate(s);
    if (rc == SB_OK) rc = b->plan.run(out, s);
    if (rc == SB_OK) {  // (errors fall through to the clean-up below: the feeds are dropped either way)
        cudaError_t e = cudaSuccess;
        if (dst) e = sb_copy2d(dst, dst_pitch, out.rgb, (size_t)w * 3, (size_t)w * 3, h, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess && dst_mask) e = sb_copy2d(dst_mask, mask_pitch, out.mask, w, w, h, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess && dst_s16) e = sb_copy2d(dst_s16, s16_pitch, out.s16, (size_t)w * 6, (size_t)w * 6, h, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) rc = cuda_fail(e, "sb_blender_blend: copy of the result", __FILE__, __LINE__);
    }
    // like OpenCV, blend() consumes the state: a new prepare() is needed before the next feed
    blender_drop_feeds(b);
    b->prepared = false;
    return rc;
}

}  // extern "C"
