// sb_compositor.cpp -- fused warp + blend with every intermediate resident in HBM.
//
// One compositor is the plan of one rig: what stitcher.py:178-189 (warp_final_resolution -> Warper.warp_images,
// create_and_warp_masks, warp_rois) and stitcher.py:241-259 (Blender.prepare / feed / blend) compute for a
// fixed set of cameras.  Creation does the host geometry once (roi detection, trig tables, padded rects,
// storage); run() enqueues warp -> pyramids -> collapse for a batch of frames without touching the host.
#include <algorithm>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "sb_plan.h"
#include "sb_shard.h"

namespace sb {
inline int rgbm_pitch_of(int w) { return (w + 31) & ~31; }

int make_warp_job(const Projector &p, const int rect[4], int src_w, int src_h, float *tab_dev, WarpJob *job, cudaStream_t s,
                  std::vector<float> &host_tab);
}
using namespace sb;

#define SB_PIPE_DEPTH 3  // buffer sets of the pipelined submit / wait path

struct sb_compositor {
    int n = 0;
    int warp_type = 0, blend_kind_requested = 0, mask_mode = 0;
    float scale = 1.f, blend_strength = 5.f;
    cudaStream_t stream = nullptr;
    std::vector<int> src_w, src_h;
    std::vector<Rect> rects;           // warped rects (pano-absolute)
    std::vector<WarpJob> jobs;         // host copy
    std::vector<WarpJob> jobsx[SB_PIPE_DEPTH - 1];  // the same jobs reading the extra source buffer sets (pipelined path)
    std::vector<uint8_t *> src_dev;    // u8x3 sources as uploaded
    std::vector<uint32_t *> src4_dev;  // the same, one word per pixel: what the warp kernel reads (repacked after every upload)
    std::vector<uint32_t *> src4_devx[SB_PIPE_DEPTH - 1];
    bool use_src4 = true;
    // YUV frames (sb_pix_fmt): src4_only[i] when the warp kernel reads image i's word-per-pixel source and never the 3-byte
    // one, which then stages the YUV upload (3 B/px >= 1.5 B/px); otherwise the YUV frame has a staging buffer of its own
    // per buffer slot.  yuv_out: the YUV panorama of each slot.  All allocated on first use.
    std::vector<char> src4_only;
    std::vector<uint8_t *> yuv_in[SB_PIPE_DEPTH];
    uint8_t *yuv_out[SB_PIPE_DEPTH] = {};
    std::vector<uint32_t *> rgbm_dev;  // warped, packed; row pitch = width rounded up to 32 pixels (128-byte rows)
    std::vector<float *> tab_dev;
    std::vector<float *> maps_dev;     // projections that are not separable: xmap | ymap of every image (built at plan time)
    std::vector<uint8_t *> usermask_dev;
    std::vector<GainData> gain;        // exposure gains per image (sb_compositor_set_gain)
    int max_w = 0, max_h = 0;
    BlendPlan plan;
    PanoOut out{};                     // device outputs
    void *flush_buf = nullptr;
    size_t flush_bytes = 0;
    std::vector<cudaEvent_t> ev;       // ev[0] = start, ev[k+1] = after launch k
    std::vector<std::string> launch_names;
    std::vector<float> launch_ms;      // per launch, averaged over the last sb_compositor_time call
    double warp_bytes = 0;
    // pipelined submit / wait: a second set of source + output buffers, copy streams, per-slot events
    bool pipe_ready = false;
    std::vector<uint8_t *> src_devx[SB_PIPE_DEPTH - 1];
    PanoOut outx[SB_PIPE_DEPTH - 1] = {};
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaEvent_t e_h2d[SB_PIPE_DEPTH] = {}, e_comp[SB_PIPE_DEPTH] = {}, e_d2h[SB_PIPE_DEPTH] = {};
    unsigned long long submitted = 0;
#ifndef SB_EMU
    cudaGraphExec_t graph_exec[SB_PIPE_DEPTH] = {};  // one captured step per buffer slot
#endif
    unsigned graph_kernels = 0;
    std::vector<cudaEvent_t> tev;  // step start / end events of sb_compositor_time
    // multi-GPU: this process composites images [first, first + count) and one column strip of the panorama
    bool sharded = false;
    int first = 0, count = 0;
    // the slab exchange runs on its own stream, in two parts, beside the kernels (see compositor_enqueue_kernels)
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t e_part[2] = {}, e_xchg[2] = {};  // partial sums of part k written / part k received
    ShardPlan shard;
};

static void compositor_free(sb_compositor *c)
{
    if (!c) return;
    cudaStream_t s = c->stream ? c->stream : default_stream();
    if (c->stream) (void)cudaStreamSynchronize(c->stream);
    for (auto p : c->src_dev) dev_free(p, s);
    for (auto p : c->src4_dev) dev_free(p, s);
    for (auto &v : c->src4_devx)
        for (auto p : v) dev_free(p, s);
    if (c->h2d) (void)cudaStreamSynchronize(c->h2d);
    if (c->d2h) (void)cudaStreamSynchronize(c->d2h);
    for (auto &v : c->yuv_in)
        for (auto p : v) dev_free(p, s);
    for (auto p : c->yuv_out) dev_free(p, s);
    for (auto p : c->rgbm_dev) dev_free(p, s);
    for (auto p : c->tab_dev) dev_free(p, s);
    for (auto p : c->maps_dev) dev_free(p, s);
    for (auto p : c->usermask_dev) dev_free(p, s);
    for (auto &g : c->gain) gain_free(&g, s);
    dev_free(c->out.rgb, s);
    dev_free(c->out.mask, s);
    dev_free(c->flush_buf, s);
    if (c->h2d) (void)cudaStreamSynchronize(c->h2d);
    if (c->d2h) (void)cudaStreamSynchronize(c->d2h);
    for (auto &v : c->src_devx)
        for (auto p : v) dev_free(p, s);
    if (c->pipe_ready) {
        for (auto &o : c->outx) {
            dev_free(o.rgb, s);
            dev_free(o.mask, s);
        }
    }
    for (int k = 0; k < SB_PIPE_DEPTH; ++k) {
        if (c->e_h2d[k]) (void)cudaEventDestroy(c->e_h2d[k]);
        if (c->e_comp[k]) (void)cudaEventDestroy(c->e_comp[k]);
        if (c->e_d2h[k]) (void)cudaEventDestroy(c->e_d2h[k]);
    }
    if (c->h2d) (void)cudaStreamDestroy(c->h2d);
    if (c->d2h) (void)cudaStreamDestroy(c->d2h);
    if (c->comm_stream) {
        (void)cudaStreamSynchronize(c->comm_stream);
        (void)cudaStreamDestroy(c->comm_stream);
    }
    for (int k = 0; k < 2; ++k) {
        if (c->e_part[k]) (void)cudaEventDestroy(c->e_part[k]);
        if (c->e_xchg[k]) (void)cudaEventDestroy(c->e_xchg[k]);
    }
#ifndef SB_EMU
    for (auto &g : c->graph_exec)
        if (g) (void)cudaGraphExecDestroy(g);
#endif
    for (auto &e : c->tev) (void)cudaEventDestroy(e);
    c->shard.release(s);
    c->plan.release(s);
    for (auto &e : c->ev)
        if (e) (void)cudaEventDestroy(e);
    if (c->stream) {
        (void)cudaStreamSynchronize(c->stream);
        (void)cudaStreamDestroy(c->stream);
    }
    delete c;
}

static int compositor_build(sb_compositor *c, const sb_rig *rig, int rank, int world)
{
    const int n = rig->n_images;
    c->n = n;
    c->sharded = world > 1;
    c->first = 0;
    c->count = n;
    if (c->sharded) ShardPlan::block_of(n, world, rank, &c->first, &c->count);
    auto mine = [&](int i) { return i >= c->first && i < c->first + c->count; };
    c->warp_type = rig->warp_type;
    c->scale = rig->scale;
    c->blend_kind_requested = rig->blend_kind;
    c->blend_strength = rig->blend_strength;
    c->mask_mode = rig->mask_mode;
    SB_TRY(ensure_device());
    SB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    cudaStream_t s = c->stream;

    c->src_w.assign(rig->src_w, rig->src_w + n);
    c->src_h.assign(rig->src_h, rig->src_h + n);
    c->rects.resize(n);
    c->jobs.resize(n);
    c->src_dev.assign(n, nullptr);
    c->src4_dev.assign(n, nullptr);
    {
        const char *e = getenv("SB_SRC4");  // SB_SRC4=0: the warp kernel reads the packed 3-byte sources (A/B switch)
        c->use_src4 = !(e && e[0] == '0');
    }
    c->rgbm_dev.assign(n, nullptr);
    c->tab_dev.assign(n, nullptr);
    c->maps_dev.assign(n, nullptr);
    c->usermask_dev.assign(n, nullptr);
    c->gain.assign(n, GainData{});
    std::vector<int> corners(2 * n), sizes(2 * n);
    std::vector<float> host_tab;
    for (int i = 0; i < n; ++i) {
        Projector p;
        projector_setup(p, rig->warp_type, rig->scale, rig->K + 9 * i, rig->R + 9 * i);
        int rect[4];
        projector_roi(p, c->src_w[i], c->src_h[i], rect);
        if (rect[2] <= 0 || rect[3] <= 0 || (long long)rect[2] * rect[3] > (1ll << 31)) {
            set_error("compositor: degenerate warped roi %dx%d for image %d", rect[2], rect[3], i);
            return SB_ERR_INVALID;
        }
        c->rects[i] = Rect{rect[0], rect[1], rect[2], rect[3]};
        corners[2 * i] = rect[0];
        corners[2 * i + 1] = rect[1];
        sizes[2 * i] = rect[2];
        sizes[2 * i + 1] = rect[3];
        c->max_w = std::max(c->max_w, rect[2]);
        c->max_h = std::max(c->max_h, rect[3]);
        if (!mine(i)) continue;  // another rank warps this image: only its geometry is needed here
        SB_TRY(dev_alloc((void **)&c->src_dev[i], (size_t)c->src_w[i] * 3 * c->src_h[i] + SB_SRC_PAD, s));
        SB_TRY(dev_alloc((void **)&c->rgbm_dev[i], (size_t)rgbm_pitch_of(rect[2]) * rect[3] * 4, s));
        // the row padding (never written by the warp kernel) is read by the tile kernels' 16-byte copies: weight 0
        SB_CUDA(cudaMemsetAsync(c->rgbm_dev[i], 0, (size_t)rgbm_pitch_of(rect[2]) * rect[3] * 4, s));
        SB_TRY(dev_alloc((void **)&c->tab_dev[i], warp_table_floats(rect[2], rect[3]) * sizeof(float), s));
        SB_TRY(make_warp_job(p, rect, c->src_w[i], c->src_h[i], c->tab_dev[i], &c->jobs[i], s, host_tab));
        SB_CUDA(cudaStreamSynchronize(s));  // host_tab is reused by the next image
        if (projector_needs_maps(p)) {
            SB_TRY(dev_alloc((void **)&c->maps_dev[i], (size_t)2 * rect[2] * rect[3] * sizeof(float), s));
            SB_TRY(warp_maps_upload(p, rect, c->maps_dev[i], &c->jobs[i], s));
        }
        c->jobs[i].src = c->src_dev[i];
        c->jobs[i].spitch = (long long)c->src_w[i] * 3;
        if (c->use_src4 && (long long)c->src_w[i] * c->src_h[i] < (1ll << 31)) {
            SB_TRY(dev_alloc((void **)&c->src4_dev[i], ((size_t)c->src_w[i] * c->src_h[i] + 4) * sizeof(uint32_t), s));
            c->jobs[i].src4 = c->src4_dev[i];
        }
        c->jobs[i].dst_rgbm = c->rgbm_dev[i];
        c->jobs[i].rgbm_pitch = rgbm_pitch_of(rect[2]);
        c->warp_bytes += 3.0 * c->src_w[i] * c->src_h[i] + 4.0 * rect[2] * rect[3];
    }
    c->src4_only.assign(n, 0);
    for (int i = c->first; i < c->first + c->count; ++i)
        c->src4_only[i] = warp_reads_src4_only(c->jobs.data() + c->first, c->count, i - c->first);

    // Blender.prepare (blender.py:23-38)
    const Rect roi = result_roi(corners.data(), sizes.data(), n);
    int kind, nbr;
    float sharp;
    derive_blend_params(rig->blend_kind, rig->blend_strength, roi, &kind, &nbr, &sharp);
    SB_TRY(c->plan.set_geometry(kind, nbr, sharp, roi));
    {
        // the mask byte of a warped pixel is the validity test's 0 / 255 until a caller supplies masks (SB_PD_BIN=0: A/B switch)
        const char *e = getenv("SB_PD_BIN");
        c->plan.binary_masks = !(e && e[0] == '0');
    }
    for (int i = 0; i < n; ++i) {
        FeedDesc f;
        std::memset(&f, 0, sizeof f);
        f.w = c->rects[i].w;
        f.h = c->rects[i].h;
        f.tlx = c->rects[i].x;
        f.tly = c->rects[i].y;
        f.rgbm = c->rgbm_dev[i];
        f.rgbm_pitch = rgbm_pitch_of(c->rects[i].w);
        SB_TRY(c->plan.add_feed(f));
    }
    int out_w = roi.w, out_h = roi.h;
    if (c->sharded) {
        c->plan.active_first = c->first;
        c->plan.active_count = c->count;
        SB_TRY(c->shard.build(c->plan, rank, world));
        int lo, hi;
        c->shard.strip(c->plan, &lo, &hi);
        if (c->shard.axis == 0)
            out_w = hi - lo;
        else
            out_h = hi - lo;  // row strips (feather, image blocks stacked vertically)
    }
    SB_TRY(c->plan.allocate(s));
    if (c->sharded) SB_TRY(c->shard.allocate(c->plan, s));
    std::memset(&c->out, 0, sizeof c->out);
    c->out.w = out_w;
    c->out.h = out_h;
    c->out.rgb_pitch = (long long)out_w * 3;
    c->out.mask_pitch = out_w;
    SB_TRY(dev_alloc((void **)&c->out.rgb, (size_t)std::max(out_w, 1) * 3 * std::max(out_h, 1), s));
    SB_TRY(dev_alloc((void **)&c->out.mask, (size_t)std::max(out_w, 1) * std::max(out_h, 1), s));
    SB_CUDA(cudaStreamSynchronize(s));
    return SB_OK;
}

static int compositor_enqueue_kernels(sb_compositor *c, bool events, int slot);

// One step = one CUDA graph launch: the plan is static, so the ~2(nb+1) kernel launches are captured once per
// buffer slot and replayed (the coarse levels are launch-latency bound).  SB_GRAPH=0 launches them one by one.
static int compositor_enqueue(sb_compositor *c, bool events, int slot = 0)
{
#ifndef SB_EMU
    static const bool use_graph = [] {
        const char *e = getenv("SB_GRAPH");
        return !(e && e[0] == '0');
    }();
    if (!events && use_graph && !c->sharded) {  // (the sharded step contains the NCCL exchange: launched directly)
        cudaStream_t s = c->stream;
        if (!c->graph_exec[slot]) {
            const unsigned long long before = sb_launch_count();
            SB_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
            const int rc = compositor_enqueue_kernels(c, false, slot);
            cudaGraph_t g = nullptr;
            const cudaError_t e = cudaStreamEndCapture(s, &g);
            c->graph_kernels = (unsigned)(sb_launch_count() - before);
            adjust_launch_count(-(long long)c->graph_kernels);  // captured, not executed
            if (rc != SB_OK) {
                if (g) (void)cudaGraphDestroy(g);
                return rc;
            }
            if (e != cudaSuccess) return cuda_fail(e, "cudaStreamEndCapture", __FILE__, __LINE__);
            const cudaError_t ei = cudaGraphInstantiate(&c->graph_exec[slot], g, 0);
            (void)cudaGraphDestroy(g);
            if (ei != cudaSuccess) return cuda_fail(ei, "cudaGraphInstantiate", __FILE__, __LINE__);
        }
        SB_CUDA(cudaGraphLaunch(c->graph_exec[slot], s));
        adjust_launch_count((long long)c->graph_kernels);
        return SB_OK;
    }
#endif
    return compositor_enqueue_kernels(c, events, slot);
}

// sharded step: pyrDown of level l -> l+1 for the own images
static int shard_pyrdown(sb_compositor *c, cudaStream_t s, int l)
{
    BlendPlan &P = c->plan;
    const int n = (int)P.imgs.size();
    int mw = 0, mh = 0;
    for (int i = c->first; i < c->first + c->count; ++i) {
        mw = std::max(mw, P.imgs[i].pw >> (l + 1));
        mh = std::max(mh, P.imgs[i].ph >> (l + 1));
    }
    return launch_pyrdown(P.imgs_dev, P.imgs.data(), P.pyr_dev + (size_t)l * n, c->first, c->count, l, mw, mh, s, P.binary_masks);
}

// sharded step, local part: pyramids of the own images, then the partial sums every neighbour needs
static int shard_feather_weights(sb_compositor *c, cudaStream_t s)
{
    BlendPlan &P = c->plan;
    return launch_feather_weights(P.imgs_dev + c->first, P.imgs.data() + c->first, c->count, P.sharpness, s);
}

static int shard_local(sb_compositor *c, cudaStream_t s, const std::function<int(const std::string &)> &mark)
{
    if (c->plan.kind == SB_BLEND_FEATHER) {
        SB_TRY(shard_feather_weights(c, s));
        SB_TRY(mark("feather_weights"));
        SB_TRY(c->shard.feather_partial_out(c->plan, s));
        SB_TRY(mark("partial_out"));
        return SB_OK;
    }
    for (int l = 0; l < c->plan.nb; ++l) {
        SB_TRY(shard_pyrdown(c, s, l));
        SB_TRY(mark("pyrdown_l" + std::to_string(l)));
    }
    SB_TRY(c->shard.partial_out(c->plan, s));
    SB_TRY(mark("partial_out"));
    return SB_OK;
}

static int compositor_enqueue_kernels(sb_compositor *c, bool events, int slot)
{
    cudaStream_t s = c->stream;
    size_t k = 0;
    auto mark = [&](const std::string &name) -> int {
        if (!events) return SB_OK;
        if (c->ev.size() <= k) {
            cudaEvent_t e;
            SB_CUDA(cudaEventCreate(&e));
            c->ev.push_back(e);
        }
        SB_CUDA(cudaEventRecord(c->ev[k], s));
        if (k > 0) {
            if (c->launch_names.size() < k) c->launch_names.push_back(name);
        }
        ++k;
        return SB_OK;
    };
    SB_TRY(mark("start"));
    const WarpJob *jobs = slot ? c->jobsx[slot - 1].data() : c->jobs.data();
    SB_TRY(launch_warp(jobs + c->first, c->count, s));
    SB_TRY(mark("warp"));
    const PanoOut &out = slot ? c->outx[slot - 1] : c->out;
    if (!c->sharded) return c->plan.run(out, s, events ? std::function<int(const std::string &)>(mark) : nullptr);
    if (!c->comm_stream) {
        SB_CUDA(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            SB_CUDA(cudaEventCreateWithFlags(&c->e_part[k], cudaEventDisableTiming));
            SB_CUDA(cudaEventCreateWithFlags(&c->e_xchg[k], cudaEventDisableTiming));
        }
    }
    BlendPlan &P0 = c->plan;
    if (P0.kind == SB_BLEND_FEATHER) {
        // single level: distance-transform weights of the own images, partial sums for the neighbours, one exchange, finish
        SB_TRY(shard_feather_weights(c, s));
        SB_TRY(mark("feather_weights"));
        if (c->shard.connected) {
            const unsigned step = ++c->shard.step;
            if (step > 1) SB_CUDA(cudaStreamWaitEvent(s, c->e_xchg[1], 0));  // the previous step's copies have left the send buffers
            SB_TRY(c->shard.feather_partial_out(P0, s));
            SB_TRY(mark("partial_out"));
            SB_CUDA(cudaEventRecord(c->e_part[0], s));
            SB_CUDA(cudaStreamWaitEvent(c->comm_stream, c->e_part[0], 0));
            SB_TRY(c->shard.wait_consumed(c->comm_stream, step - 1));
            SB_TRY(c->shard.push(c->comm_stream, 0));
            SB_TRY(c->shard.signal_data(c->comm_stream, 0, step));
            SB_CUDA(cudaEventRecord(c->e_xchg[1], c->comm_stream));
            SB_TRY(c->shard.wait_data(s, 0, step));
            SB_TRY(c->shard.feather_finish(P0, out, s));
            SB_TRY(c->shard.signal_consumed(s, step));
        } else {
            SB_TRY(c->shard.feather_partial_out(P0, s));
            SB_TRY(mark("partial_out"));
            SB_CUDA(cudaEventRecord(c->e_part[0], s));
            SB_CUDA(cudaStreamWaitEvent(c->comm_stream, c->e_part[0], 0));
            SB_TRY(c->shard.exchange(c->comm_stream, -1));
            SB_CUDA(cudaEventRecord(c->e_xchg[0], c->comm_stream));
            SB_CUDA(cudaStreamWaitEvent(s, c->e_xchg[0], 0));
            SB_TRY(c->shard.feather_finish(P0, out, s));
        }
        SB_TRY(mark("feather_finish"));
        return SB_OK;
    }
    if (c->shard.connected) {
        // Exchange over mapped peer memory (sb_peer.cpp): the slabs go from the local send buffers into the owners' arenas
        // with copy-engine copies on the communication stream, beside the pyramid kernels; flags written / awaited by
        // stream memory operations order the ranks (no host round trip, no NCCL call in the step).
        const unsigned step = ++c->shard.step;
        const bool direct = c->shard.direct_stores;
        cudaStream_t cs = direct ? s : c->comm_stream;
        SB_TRY(shard_pyrdown(c, s, 0));
        SB_TRY(mark("pyrdown_l0"));
        if (step > 1 && !direct) SB_CUDA(cudaStreamWaitEvent(s, c->e_xchg[1], 0));  // the previous step's copies have left the send buffers
        if (direct) SB_TRY(c->shard.wait_consumed(s, step - 1));
        SB_TRY(c->shard.partial_out(P0, s, 0, 0, direct));
        SB_TRY(mark("partial_l0"));
        if (!direct) {
            SB_CUDA(cudaEventRecord(c->e_part[0], s));
            SB_CUDA(cudaStreamWaitEvent(cs, c->e_part[0], 0));
            SB_TRY(c->shard.wait_consumed(cs, step - 1));  // the neighbours have read what the previous step delivered
            SB_TRY(c->shard.push(cs, 0));
        }
        SB_TRY(c->shard.signal_data(cs, 0, step));
        for (int l = 1; l < P0.nb; ++l) {
            SB_TRY(shard_pyrdown(c, s, l));
            SB_TRY(mark("pyrdown_l" + std::to_string(l)));
        }
        SB_TRY(c->shard.partial_out(P0, s, 1, P0.nb, direct));
        SB_TRY(mark("partial_coarse"));
        if (!direct) {
            SB_CUDA(cudaEventRecord(c->e_part[1], s));
            SB_CUDA(cudaStreamWaitEvent(cs, c->e_part[1], 0));
            SB_TRY(c->shard.push(cs, 1));
        }
        SB_TRY(c->shard.signal_data(cs, 1, step));
        if (!direct) SB_CUDA(cudaEventRecord(c->e_xchg[1], cs));
        SB_TRY(c->shard.wait_data(s, 1, step));
        SB_TRY(c->shard.finish(P0, out, s, P0.nb, 1));
        SB_TRY(mark("finish_coarse"));  // includes waiting for the coarse slabs of the neighbours
        SB_TRY(c->shard.wait_data(s, 0, step));
        SB_TRY(c->shard.finish(P0, out, s, 0, 0));
        SB_TRY(c->shard.signal_consumed(s, step));
        SB_TRY(mark("finish_l0"));      // includes waiting for the level-0 slabs
        return SB_OK;
    }
    // The exchange overlaps the kernels.  Level 0 of the partial sums -- three quarters of the bytes -- needs only the
    // first pyrDown, and the collapse reads it last: its slabs travel on the communication stream while the rest of the
    // pyramid, the coarser partial sums, their (small) exchange and the collapse of levels nb..1 run.
    BlendPlan &P = c->plan;
    SB_TRY(shard_pyrdown(c, s, 0));
    SB_TRY(mark("pyrdown_l0"));
    SB_TRY(c->shard.partial_out(P, s, 0, 0));
    SB_TRY(mark("partial_l0"));
    SB_CUDA(cudaEventRecord(c->e_part[0], s));
    SB_CUDA(cudaStreamWaitEvent(c->comm_stream, c->e_part[0], 0));
    SB_TRY(c->shard.exchange(c->comm_stream, 0));
    SB_CUDA(cudaEventRecord(c->e_xchg[0], c->comm_stream));
    for (int l = 1; l < P.nb; ++l) {
        SB_TRY(shard_pyrdown(c, s, l));
        SB_TRY(mark("pyrdown_l" + std::to_string(l)));
    }
    SB_TRY(c->shard.partial_out(P, s, 1, P.nb));
    SB_TRY(mark("partial_coarse"));
    SB_CUDA(cudaEventRecord(c->e_part[1], s));
    SB_CUDA(cudaStreamWaitEvent(c->comm_stream, c->e_part[1], 0));
    SB_TRY(c->shard.exchange(c->comm_stream, 1));
    SB_CUDA(cudaEventRecord(c->e_xchg[1], c->comm_stream));
    SB_CUDA(cudaStreamWaitEvent(s, c->e_xchg[1], 0));
    SB_TRY(c->shard.finish(P, out, s, P.nb, 1));
    SB_TRY(mark("finish_coarse"));  // includes waiting for the coarse slabs of the neighbours
    SB_CUDA(cudaStreamWaitEvent(s, c->e_xchg[0], 0));
    SB_TRY(c->shard.finish(P, out, s, 0, 0));
    SB_TRY(mark("finish_l0"));      // includes waiting for the level-0 slabs
    return SB_OK;
}

// second buffer set + copy streams for sb_compositor_submit / _wait
static int compositor_pipe_init(sb_compositor *c)
{
    if (c->pipe_ready) return SB_OK;
    cudaStream_t s = c->stream;
    for (int k = 0; k < SB_PIPE_DEPTH - 1; ++k) {
        c->src_devx[k].assign(c->n, nullptr);
        c->jobsx[k] = c->jobs;
        for (int i = 0; i < c->n; ++i) {
            SB_TRY(dev_alloc((void **)&c->src_devx[k][i], (size_t)c->src_w[i] * 3 * c->src_h[i] + SB_SRC_PAD, s));
            c->jobsx[k][i].src = c->src_devx[k][i];
            if (c->jobs[i].src4) {
                if (c->src4_devx[k].empty()) c->src4_devx[k].assign(c->n, nullptr);
                SB_TRY(dev_alloc((void **)&c->src4_devx[k][i], ((size_t)c->src_w[i] * c->src_h[i] + 4) * sizeof(uint32_t), s));
                c->jobsx[k][i].src4 = c->src4_devx[k][i];
            }
        }
        c->outx[k] = c->out;
        c->outx[k].rgb = nullptr;
        c->outx[k].mask = nullptr;
        SB_TRY(dev_alloc((void **)&c->outx[k].rgb, (size_t)c->out.w * 3 * c->out.h, s));
        SB_TRY(dev_alloc((void **)&c->outx[k].mask, (size_t)c->out.w * c->out.h, s));
    }
    SB_CUDA(cudaStreamCreateWithFlags(&c->h2d, cudaStreamNonBlocking));
    SB_CUDA(cudaStreamCreateWithFlags(&c->d2h, cudaStreamNonBlocking));
    for (int k = 0; k < SB_PIPE_DEPTH; ++k) {
        SB_CUDA(cudaEventCreateWithFlags(&c->e_h2d[k], cudaEventDisableTiming));
        SB_CUDA(cudaEventCreateWithFlags(&c->e_comp[k], cudaEventDisableTiming));
        SB_CUDA(cudaEventCreateWithFlags(&c->e_d2h[k], cudaEventDisableTiming));
    }
    SB_CUDA(cudaStreamSynchronize(s));
    c->pipe_ready = true;
    return SB_OK;
}

// ---- frames in other pixel formats (sb_pix_fmt) ----------------------------------------------------------------------
static bool valid_fmt(int fmt) { return fmt == SB_PIX_BGR || fmt == SB_PIX_NV12 || fmt == SB_PIX_I420; }

static uint8_t *src_of(sb_compositor *c, int slot, int i) { return slot ? c->src_devx[slot - 1][i] : c->src_dev[i]; }
static uint32_t *src4_of(sb_compositor *c, int slot, int i)
{
    return slot ? (c->src4_devx[slot - 1].empty() ? nullptr : c->src4_devx[slot - 1][i]) : c->src4_dev[i];
}
static uint8_t *yuv_stage_of(sb_compositor *c, int slot, int i) { return c->src4_only[i] ? src_of(c, slot, i) : c->yuv_in[slot][i]; }

// the buffers a YUV step of `slot` needs (sources staged when in_fmt is YUV, the panorama when out_fmt is YUV), allocated
// on first use; synchronises the compute stream after an allocation, so that any stream may use them next
static int yuv_buffers(sb_compositor *c, int slot, int in_fmt, int out_fmt)
{
    cudaStream_t s = c->stream;
    bool allocated = false;
    if (in_fmt != SB_PIX_BGR) {
        auto &v = c->yuv_in[slot];
        if (v.empty()) v.assign(c->n, nullptr);
        for (int i = 0; i < c->n; ++i)
            if (!c->src4_only[i] && !v[i]) {
                SB_TRY(dev_alloc((void **)&v[i], yuv_bytes(c->src_w[i], c->src_h[i]), s));
                allocated = true;
            }
    }
    if (out_fmt != SB_PIX_BGR && !c->yuv_out[slot]) {
        SB_TRY(dev_alloc((void **)&c->yuv_out[slot], yuv_bytes(c->out.w, c->out.h), s));
        allocated = true;
    }
    if (allocated) SB_CUDA(cudaStreamSynchronize(s));
    return SB_OK;
}

// cv.cvtColor(COLOR_YUV2BGR_*) of the staged frame of image i into exactly the source the warp kernel reads
static int yuv_convert_source(sb_compositor *c, int slot, int i, int fmt, cudaStream_t s)
{
    const int w = c->src_w[i], h = c->src_h[i];
    const YuvPlanes in = yuv_dense_planes(fmt, yuv_stage_of(c, slot, i), w, h);
    if (c->src4_only[i]) return launch_yuv420_to_src(fmt, in, w, h, nullptr, 0, src4_of(c, slot, i), w, s);
    return launch_yuv420_to_src(fmt, in, w, h, src_of(c, slot, i), (long long)w * 3, nullptr, 0, s);
}

// the checks a YUV frame of the panorama (is_out) or of source image i has to pass
static int yuv_frame_ok(const sb_compositor *c, const char *who, int fmt, bool is_out, int i)
{
    if (fmt == SB_PIX_BGR) return SB_OK;
    if (c->sharded) {
        set_error("%s: YUV frames need a single-GPU compositor", who);
        return SB_ERR_STATE;
    }
    const int w = is_out ? c->out.w : c->src_w[i], h = is_out ? c->out.h : c->src_h[i];
    if ((w | h) & 1) {
        if (is_out)
            set_error("%s: a YUV 4:2:0 panorama needs an even width and height, the panorama is %dx%d", who, w, h);
        else
            set_error("%s: a YUV 4:2:0 frame needs an even width and height, image %d is %dx%d", who, i, w, h);
        return SB_ERR_INVALID;
    }
    return SB_OK;
}

static int upload_frame(sb_compositor *c, int i, int fmt, const uint8_t *const planes[3], const size_t pitches[3], int pinned,
                        const char *who)
{
    if (!c || i < 0 || i >= c->n || !valid_fmt(fmt) || !planes || !pitches) {
        set_error("%s: invalid argument", who);
        return SB_ERR_INVALID;
    }
    if (fmt == SB_PIX_BGR) {
        const uint8_t *src = planes[0];
        const size_t pitch = pitches[0];
        if (!src || pitch < (size_t)c->src_w[i] * 3) {
            set_error("%s: invalid argument", who);
            return SB_ERR_INVALID;
        }
        if (!c->src_dev[i]) {
            set_error("%s: image %d belongs to another rank (this rank owns %d..%d)", who, i, c->first, c->first + c->count - 1);
            return SB_ERR_INVALID;
        }
        SB_CUDA(sb_copy2d(c->src_dev[i], (size_t)c->src_w[i] * 3, src, pitch, (size_t)c->src_w[i] * 3, c->src_h[i],
                          cudaMemcpyHostToDevice, c->stream));
        if (c->src4_dev[i]) SB_TRY(launch_repack_rgbx(c->src_dev[i], c->src4_dev[i], (long long)c->src_w[i] * c->src_h[i], c->stream));
    } else {
        SB_TRY(yuv_frame_ok(c, who, fmt, false, i));
        if (!yuv_planes_ok(fmt, planes, pitches, c->src_w[i])) {
            set_error("%s: image %d: missing plane or short pitch", who, i);
            return SB_ERR_INVALID;
        }
        SB_TRY(yuv_buffers(c, 0, fmt, SB_PIX_BGR));
        SB_CUDA(yuv_copy(yuv_stage_of(c, 0, i), planes, pitches, fmt, c->src_w[i], c->src_h[i], cudaMemcpyHostToDevice, c->stream));
        SB_TRY(yuv_convert_source(c, 0, i, fmt, c->stream));
    }
    if (!pinned) SB_CUDA(cudaStreamSynchronize(c->stream));
    return SB_OK;
}

static int download_frame(sb_compositor *c, int fmt, uint8_t *const planes[3], const size_t pitches[3], uint8_t *dst_mask,
                          size_t mask_pitch, const char *who)
{
    uint8_t *dst = planes ? planes[0] : nullptr;
    if (!c || !valid_fmt(fmt) || (dst && !pitches) || (dst_mask && mask_pitch < (size_t)c->out.w) ||
        (dst && fmt == SB_PIX_BGR && pitches[0] < (size_t)c->out.w * 3)) {
        set_error("%s: invalid argument", who);
        return SB_ERR_INVALID;
    }
    if (dst && fmt != SB_PIX_BGR) {
        SB_TRY(yuv_frame_ok(c, who, fmt, true, 0));
        if (!yuv_planes_ok(fmt, planes, pitches, c->out.w)) {
            set_error("%s: missing plane or short pitch", who);
            return SB_ERR_INVALID;
        }
        SB_TRY(yuv_buffers(c, 0, SB_PIX_BGR, fmt));
        // slot 0's YUV panorama may still be on its way to the host from a submitted step
        if (c->pipe_ready) SB_CUDA(cudaStreamWaitEvent(c->stream, c->e_d2h[0], 0));
        SB_TRY(launch_bgr_to_yuv420(fmt, c->out.rgb, c->out.rgb_pitch, c->out.w, c->out.h, yuv_dense_out(fmt, c->yuv_out[0], c->out.w, c->out.h),
                                    c->stream));
        SB_CUDA(yuv_copy(c->yuv_out[0], planes, pitches, fmt, c->out.w, c->out.h, cudaMemcpyDeviceToHost, c->stream));
    } else if (dst) {
        SB_CUDA(sb_copy2d(dst, pitches[0], c->out.rgb, (size_t)c->out.rgb_pitch, (size_t)c->out.w * 3, c->out.h, cudaMemcpyDeviceToHost,
                          c->stream));
    }
    if (dst_mask)
        SB_CUDA(sb_copy2d(dst_mask, mask_pitch, c->out.mask, (size_t)c->out.mask_pitch, c->out.w, c->out.h,
                                  cudaMemcpyDeviceToHost, c->stream));
    SB_CUDA(cudaStreamSynchronize(c->stream));
    return SB_OK;
}

// Pipelined end-to-end step: H2D of this batch, warp + blend, D2H of the panorama are enqueued on three
// streams and chained with events; with three buffer sets the copies of a step overlap the kernels and copies of its neighbours.
static int submit_frames(sb_compositor *c, int in_fmt, const uint8_t *const *planes, const size_t *pitches, int out_fmt,
                         uint8_t *const out_planes[3], const size_t out_pitches[3], uint8_t *dst_mask, size_t mask_pitch,
                         unsigned long long *ticket, const char *who)
{
    uint8_t *dst = out_planes ? out_planes[0] : nullptr;
    if (!c || !valid_fmt(in_fmt) || !valid_fmt(out_fmt) || !planes || !pitches || (dst && !out_pitches) ||
        (dst && out_fmt == SB_PIX_BGR && out_pitches[0] < (size_t)c->out.w * 3) || (dst_mask && mask_pitch < (size_t)c->out.w)) {
        set_error("%s: invalid argument", who);
        return SB_ERR_INVALID;
    }
    if (c->sharded) {
        set_error("%s: the pipelined path is single-GPU; use upload / run / download on a sharded compositor", who);
        return SB_ERR_STATE;
    }
    for (int i = 0; i < c->n; ++i) {
        if (in_fmt == SB_PIX_BGR ? (!planes[3 * i] || pitches[3 * i] < (size_t)c->src_w[i] * 3) : false) {
            set_error("%s: invalid source %d", who, i);
            return SB_ERR_INVALID;
        }
        SB_TRY(yuv_frame_ok(c, who, in_fmt, false, i));
        if (in_fmt != SB_PIX_BGR && !yuv_planes_ok(in_fmt, planes + 3 * i, pitches + 3 * i, c->src_w[i])) {
            set_error("%s: invalid source %d: missing plane or short pitch", who, i);
            return SB_ERR_INVALID;
        }
    }
    if (dst && out_fmt != SB_PIX_BGR) {
        SB_TRY(yuv_frame_ok(c, who, out_fmt, true, 0));
        if (!yuv_planes_ok(out_fmt, out_planes, out_pitches, c->out.w)) {
            set_error("%s: missing panorama plane or short pitch", who);
            return SB_ERR_INVALID;
        }
    }
    SB_TRY(compositor_pipe_init(c));
    const unsigned long long t = c->submitted;
    const int slot = (int)(t % SB_PIPE_DEPTH);
    SB_TRY(yuv_buffers(c, slot, in_fmt, dst ? out_fmt : SB_PIX_BGR));
    const PanoOut &o = slot ? c->outx[slot - 1] : c->out;
    // sources of this slot are free once the previous compute that read them has finished; on a slot's first use
    // that is whatever upload() / run() / sb_compositor_time() queued on the compute stream before this submit
    // (download() is synchronous, so the output buffers need no such guard)
    if (t < SB_PIPE_DEPTH) SB_CUDA(cudaEventRecord(c->e_comp[slot], c->stream));
    SB_CUDA(cudaStreamWaitEvent(c->h2d, c->e_comp[slot], 0));
    for (int i = 0; i < c->n; ++i) {
        if (in_fmt == SB_PIX_BGR)
            SB_CUDA(sb_copy2d(src_of(c, slot, i), (size_t)c->src_w[i] * 3, planes[3 * i], pitches[3 * i], (size_t)c->src_w[i] * 3, c->src_h[i],
                              cudaMemcpyHostToDevice, c->h2d));
        else
            SB_CUDA(yuv_copy(yuv_stage_of(c, slot, i), planes + 3 * i, pitches + 3 * i, in_fmt, c->src_w[i], c->src_h[i],
                             cudaMemcpyHostToDevice, c->h2d));
    }
    // the repack / conversion kernels follow the LAST copy (same stream): a kernel between two copies would leave the PCIe
    // link idle for its launch + run time, eight times per step
    for (int i = 0; i < c->n; ++i) {
        if (in_fmt != SB_PIX_BGR) {
            SB_TRY(yuv_convert_source(c, slot, i, in_fmt, c->h2d));
            continue;
        }
        uint32_t *s4 = src4_of(c, slot, i);
        if (s4) SB_TRY(launch_repack_rgbx(src_of(c, slot, i), s4, (long long)c->src_w[i] * c->src_h[i], c->h2d));
    }
    SB_CUDA(cudaEventRecord(c->e_h2d[slot], c->h2d));
    SB_CUDA(cudaStreamWaitEvent(c->stream, c->e_h2d[slot], 0));
    // the output buffers of this slot are free once their previous download has finished
    if (t >= SB_PIPE_DEPTH) SB_CUDA(cudaStreamWaitEvent(c->stream, c->e_d2h[slot], 0));
    SB_TRY(compositor_enqueue(c, false, slot));
    const bool yuv_out = dst && out_fmt != SB_PIX_BGR;
    if (yuv_out)  // after the step's graph, on the compute stream
        SB_TRY(launch_bgr_to_yuv420(out_fmt, o.rgb, o.rgb_pitch, o.w, o.h, yuv_dense_out(out_fmt, c->yuv_out[slot], o.w, o.h), c->stream));
    SB_CUDA(cudaEventRecord(c->e_comp[slot], c->stream));
    SB_CUDA(cudaStreamWaitEvent(c->d2h, c->e_comp[slot], 0));
    if (yuv_out)
        SB_CUDA(yuv_copy(c->yuv_out[slot], out_planes, out_pitches, out_fmt, o.w, o.h, cudaMemcpyDeviceToHost, c->d2h));
    else if (dst)
        SB_CUDA(sb_copy2d(dst, out_pitches[0], o.rgb, (size_t)o.rgb_pitch, (size_t)o.w * 3, o.h, cudaMemcpyDeviceToHost, c->d2h));
    if (dst_mask)
        SB_CUDA(sb_copy2d(dst_mask, mask_pitch, o.mask, (size_t)o.mask_pitch, o.w, o.h, cudaMemcpyDeviceToHost, c->d2h));
    SB_CUDA(cudaEventRecord(c->e_d2h[slot], c->d2h));
    c->submitted = t + 1;
    if (ticket) *ticket = t;
    return SB_OK;
}

extern "C" {

sb_compositor *sb_compositor_create(const sb_rig *rig)
{
    if (!rig || rig->n_images <= 0 || rig->n_images > SB_MAX_IMAGES || !rig->src_w || !rig->src_h || !rig->K || !rig->R ||
        rig->warp_type < SB_WARP_SPHERICAL || rig->warp_type > SB_WARP_TRANSVERSE_MERCATOR || rig->blend_kind < SB_BLEND_NO ||
        rig->blend_kind > SB_BLEND_MULTIBAND) {
        set_error("sb_compositor_create: invalid rig");
        return nullptr;
    }
    sb_compositor *c = new sb_compositor;
    if (compositor_build(c, rig, 0, 1) != SB_OK) {
        compositor_free(c);
        return nullptr;
    }
    return c;
}

// One panorama over `world` GPUs (one process each): this rank warps and pyramids images
// [rank*n/world, (rank+1)*n/world) and owns one column strip of the panorama (sb_shard.h).
sb_compositor *sb_compositor_create_sharded(const sb_rig *rig, int rank, int world)
{
    if (!rig || rig->n_images <= 0 || rig->n_images > SB_MAX_IMAGES || !rig->src_w || !rig->src_h || !rig->K || !rig->R ||
        rig->warp_type < SB_WARP_SPHERICAL || rig->warp_type > SB_WARP_TRANSVERSE_MERCATOR || world < 1 || rank < 0 || rank >= world) {
        set_error("sb_compositor_create_sharded: invalid argument");
        return nullptr;
    }
    sb_compositor *c = new sb_compositor;
    if (compositor_build(c, rig, rank, world) != SB_OK) {
        compositor_free(c);
        return nullptr;
    }
    return c;
}

int sb_compositor_shard_info(const sb_compositor *c, int *first_image, int *n_local, int strip[2])
{
    if (!c) {
        set_error("sb_compositor_shard_info: null handle");
        return SB_ERR_INVALID;
    }
    if (first_image) *first_image = c->first;
    if (n_local) *n_local = c->count;
    if (strip) {
        strip[0] = 0;
        strip[1] = c->plan.roi.w;
        if (c->sharded) c->shard.strip(c->plan, &strip[0], &strip[1]);  // columns, or rows when sb_compositor_shard_axis() == 1
    }
    return SB_OK;
}

// Transport hooks: run the two halves of a sharded step separately and reach the slab buffers, so that a caller can
// move the slabs itself (tests do, with plain copies; sb_compositor_run uses NCCL).
int sb_compositor_shard_phase(sb_compositor *c, int phase)
{
    if (!c || !c->sharded || phase < 0 || phase > 1) {
        set_error("sb_compositor_shard_phase: invalid argument");
        return SB_ERR_INVALID;
    }
    cudaStream_t s = c->stream;
    auto nomark = [](const std::string &) -> int { return SB_OK; };
    if (phase == 0) {
        SB_TRY(launch_warp(c->jobs.data() + c->first, c->count, s));
        SB_TRY(shard_local(c, s, std::function<int(const std::string &)>(nomark)));
    } else if (c->plan.kind == SB_BLEND_FEATHER) {
        SB_TRY(c->shard.feather_finish(c->plan, c->out, s));
    } else {
        SB_TRY(c->shard.finish(c->plan, c->out, s));
    }
    SB_CUDA(cudaStreamSynchronize(s));
    return SB_OK;
}

int sb_compositor_shard_axis(const sb_compositor *c) { return c && c->sharded ? c->shard.axis : 0; }

int sb_compositor_shard_slab(sb_compositor *c, int peer, int outgoing, void **dev_ptr, size_t *bytes)
{
    if (!c || !c->sharded || peer < 0 || peer >= c->shard.world || peer == c->shard.rank || !dev_ptr || !bytes) {
        set_error("sb_compositor_shard_slab: invalid argument");
        return SB_ERR_INVALID;
    }
    const PeerSlab &p = outgoing ? c->shard.send[peer] : c->shard.recv[peer];
    *dev_ptr = p.buf;
    *bytes = p.bytes;
    return SB_OK;
}

void sb_compositor_destroy(sb_compositor *c) { compositor_free(c); }

int sb_compositor_geometry(const sb_compositor *c, int *rects, int pano_roi[4], int *num_bands)
{
    if (!c) {
        set_error("sb_compositor_geometry: null handle");
        return SB_ERR_INVALID;
    }
    if (rects)
        for (int i = 0; i < c->n; ++i) {
            rects[4 * i] = c->rects[i].x;
            rects[4 * i + 1] = c->rects[i].y;
            rects[4 * i + 2] = c->rects[i].w;
            rects[4 * i + 3] = c->rects[i].h;
        }
    if (pano_roi) {
        pano_roi[0] = c->plan.roi.x;
        pano_roi[1] = c->plan.roi.y;
        pano_roi[2] = c->plan.roi.w;
        pano_roi[3] = c->plan.roi.h;
    }
    if (num_bands) *num_bands = c->plan.kind == SB_BLEND_MULTIBAND ? c->plan.nb : -1;
    return SB_OK;
}

int sb_compositor_model_bytes(const sb_compositor *c, double *total_bytes, double *per_launch, int cap)
{
    if (!c) {
        set_error("sb_compositor_model_bytes: null handle");
        return SB_ERR_INVALID;
    }
    std::vector<double> v;
    v.push_back(c->warp_bytes);
    for (const auto &kv : c->plan.launch_bytes()) v.push_back(kv.second);
    double tot = 0;
    for (double b : v) tot += b;
    if (total_bytes) *total_bytes = tot;
    if (per_launch)
        for (int i = 0; i < cap && i < (int)v.size(); ++i) per_launch[i] = v[i];
    return (int)v.size();
}

int sb_compositor_upload(sb_compositor *c, int i, const uint8_t *src, size_t pitch, int pinned)
{
    const uint8_t *planes[3] = {src, nullptr, nullptr};
    const size_t pitches[3] = {pitch, 0, 0};
    return upload_frame(c, i, SB_PIX_BGR, planes, pitches, pinned, "sb_compositor_upload");
}

int sb_compositor_upload_frame(sb_compositor *c, int i, int fmt, const uint8_t *const planes[3], const size_t pitches[3], int pinned)
{
    return upload_frame(c, i, fmt, planes, pitches, pinned, "sb_compositor_upload_frame");
}

int sb_compositor_set_mask(sb_compositor *c, int i, const uint8_t *mask, size_t pitch)
{
    if (!c || i < 0 || i >= c->n || !mask || pitch < (size_t)c->rects[i].w || !c->rgbm_dev[i]) {
        set_error("sb_compositor_set_mask: invalid argument (or an image of another rank)");
        return SB_ERR_INVALID;
    }
    // the blend mask of image i in warped coordinates (what stitcher.py:223-239 hands to Blender.feed); it replaces
    // the validity mask in the weight byte of the packed warped image from the next run on
    const int w = c->rects[i].w, h = c->rects[i].h;
    if (!c->usermask_dev[i]) SB_TRY(dev_alloc((void **)&c->usermask_dev[i], (size_t)w * h, c->stream));
    SB_CUDA(sb_copy2d(c->usermask_dev[i], w, mask, pitch, w, h, cudaMemcpyHostToDevice, c->stream));
    SB_CUDA(cudaStreamSynchronize(c->stream));
    c->jobs[i].blend_mask = c->usermask_dev[i];
    c->jobs[i].blend_mask_pitch = w;
    c->jobs[i].blend_mask_and = 0;
    c->plan.binary_masks = false;  // a caller's mask may hold gray values
    for (auto &jx : c->jobsx)
        if (!jx.empty()) {
            jx[i].blend_mask = c->usermask_dev[i];
            jx[i].blend_mask_pitch = w;
            jx[i].blend_mask_and = 0;
        }
#ifndef SB_EMU
    for (auto &g : c->graph_exec)  // the jobs are baked into the captured launches: re-capture
        if (g) {
            (void)cudaGraphExecDestroy(g);
            g = nullptr;
        }
#endif
    return SB_OK;
}

int sb_compositor_set_seam_mask(sb_compositor *c, int i, const uint8_t *seam, size_t seam_pitch, int sw, int sh)
{
    if (!c || i < 0 || i >= c->n || !seam || sw <= 0 || sh <= 0 || seam_pitch < (size_t)sw || !c->rgbm_dev[i]) {
        set_error("sb_compositor_set_seam_mask: invalid argument (or an image of another rank)");
        return SB_ERR_INVALID;
    }
    // SeamFinder.resize(seam_mask, warped mask) (seam_finder.py:38-43, stitcher.py:223-225) without the host round
    // trip: the LOW-resolution seam mask is dilated and resized on the device; the AND with the warped validity mask
    // happens in the warp kernel, which computes that mask anyway
    const int w = c->rects[i].w, h = c->rects[i].h;
    if (!c->usermask_dev[i]) SB_TRY(dev_alloc((void **)&c->usermask_dev[i], (size_t)w * h, c->stream));
    SB_TRY(seam_resize_device(seam, seam_pitch, sw, sh, nullptr, 0, c->usermask_dev[i], w, w, h, c->stream));
    c->jobs[i].blend_mask = c->usermask_dev[i];
    c->jobs[i].blend_mask_pitch = w;
    c->jobs[i].blend_mask_and = 1;
    c->plan.binary_masks = false;  // the resized seam mask is bilinear: gray along the seam
    for (auto &jx : c->jobsx)
        if (!jx.empty()) {
            jx[i].blend_mask = c->usermask_dev[i];
            jx[i].blend_mask_pitch = w;
            jx[i].blend_mask_and = 1;
        }
#ifndef SB_EMU
    for (auto &g : c->graph_exec)  // the jobs are baked into the captured launches: re-capture
        if (g) {
            (void)cudaGraphExecDestroy(g);
            g = nullptr;
        }
#endif
    return SB_OK;
}

int sb_compositor_set_gain(sb_compositor *c, int i, const float *gain_map, int gw, int gh, int gc, const double *gain_scalar)
{
    if (!c || i < 0 || i >= c->n || !c->rgbm_dev[i] || (gain_map && gain_scalar) ||
        (gain_map && (gw <= 0 || gh <= 0 || (gc != 1 && gc != 3)))) {
        set_error("sb_compositor_set_gain: invalid argument (or an image of another rank)");
        return SB_ERR_INVALID;
    }
    // ExposureErrorCompensator.apply(i, corner, warped image, mask) (exposure_error_compensator.py:43-45,
    // stitcher.py:219-221) fused into the warp's epilogue: the warped image never exists uncompensated
    SB_CUDA(cudaStreamSynchronize(c->stream));  // the previous run may still read the old gain buffers
    WarpJob fields = c->jobs[i];
    SB_TRY(gain_upload(&fields, &c->gain[i], c->rects[i].w, c->rects[i].h, gain_map, gw, gh, gc, gain_scalar, c->stream));
    auto copy_gain = [&](WarpJob &j) {
        j.gain_mode = fields.gain_mode;
        j.gain_gw = fields.gain_gw;
        j.gain_gc = fields.gain_gc;
        j.gain_map = fields.gain_map;
        j.gain_tx = fields.gain_tx;
        j.gain_ty = fields.gain_ty;
        j.gain_fx = fields.gain_fx;
        j.gain_fy = fields.gain_fy;
        j.gain_lut = fields.gain_lut;
    };
    copy_gain(c->jobs[i]);
    for (auto &jx : c->jobsx)
        if (!jx.empty()) copy_gain(jx[i]);
#ifndef SB_EMU
    for (auto &g : c->graph_exec)  // the jobs are baked into the captured launches: re-capture
        if (g) {
            (void)cudaGraphExecDestroy(g);
            g = nullptr;
        }
#endif
    return SB_OK;
}

int sb_compositor_run(sb_compositor *c)
{
    if (!c) {
        set_error("sb_compositor_run: null handle");
        return SB_ERR_INVALID;
    }
    return compositor_enqueue(c, false);
}

int sb_compositor_sync(sb_compositor *c)
{
    if (!c) return SB_ERR_INVALID;
    SB_CUDA(cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_compositor_download(sb_compositor *c, uint8_t *dst, size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch)
{
    uint8_t *const planes[3] = {dst, nullptr, nullptr};
    const size_t pitches[3] = {dst_pitch, 0, 0};
    return download_frame(c, SB_PIX_BGR, planes, pitches, dst_mask, mask_pitch, "sb_compositor_download");
}

int sb_compositor_download_frame(sb_compositor *c, int fmt, uint8_t *const planes[3], const size_t pitches[3], uint8_t *dst_mask,
                                 size_t mask_pitch)
{
    return download_frame(c, fmt, planes, pitches, dst_mask, mask_pitch, "sb_compositor_download_frame");
}

int sb_compositor_submit(sb_compositor *c, const uint8_t *const *srcs, const size_t *pitches, uint8_t *dst, size_t dst_pitch,
                         uint8_t *dst_mask, size_t mask_pitch, unsigned long long *ticket)
{
    std::vector<const uint8_t *> planes;
    std::vector<size_t> plane_pitches;
    if (c && srcs && pitches) {  // one plane per source
        planes.assign((size_t)3 * c->n, nullptr);
        plane_pitches.assign((size_t)3 * c->n, 0);
        for (int i = 0; i < c->n; ++i) {
            planes[3 * i] = srcs[i];
            plane_pitches[3 * i] = pitches[i];
        }
    }
    uint8_t *const out[3] = {dst, nullptr, nullptr};
    const size_t out_pitches[3] = {dst_pitch, 0, 0};
    return submit_frames(c, SB_PIX_BGR, planes.empty() ? nullptr : planes.data(), plane_pitches.empty() ? nullptr : plane_pitches.data(),
                         SB_PIX_BGR, out, out_pitches, dst_mask, mask_pitch, ticket, "sb_compositor_submit");
}

int sb_compositor_submit_frames(sb_compositor *c, int in_fmt, const uint8_t *const *planes, const size_t *pitches, int out_fmt,
                                uint8_t *const out_planes[3], const size_t out_pitches[3], uint8_t *dst_mask, size_t mask_pitch,
                                unsigned long long *ticket)
{
    return submit_frames(c, in_fmt, planes, pitches, out_fmt, out_planes, out_pitches, dst_mask, mask_pitch, ticket,
                         "sb_compositor_submit_frames");
}

int sb_compositor_wait(sb_compositor *c, unsigned long long ticket)
{
    if (!c || !c->pipe_ready || ticket >= c->submitted || ticket + SB_PIPE_DEPTH < c->submitted) {
        set_error("sb_compositor_wait: ticket %llu is not in flight", ticket);
        return SB_ERR_STATE;
    }
    SB_CUDA(cudaEventSynchronize(c->e_d2h[ticket % SB_PIPE_DEPTH]));
    return SB_OK;
}

int sb_compositor_download_warped(sb_compositor *c, int i, uint8_t *dst, size_t dst_pitch, uint8_t *dst_mask, size_t mask_pitch)
{
    if (!c || i < 0 || i >= c->n || !c->rgbm_dev[i]) {
        set_error("sb_compositor_download_warped: invalid argument (or an image of another rank)");
        return SB_ERR_INVALID;
    }
    const int w = c->rects[i].w, h = c->rects[i].h;
    const size_t wp = (size_t)rgbm_pitch_of(w);
    std::vector<uint32_t> tmp(wp * h);
    SB_CUDA(cudaMemcpyAsync(tmp.data(), c->rgbm_dev[i], tmp.size() * 4, cudaMemcpyDeviceToHost, c->stream));
    SB_CUDA(cudaStreamSynchronize(c->stream));
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            const uint32_t p = tmp[(size_t)y * wp + x];
            if (dst) {
                uint8_t *d = dst + (size_t)y * dst_pitch + (size_t)x * 3;
                d[0] = p & 255;
                d[1] = (p >> 8) & 255;
                d[2] = (p >> 16) & 255;
            }
            if (dst_mask) dst_mask[(size_t)y * mask_pitch + x] = (uint8_t)(p >> 24);
        }
    return SB_OK;
}

// Throughput with several batches in flight: `iters` steps dealt round-robin to n compositors of the same rig (each
// has its own stream and buffers, so the small latency-bound kernels of one step overlap the large kernels of
// another).  One start event; every stream waits for it; the time is up to the LAST stream's end event.
int sb_compositor_time_multi(sb_compositor *const *cs, int n, int iters, float *ms_total)
{
    if (!cs || n < 1 || n > 8 || iters <= 0 || !ms_total) {
        set_error("sb_compositor_time_multi: invalid argument");
        return SB_ERR_INVALID;
    }
    for (int k = 0; k < n; ++k)
        if (!cs[k] || cs[k]->sharded) {
            set_error("sb_compositor_time_multi: null or sharded compositor");
            return SB_ERR_INVALID;
        }
    cudaEvent_t start = nullptr, ends[8] = {};
    SB_CUDA(cudaEventCreate(&start));
    for (int k = 0; k < n; ++k) SB_CUDA(cudaEventCreate(&ends[k]));
    SB_CUDA(cudaEventRecord(start, cs[0]->stream));
    for (int k = 1; k < n; ++k) SB_CUDA(cudaStreamWaitEvent(cs[k]->stream, start, 0));
    int rc = SB_OK;
    for (int it = 0; it < iters && rc == SB_OK; ++it) rc = compositor_enqueue(cs[it % n], false);
    float worst = 0.f;
    for (int k = 0; k < n; ++k) {
        if (cudaEventRecord(ends[k], cs[k]->stream) != cudaSuccess || cudaEventSynchronize(ends[k]) != cudaSuccess) rc = rc == SB_OK ? SB_ERR_CUDA : rc;
        float t = 0.f;
        if (rc == SB_OK && cudaEventElapsedTime(&t, start, ends[k]) == cudaSuccess) worst = t > worst ? t : worst;
    }
    (void)cudaEventDestroy(start);
    for (int k = 0; k < n; ++k) (void)cudaEventDestroy(ends[k]);
    if (rc != SB_OK && rc == SB_ERR_CUDA) set_error("sb_compositor_time_multi: CUDA failure while timing");
    *ms_total = worst;
    return rc;
}

int sb_compositor_time(sb_compositor *c, int iters, int flush_l2, float *ms_total)
{
    if (!c || iters <= 0 || !ms_total) {
        set_error("sb_compositor_time: invalid argument");
        return SB_ERR_INVALID;
    }
    cudaStream_t s = c->stream;
    if (flush_l2 && !c->flush_buf) {
        c->flush_bytes = (size_t)256 << 20;  // 2x the 126 MB L2
        SB_TRY(dev_alloc(&c->flush_buf, c->flush_bytes, s));
    }
    float total = 0.f;
    // pass 1: whole steps exactly as sb_compositor_run issues them (one graph launch), one event pair per step
    // (the host enqueues ahead of the device: no host synchronisation between steps; with flush_l2 the flush
    // kernel runs between a step's end event and the next step's start event)
    while ((int)c->tev.size() < 2 * iters) {
        cudaEvent_t e;
        SB_CUDA(cudaEventCreate(&e));
        c->tev.push_back(e);
    }
    for (int it = 0; it < iters; ++it) {
        if (flush_l2) SB_TRY(launch_flush_l2(c->flush_buf, c->flush_bytes, s));
        if (flush_l2 || it == 0) SB_CUDA(cudaEventRecord(c->tev[2 * it], s));
        SB_TRY(compositor_enqueue(c, false));
        if (flush_l2 || it == iters - 1) SB_CUDA(cudaEventRecord(c->tev[2 * it + 1], s));
    }
    SB_CUDA(cudaStreamSynchronize(s));
    if (flush_l2) {
        for (int it = 0; it < iters; ++it) {
            float t = 0;
            SB_CUDA(cudaEventElapsedTime(&t, c->tev[2 * it], c->tev[2 * it + 1]));
            total += t;
        }
    } else {
        SB_CUDA(cudaEventElapsedTime(&total, c->tev[0], c->tev[2 * (iters - 1) + 1]));
    }
    *ms_total = total;
    // pass 2: per-kernel breakdown (individual launches with an event after each), a few iterations
    iters = iters < 5 ? iters : 5;
    total = 0.f;
    c->launch_ms.clear();
    for (int it = 0; it < iters; ++it) {
        if (flush_l2) SB_TRY(launch_flush_l2(c->flush_buf, c->flush_bytes, s));
        SB_TRY(compositor_enqueue(c, true));
        const size_t nl = c->launch_names.size();
        SB_CUDA(cudaEventSynchronize(c->ev[nl]));
        if (c->launch_ms.size() != nl) c->launch_ms.assign(nl, 0.f);
        for (size_t k = 0; k < nl; ++k) {
            float t = 0;
            SB_CUDA(cudaEventElapsedTime(&t, c->ev[k], c->ev[k + 1]));
            c->launch_ms[k] += t;
        }
        float t = 0;
        SB_CUDA(cudaEventElapsedTime(&t, c->ev[0], c->ev[nl]));
        total += t;
    }
    for (float &v : c->launch_ms) v /= (float)iters;
    return SB_OK;
}

int sb_compositor_stage_times(sb_compositor *c, const char **names, float *ms, int cap)
{
    if (!c) return 0;
    int k = (int)std::min<size_t>((size_t)cap, c->launch_ms.size());
    for (int i = 0; i < k; ++i) {
        if (names) names[i] = c->launch_names[i].c_str();
        if (ms) ms[i] = c->launch_ms[i];
    }
    return k;
}

}  // extern "C"
