// sb_warp.cu -- fused backward-map warp: image (fixed-point bilinear, BORDER_REFLECT) and validity mask
// (nearest, BORDER_CONSTANT) in one pass, no float maps in memory.
//
// Replaces, per output pixel, what cv.PyRotationWarper.warp does in three passes
// (stitching/warper.py:43-52 image, :58-68 mask): buildMaps -> remap(INTER_LINEAR, BORDER_REFLECT) and
// buildMaps -> remap(INTER_NEAREST, BORDER_CONSTANT).
//
// Arithmetic contract (bit-exact with the reference's CPU path):
//   projection  x_ = rowA[v]*colX[u], y_ = rowY[v], z_ = rowA[v]*colZ[u]      (host libm tables)
//               (x,y,z) = k_rinv * (x_,y_,z_)  plain fp32, (a+b)+c, every op rounded, no FMA
//               spherical/cylindrical: z > 0 ? (x/z, y/z) : (-1,-1);  plane: always divide
//   bilinear    sx = cvRound(x*32) (half-even, INT_MIN when unrepresentable), ix = sat16(sx>>5),
//               fx = sx&31; 4 taps with 15-bit weights (32-fy)(32-fx)*32 ..., (sum + 2^14) >> 15
//   mask        255 iff 0 <= sat16(cvRound(x)) < W and 0 <= sat16(cvRound(y)) < H
//
// The job descriptors travel BY VALUE in the kernel parameter block (constant bank, up to SB_WARP_BATCH images
// per launch): the profile of the first version showed 20 of 31 loads per pixel re-reading them from global memory.
#include "sb_device.cuh"
#include "sb_launch.h"

namespace sb {

namespace {

constexpr int WARP_BX = 32, WARP_BY = 8;

struct WarpBatch {
    WarpJob j[SB_WARP_BATCH];
};

__device__ __forceinline__ void project(const WarpJob &j, int u, int v, float &x, float &y)
{
    if (j.xmap) {  // a projection that is not separable: the host built the maps (sb_geometry.cpp projector_maps)
        const size_t o = (size_t)v * (size_t)j.dw + (size_t)u;
        x = __ldg(j.xmap + o);
        y = __ldg(j.ymap + o);
        return;
    }
    const float cx = __ldg(j.colX + u), cz = __ldg(j.colZ + u);
    const float ra = __ldg(j.rowA + v), ry = __ldg(j.rowY + v);
    const float x_ = fmul(ra, cx), y_ = ry, z_ = fmul(ra, cz);
    x = fadd(fadd(fmul(j.k[0], x_), fmul(j.k[1], y_)), fmul(j.k[2], z_));
    y = fadd(fadd(fmul(j.k[3], x_), fmul(j.k[4], y_)), fmul(j.k[5], z_));
    const float z = fadd(fadd(fmul(j.k[6], x_), fmul(j.k[7], y_)), fmul(j.k[8], z_));
    if (j.always_divide || z > 0.f) {
        x = fdiv(x, z);
        y = fdiv(y, z);
    } else {
        x = -1.f;
        y = -1.f;
    }
}

// ExposureErrorCompensator.apply on one warped pixel (stitching/exposure_error_compensator.py:43-45 -> cv.detail
// compensators, stitcher.py:219-221), see oracle/stitch_oracle.c for the pinned arithmetic:
//   mode 1 (gain_blocks / channel_blocks): the float32 gain map resized to the warped size -- horizontal pass first, each
//     pass a + (b - a) t as ONE fused multiply-add -- then saturate(cvRound(float(value) * gain)) with a float32 product;
//   mode 2 (gain / channel): saturate(cvRound(double(value) * gain)), tabulated per channel on the host.
__device__ __forceinline__ void apply_gain(const WarpJob &j, int u, int v, unsigned &r, unsigned &g, unsigned &b)
{
    if (j.gain_mode == 2) {
        r = j.gain_lut[r];
        g = j.gain_lut[256 + g];
        b = j.gain_lut[512 + b];
        return;
    }
    const int x0 = j.gain_tx[u], x1 = j.gain_tx[j.dw + u], y0 = j.gain_ty[v], y1 = j.gain_ty[j.dh + v];
    const float fx = j.gain_fx[u], fy = j.gain_fy[v];
    const int gc = j.gain_gc;
    const float *r0 = j.gain_map + (long long)y0 * j.gain_gw * gc, *r1 = j.gain_map + (long long)y1 * j.gain_gw * gc;
    unsigned c[3] = {r, g, b};
    float gain = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (k == 0 || gc == 3) {
            const float a0 = r0[x0 * gc + k], b0 = r0[x1 * gc + k], a1 = r1[x0 * gc + k], b1 = r1[x1 * gc + k];
            const float h0 = fmaf(fadd(b0, -a0), fx, a0), h1 = fmaf(fadd(b1, -a1), fx, a1);
            gain = fmaf(fadd(h1, -h0), fy, h0);
        }
        const int q = __float2int_rn(fmul((float)c[k], gain));  // |value * gain| is far below 2^31
        c[k] = (unsigned)sat_u8(q);
    }
    r = c[0];
    g = c[1];
    b = c[2];
}

__device__ __forceinline__ void store_pixel(const WarpJob &j, int u, int v, unsigned r, unsigned g, unsigned b, unsigned m)
{
    if (j.gain_mode) apply_gain(j, u, v, r, g, b);
    if (j.dst_rgb) {
        uint8_t *d = j.dst_rgb + (long long)v * j.dst_pitch + 3 * u;
        d[0] = (uint8_t)r;
        d[1] = (uint8_t)g;
        d[2] = (uint8_t)b;
    }
    if (j.dst_rgbm) {
        if (j.blend_mask) {
            const unsigned bm = j.blend_mask[(long long)v * j.blend_mask_pitch + u];
            m = j.blend_mask_and ? (bm & m) : bm;
        }
        j.dst_rgbm[(unsigned)v * (unsigned)j.rgbm_pitch + (unsigned)u] = r | (g << 8) | (b << 16) | (m << 24);
    }
}

// simple variant: one thread per output pixel, byte gathers
__global__ void __launch_bounds__(WARP_BX *WARP_BY) k_warp_gather(const __grid_constant__ WarpBatch B)
{
    const WarpJob &j = B.j[blockIdx.z];
    const int u = blockIdx.x * WARP_BX + threadIdx.x;
    const int v = blockIdx.y * WARP_BY + threadIdx.y;
    if (u >= j.dw || v >= j.dh) return;

    float x, y;
    project(j, u, v, x, y);

    // validity mask: nearest neighbour into an all-255 source, constant-0 border
    const int nx = sat_s16(cvt_rn_x86(x)), ny = sat_s16(cvt_rn_x86(y));
    const unsigned m = ((unsigned)nx < (unsigned)j.sw && (unsigned)ny < (unsigned)j.sh) ? 255u : 0u;
    if (j.dst_mask) j.dst_mask[(long long)v * j.mask_pitch + u] = (uint8_t)m;
    if (!j.dst_rgb && !j.dst_rgbm) return;

    const int sx = cvt_rn_x86(fmul(x, 32.f)), sy = cvt_rn_x86(fmul(y, 32.f));
    const int ix = sat_s16(sx >> 5), iy = sat_s16(sy >> 5);
    const int fx = sx & 31, fy = sy & 31;
    const int x0 = reflect(ix, j.sw), x1 = reflect(ix + 1, j.sw);
    const int y0 = reflect(iy, j.sh), y1 = reflect(iy + 1, j.sh);
    const int w00 = (32 - fy) * (32 - fx) * 32, w01 = (32 - fy) * fx * 32;
    const int w10 = fy * (32 - fx) * 32, w11 = fy * fx * 32;
    const uint8_t *r0 = j.src + (long long)y0 * j.spitch, *r1 = j.src + (long long)y1 * j.spitch;
    unsigned out[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        int acc = __ldg(r0 + x0 * 3 + c) * w00 + __ldg(r0 + x1 * 3 + c) * w01 + __ldg(r1 + x0 * 3 + c) * w10 +
                  __ldg(r1 + x1 * 3 + c) * w11;
        out[c] = (unsigned)sat_u8((acc + (1 << 14)) >> 15);
    }
    store_pixel(j, u, v, out[0], out[1], out[2], m);
}

// Fast variant: the two horizontally adjacent source pixels of a bilinear footprint are 6 contiguous bytes;
// fetch them with one (or two) aligned 8-byte loads instead of six byte loads.  Callers allocate the source
// with SB_SRC_PAD spare bytes so that the second aligned word may straddle the end of the image.
__device__ __forceinline__ void fetch_pair(const uint8_t *__restrict__ src, unsigned row_off, int x0, int x1, unsigned &p0, unsigned &p1)
{
    if (x1 == x0 + 1) {
        const unsigned long long addr = (unsigned long long)src + row_off + 3u * (unsigned)x0;
        const unsigned o = (unsigned)addr & 7u;
        const uint2 *q = reinterpret_cast<const uint2 *>(addr - o);
        const uint2 lo = __ldg(q);
        // bytes o .. o+5 of the 16-byte window (lo, hi): shift the 32-bit words with funnel shifts
        const unsigned sh = 8u * (o & 3u);
        unsigned w0 = lo.x, w1 = lo.y, w2 = 0u;
        if (o > 2) {
            const uint2 hi = __ldg(q + 1);
            w2 = hi.x;
            if (o >= 4) {
                w0 = lo.y;
                w1 = hi.x;
                w2 = hi.y;
            }
        }
        const unsigned a = __funnelshift_r(w0, w1, sh), b = __funnelshift_r(w1, w2, sh);  // bytes 0-3 and 4-7 from the start
        p0 = a & 0xffffffu;
        p1 = __funnelshift_r(a, b, 24) & 0xffffffu;
    } else {  // the footprint straddles a reflected border
        const uint8_t *a = src + row_off + 3 * x0, *b = src + row_off + 3 * x1;
        p0 = (unsigned)__ldg(a) | ((unsigned)__ldg(a + 1) << 8) | ((unsigned)__ldg(a + 2) << 16);
        p1 = (unsigned)__ldg(b) | ((unsigned)__ldg(b + 1) << 8) | ((unsigned)__ldg(b + 2) << 16);
    }
}

// Generic fast variant (sb_warp with separate image / mask outputs, sources wider than int16): one pixel per thread.
__global__ void __launch_bounds__(WARP_BX *WARP_BY) k_warp_wide(const __grid_constant__ WarpBatch B)
{
    const WarpJob &j = B.j[blockIdx.z];
    const int u = blockIdx.x * WARP_BX + threadIdx.x;
    const int v = blockIdx.y * WARP_BY + threadIdx.y;
    if (u >= j.dw || v >= j.dh) return;
    const int sw = j.sw, sh = j.sh;

    float x, y;
    project(j, u, v, x, y);
    const int nx = sat_s16(cvt_rn_x86(x)), ny = sat_s16(cvt_rn_x86(y));
    const unsigned m = ((unsigned)nx < (unsigned)sw && (unsigned)ny < (unsigned)sh) ? 255u : 0u;
    if (j.dst_mask) j.dst_mask[(long long)v * j.mask_pitch + u] = (uint8_t)m;
    if (!j.dst_rgb && !j.dst_rgbm) return;

    const int sx = cvt_rn_x86(fmul(x, 32.f)), sy = cvt_rn_x86(fmul(y, 32.f));
    const int fx = sx & 31, fy = sy & 31;
    const int ix = sat_s16(sx >> 5), iy = sat_s16(sy >> 5);
    unsigned a0, a1, b0, b1;
    const unsigned pitch = (unsigned)j.spitch;  // coordinates are int16-saturated: offsets stay below 2^32
    if ((unsigned)ix < (unsigned)(sw - 1) && (unsigned)iy < (unsigned)(sh - 1)) {
        // the 2x2 footprint lies inside the image: no border rule applies, the pairs are adjacent
        const unsigned off = (unsigned)iy * pitch;
        fetch_pair(j.src, off, ix, ix + 1, a0, a1);
        fetch_pair(j.src, off + pitch, ix, ix + 1, b0, b1);
    } else {
        const int x0 = reflect(ix, sw), x1 = reflect(ix + 1, sw);
        const int y0 = reflect(iy, sh), y1 = reflect(iy + 1, sh);
        fetch_pair(j.src, (unsigned)y0 * pitch, x0, x1, a0, a1);
        fetch_pair(j.src, (unsigned)y1 * pitch, x0, x1, b0, b1);
    }
    // (sum_k w_k p_k + 2^14) >> 15 with w = 32 (32-fy|fy)(32-fx|fx), evaluated as two exact lerps:
    //   h = (32-fx) a + fx b  (<= 8160),  s = (32-fy) h0 + fy h1  (<= 261120),  out = (s + 512) >> 10
    // red and blue share a register as two 16-bit lanes through the horizontal lerp
    const unsigned M = 0x00ff00ffu;
    const unsigned gx = (unsigned)fx, hx = 32u - gx;
    const unsigned h0rb = (a0 & M) * hx + (a1 & M) * gx, h1rb = (b0 & M) * hx + (b1 & M) * gx;
    const unsigned h0g = ((a0 >> 8) & 255u) * hx + ((a1 >> 8) & 255u) * gx, h1g = ((b0 >> 8) & 255u) * hx + ((b1 >> 8) & 255u) * gx;
    const unsigned gy = (unsigned)fy, hy = 32u - gy;
    const unsigned r = ((h0rb & 0xffffu) * hy + (h1rb & 0xffffu) * gy + 512u) >> 10;
    const unsigned b = ((h0rb >> 16) * hy + (h1rb >> 16) * gy + 512u) >> 10;
    const unsigned g = (h0g * hy + h1g * gy + 512u) >> 10;
    store_pixel(j, u, v, r, g, b, m);
}

// ---- the compositor's kernel: packed RGBM output only, source sides <= 32767 (int16 saturation can then neither
// move a coordinate across the inside test nor touch a footprint that lies inside the image), TWO horizontally
// adjacent output pixels per thread (descriptor reads, row tables and the k*y_ products are shared; 8-byte table
// loads and stores).

// six bytes starting at src + off as two words (bytes 0-3, bytes 4-7): three aligned 4-byte loads and two funnel
// shifts, no selects.  Reads at most 11 bytes past the aligned start (SB_SRC_PAD covers the end of the image).
__device__ __forceinline__ void fetch6(const uint8_t *__restrict__ src, unsigned off, unsigned &lo, unsigned &hi)
{
    const unsigned long long addr = (unsigned long long)src + off;
    const unsigned *q = reinterpret_cast<const unsigned *>(addr & ~3ull);
    const unsigned w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
    const unsigned sh = ((unsigned)addr & 3u) * 8u;
    lo = __funnelshift_r(w0, w1, sh);
    hi = __funnelshift_r(w1, w2, sh);
}

// the bilinear sum of a 2x2 footprint given as rows of six bytes (l = bytes 0-3, h = bytes 4-7): two exact lerps as
// above; PRMT places red|blue (per row) and green (both rows) into 16-bit lanes, the vertical lerp is a two-way
// 16x8-bit dot product (IDP.2A) per channel.  Returns r | g<<8 | b<<16.
template <bool DP2A>
__device__ __forceinline__ unsigned lerp6(unsigned l0, unsigned h0, unsigned l1, unsigned h1, unsigned fx, unsigned fy)
{
    h0 &= 0xffffu;
    h1 &= 0xffffu;
    const unsigned hx = 32u - fx, hy = 32u - fy;
    const unsigned rb0 = __byte_perm(l0, h0, 0x7270) * hx + __byte_perm(l0, h0, 0x7573) * fx;  // [r | b<<16] of row 0
    const unsigned rb1 = __byte_perm(l1, h1, 0x7270) * hx + __byte_perm(l1, h1, 0x7573) * fx;
    const unsigned g01 = (__byte_perm(l0, l1, 0x5511) & 0x00ff00ffu) * hx + __byte_perm(h0, h1, 0x6420) * fx;  // [row0 | row1<<16]
    unsigned r, g, b;
    if (DP2A) {
        const unsigned wy = hy | (fy << 8);
        r = __dp2a_lo(__byte_perm(rb0, rb1, 0x5410), wy, 512u);
        b = __dp2a_lo(__byte_perm(rb0, rb1, 0x7632), wy, 512u);
        g = __dp2a_lo(g01, wy, 512u);
    } else {
        r = (rb0 & 0xffffu) * hy + (rb1 & 0xffffu) * fy + 512u;
        b = (rb0 >> 16) * hy + (rb1 >> 16) * fy + 512u;
        g = (g01 & 0xffffu) * hy + (g01 >> 16) * fy + 512u;
    }
    return (r >> 10) | ((g >> 2) & 0xff00u) | ((b << 6) & 0xff0000u);
}

// the general rule for one pixel, from the projected numerators: exact division, x86 rounding, int16 saturation,
// BORDER_REFLECT, validity from the nearest-neighbour test.  Called for the few pixels the streamlined path of
// k_warp_rgbm does not cover (footprint on the border or outside, z <= 0, values outside the shortcut's ranges).
__device__ SB_NOINLINE unsigned sample_general(const uint8_t *__restrict__ src, const uint32_t *__restrict__ src4, int sw, int sh, unsigned pitch,
                                                float x, float y, float z, int always_divide)
{
    if (always_divide || z > 0.f) {
        x = fdiv(x, z);
        y = fdiv(y, z);
    } else {
        x = -1.f;
        y = -1.f;
    }
    const unsigned m = ((unsigned)cvt_rn_x86(x) < (unsigned)sw && (unsigned)cvt_rn_x86(y) < (unsigned)sh) ? 255u : 0u;
    const int sx = cvt_rn_x86(fmul(x, 32.f)), sy = cvt_rn_x86(fmul(y, 32.f));
    const int ix = sat_s16(sx >> 5), iy = sat_s16(sy >> 5);
    const int x0 = reflect(ix, sw), x1 = reflect(ix + 1, sw);
    const int y0 = reflect(iy, sh), y1 = reflect(iy + 1, sh);
    unsigned a0, a1, b0, b1;
    if (src4) {  // one word per pixel
        const unsigned r0 = (unsigned)y0 * (unsigned)sw, r1 = (unsigned)y1 * (unsigned)sw;
        a0 = __ldg(src4 + r0 + x0);
        a1 = __ldg(src4 + r0 + x1);
        b0 = __ldg(src4 + r1 + x0);
        b1 = __ldg(src4 + r1 + x1);
    } else {
        fetch_pair(src, (unsigned)y0 * pitch, x0, x1, a0, a1);
        fetch_pair(src, (unsigned)y1 * pitch, x0, x1, b0, b1);
    }
    // as six-byte rows: left pixel in bytes 0-2, right pixel in bytes 3-5
    return lerp6<false>(a0 | (a1 << 24), a1 >> 8, b0 | (b1 << 24), b1 >> 8, (unsigned)sx & 31u, (unsigned)sy & 31u) | (m << 24);
}

// the same bilinear sum from four pixel words r | g<<8 | b<<16 (byte 3 zero: it doubles as the zero byte of the PRMTs)
__device__ __forceinline__ unsigned lerp4(unsigned p00, unsigned p01, unsigned p10, unsigned p11, unsigned fx, unsigned fy)
{
    const unsigned M = 0x00ff00ffu, hx = 32u - fx, hy = 32u - fy;
    const unsigned rb0 = (p00 & M) * hx + (p01 & M) * fx;  // [r | b<<16] of row 0
    const unsigned rb1 = (p10 & M) * hx + (p11 & M) * fx;
    const unsigned g01 = __byte_perm(p00, p10, 0x7531) * hx + __byte_perm(p01, p11, 0x7531) * fx;  // green [row0 | row1<<16]
    const unsigned wy = hy | (fy << 8);
    const unsigned r = __dp2a_lo(__byte_perm(rb0, rb1, 0x5410), wy, 512u);
    const unsigned b = __dp2a_lo(__byte_perm(rb0, rb1, 0x7632), wy, 512u);
    const unsigned g = __dp2a_lo(g01, wy, 512u);
    return (r >> 10) | ((g >> 2) & 0xff00u) | ((b << 6) & 0xff0000u);
}

// SRC4: the sources are one word per pixel (WarpJob::src4): four aligned loads at two addresses per footprint instead of six
// loads, two funnel shifts and the byte-address arithmetic of the packed 3-byte layout
template <bool HAS_BM, bool DP2A, bool SRC4>
__global__ void __launch_bounds__(WARP_BX *WARP_BY, 8) k_warp_rgbm(const __grid_constant__ WarpBatch B)
{
    grid_dependency_sync();
    const WarpJob &j = B.j[blockIdx.z];
    const int u = 2 * (blockIdx.x * WARP_BX + threadIdx.x);
    const int v = blockIdx.y * WARP_BY + threadIdx.y;
    if (u >= j.dw || v >= j.dh) return;
    // column tables are padded to an even length and 8-byte aligned (warp_table_floats)
    const float2 cx = __ldg(reinterpret_cast<const float2 *>(j.colX + u)), cz = __ldg(reinterpret_cast<const float2 *>(j.colZ + u));
    const float ra = __ldg(j.rowA + v), ry = __ldg(j.rowY + v);
    const float ty0 = fmul(j.k[1], ry), ty1 = fmul(j.k[4], ry), ty2 = fmul(j.k[7], ry);
    const unsigned pitch = (unsigned)j.spitch;
    float xn[2], yn[2], zn[2], x32[2], y32[2];
    bool fast = true;
#pragma unroll
    for (int p = 0; p < 2; ++p) {
        const float x_ = fmul(ra, p ? cx.y : cx.x), z_ = fmul(ra, p ? cz.y : cz.x);
        xn[p] = fadd(fadd(fmul(j.k[0], x_), ty0), fmul(j.k[2], z_));
        yn[p] = fadd(fadd(fmul(j.k[3], x_), ty1), fmul(j.k[5], z_));
        zn[p] = fadd(fadd(fmul(j.k[6], x_), ty2), fmul(j.k[8], z_));
        const float rr = rcp_refined(zn[p]);
        x32[p] = fmul(fdiv_by(xn[p], zn[p], rr), 32.f);
        y32[p] = fmul(fdiv_by(yn[p], zn[p], rr), 32.f);
        // The streamlined path: z in the shortcut division's range (which implies z > 0) and the 2x2 footprint inside
        // the image, i.e. 0 <= cvRound(32x) >> 5 <= sw-2, decided on the floats: cvRound is half-even and the upper
        // threshold 32(sw-1)-0.5 is exact and rounds up to the even 32(sw-1).  The lower threshold is 2^-30 rather
        // than -0.5, which keeps zero and tiny quotients (outside the shortcut's range) out; the sliver in between,
        // 1/32 of the first source column, takes the general path.  NaN fails every test.  In this region x lies in
        // (0, sw-1-1/64), so the nearest-neighbour validity test holds as well: the mask byte is 255.
        fast = fast && zn[p] >= 0x1p-60f && zn[p] <= 0x1p60f && x32[p] >= 0x1p-30f && x32[p] < j.xin_hi && y32[p] >= 0x1p-30f &&
               y32[p] < j.yin_hi;
    }
    unsigned out[2];
    if (fast) {
        unsigned l0[2], h0[2], l1[2], h1[2], sx[2], sy[2];
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            sx[p] = (unsigned)__float2int_rn(x32[p]);
            sy[p] = (unsigned)__float2int_rn(y32[p]);
            if (SRC4) {
                const uint32_t *q = j.src4 + ((sy[p] >> 5) * (unsigned)j.sw + (sx[p] >> 5));
                l0[p] = __ldg(q);
                h0[p] = __ldg(q + 1);
                l1[p] = __ldg(q + j.sw);
                h1[p] = __ldg(q + j.sw + 1);
            } else {
                const unsigned off = (sy[p] >> 5) * pitch + 3u * (sx[p] >> 5);
                fetch6(j.src, off, l0[p], h0[p]);
                fetch6(j.src, off + pitch, l1[p], h1[p]);
            }
        }
#pragma unroll
        for (int p = 0; p < 2; ++p)
            out[p] = (SRC4 ? lerp4(l0[p], h0[p], l1[p], h1[p], sx[p] & 31u, sy[p] & 31u)
                           : lerp6<DP2A>(l0[p], h0[p], l1[p], h1[p], sx[p] & 31u, sy[p] & 31u)) | 0xff000000u;
    } else {
#pragma unroll
        for (int p = 0; p < 2; ++p)
            out[p] = sample_general(j.src, SRC4 ? j.src4 : nullptr, j.sw, j.sh, pitch, xn[p], yn[p], zn[p], j.always_divide);
    }
    if (HAS_BM) {  // the batch has per-pixel extras: exposure gains and / or blend masks (each optional per image)
        if (j.gain_mode) {
#pragma unroll
            for (int p = 0; p < 2; ++p)
                if (p == 0 || u + 1 < j.dw) {
                    unsigned r = out[p] & 255u, g = (out[p] >> 8) & 255u, b = (out[p] >> 16) & 255u;
                    apply_gain(j, u + p, v, r, g, b);
                    out[p] = (out[p] & 0xff000000u) | r | (g << 8) | (b << 16);
                }
        }
        if (j.blend_mask) {
            const uint8_t *bm = j.blend_mask + (unsigned)v * (unsigned)j.blend_mask_pitch + (unsigned)u;
            // a user blend mask replaces the validity byte; a seam mask (sb_compositor_set_seam_mask) is ANDed with it
#pragma unroll
            for (int p = 0; p < 2; ++p)
                if (p == 0 || u + 1 < j.dw) {
                    const unsigned b = (unsigned)bm[p] << 24;
                    out[p] = j.blend_mask_and ? (out[p] & (b | 0x00ffffffu)) : ((out[p] & 0x00ffffffu) | b);
                }
        }
    }
    uint32_t *d = j.dst_rgbm + (unsigned)v * (unsigned)j.rgbm_pitch + (unsigned)u;  // pitch is a multiple of 64: 8-byte aligned
    if (u + 1 < j.dw)
        *reinterpret_cast<uint2 *>(d) = make_uint2(out[0], out[1]);
    else
        d[0] = out[0];
}

// u8x3 -> one word per pixel, four pixels per thread (12 contiguous bytes in, one 16-byte store out)
__global__ void __launch_bounds__(256) k_repack_rgbx(const uint8_t *__restrict__ rgb, uint32_t *__restrict__ dst, long long pixels)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = 4 * t;
    if (p >= pixels) return;
    if (p + 4 <= pixels) {
        const unsigned *q = reinterpret_cast<const unsigned *>(rgb) + 3 * t;  // the buffers come from the allocator: 256-byte aligned
        const unsigned w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
        uint4 o;
        o.x = w0 & 0x00ffffffu;
        o.y = __funnelshift_r(w0, w1, 24) & 0x00ffffffu;
        o.z = __funnelshift_r(w1, w2, 16) & 0x00ffffffu;
        o.w = w2 >> 8;
        *reinterpret_cast<uint4 *>(dst + p) = o;
    } else {
        for (long long k = p; k < pixels; ++k)
            dst[k] = (unsigned)rgb[3 * k] | ((unsigned)rgb[3 * k + 1] << 8) | ((unsigned)rgb[3 * k + 2] << 16);
    }
}

__global__ void k_pack_rgbm(const uint8_t *__restrict__ rgb, long long rgb_pitch, const uint8_t *__restrict__ mask,
                            long long mask_pitch, uint32_t *__restrict__ dst, long long dst_pitch, int w, int h)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const uint8_t *p = rgb + (long long)y * rgb_pitch + (long long)x * 3;
    const unsigned m = mask[(long long)y * mask_pitch + x];
    dst[(long long)y * dst_pitch + x] = (unsigned)p[0] | ((unsigned)p[1] << 8) | ((unsigned)p[2] << 16) | (m << 24);
}

}  // namespace

int launch_repack_rgbx(const uint8_t *rgb, uint32_t *dst, long long pixels, cudaStream_t s)
{
    if (pixels <= 0) return SB_OK;
    const long long threads = (pixels + 3) / 4;
    launch(k_repack_rgbx, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, s, rgb, dst, pixels);
    return launch_check("k_repack_rgbx");
}

// which fast warp kernel a batch of jobs qualifies for (launch_warp)
static void classify_batch(const WarpJob *j, int cnt, bool &rgbm_only, bool &has_bm, bool &src4)
{
    rgbm_only = true, has_bm = false, src4 = true;
    for (int i = 0; i < cnt; ++i) {
        src4 = src4 && j[i].src4 != nullptr;
        rgbm_only = rgbm_only && !j[i].xmap && j[i].dst_rgbm && !j[i].dst_rgb && !j[i].dst_mask && j[i].sw <= 32767 && j[i].sh <= 32767 &&
                    j[i].sw >= 2 && j[i].sh >= 2 && j[i].rgbm_pitch % 2 == 0;
        has_bm = has_bm || j[i].blend_mask || j[i].gain_mode;  // per-pixel extras anywhere in the batch
    }
}

bool warp_reads_src4_only(const WarpJob *jobs, int n_jobs, int i)
{
    if (use_simple_kernels()) return false;
    const int first = i - i % SB_WARP_BATCH;
    const int cnt = n_jobs - first < SB_WARP_BATCH ? n_jobs - first : SB_WARP_BATCH;
    bool rgbm_only, has_bm, src4;
    classify_batch(jobs + first, cnt, rgbm_only, has_bm, src4);
    return rgbm_only && src4;
}

int launch_warp(const WarpJob *jobs_host, int n_jobs, cudaStream_t s)
{
    for (int first = 0; first < n_jobs; first += SB_WARP_BATCH) {
        const int cnt = n_jobs - first < SB_WARP_BATCH ? n_jobs - first : SB_WARP_BATCH;
        WarpBatch B;
        int max_w = 0, max_h = 0;
        for (int i = 0; i < cnt; ++i) {
            B.j[i] = jobs_host[first + i];
            max_w = max_w > B.j[i].dw ? max_w : B.j[i].dw;
            max_h = max_h > B.j[i].dh ? max_h : B.j[i].dh;
        }
        for (int i = cnt; i < SB_WARP_BATCH; ++i) B.j[i] = B.j[0];
        if (max_w <= 0 || max_h <= 0) continue;
        dim3 block(WARP_BX, WARP_BY), grid(div_up(max_w, WARP_BX), div_up(max_h, WARP_BY), cnt);
        if (!use_simple_kernels()) {
            bool rgbm_only, has_bm, src4;
            classify_batch(B.j, cnt, rgbm_only, has_bm, src4);
            if (rgbm_only) {
                dim3 grid2(div_up(max_w, 2 * WARP_BX), div_up(max_h, WARP_BY), cnt);
                if (has_bm && src4)
                    launch_pdl(k_warp_rgbm<true, true, true>, grid2, block, 0, s, B);
                else if (has_bm)
                    launch_pdl(k_warp_rgbm<true, true, false>, grid2, block, 0, s, B);
                else if (src4)
                    launch_pdl(k_warp_rgbm<false, true, true>, grid2, block, 0, s, B);
                else
                    launch_pdl(k_warp_rgbm<false, true, false>, grid2, block, 0, s, B);
            } else {
                launch(k_warp_wide, grid, block, 0, s, B);
            }
            SB_TRY(launch_check("k_warp_wide"));
            continue;
        }
        launch(k_warp_gather, grid, block, 0, s, B);
        SB_TRY(launch_check("k_warp_gather"));
    }
    return SB_OK;
}

// ExposureErrorCompensator.apply on an image in device memory (the host-buffer entry sb_gain_apply): `g` carries the gain
// fields of a WarpJob with dw x dh = the image size
__global__ void k_gain_apply(uint8_t *__restrict__ img, long long pitch, const __grid_constant__ WarpJob g)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= g.dw || y >= g.dh) return;
    uint8_t *p = img + y * pitch + 3 * (long long)x;
    unsigned r = p[0], gg = p[1], b = p[2];
    apply_gain(g, x, y, r, gg, b);
    p[0] = (uint8_t)r;
    p[1] = (uint8_t)gg;
    p[2] = (uint8_t)b;
}

int launch_gain_apply(uint8_t *img, long long pitch, int w, int h, const WarpJob &gain_fields, cudaStream_t s)
{
    WarpJob g = gain_fields;
    g.dw = w;
    g.dh = h;
    launch(k_gain_apply, dim3(div_up(w, 32), div_up(h, 8)), dim3(32, 8), 0, s, img, pitch, g);
    return launch_check("k_gain_apply");
}

int launch_pack_rgbm(const uint8_t *rgb, long long rgb_pitch, const uint8_t *mask, long long mask_pitch, uint32_t *dst,
                     long long dst_pitch, int w, int h, cudaStream_t s)
{
    dim3 block(32, 8), grid(div_up(w, 32), div_up(h, 8));
    launch(k_pack_rgbm, grid, block, 0, s, rgb, rgb_pitch, mask, mask_pitch, dst, dst_pitch, w, h);
    return launch_check("k_pack_rgbm");
}

}  // namespace sb
