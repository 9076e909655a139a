// sb_yuv.cu -- YUV 4:2:0 frames in and out of the compositor (NV12 / I420, BT.601 limited range), bit-exact to
// cv.cvtColor(COLOR_YUV2BGR_NV12 / _I420) and cv.cvtColor(COLOR_BGR2YUV_I420).
//
// Both directions are OpenCV's fixed-point closed forms (20 fractional bits, every intermediate fits in int32):
//   YUV -> BGR  y = max(0, Y - 16) * 1220542, u = U - 128, v = V - 128, H = 1 << 19
//               R = sat8((y + H + 1673527 v) >> 20), G = sat8((y + H - 852492 v - 409993 u) >> 20), B = sat8((y + H + 2116026 u) >> 20)
//   BGR -> YUV  Y = sat8((269484 R + 528482 G + 102760 B + H + (16 << 20)) >> 20) for every pixel;
//               U = sat8((-155188 R - 305135 G + 460324 B + H + (128 << 20)) >> 20) and
//               V = sat8((460324 R - 385875 G - 74448 B + H + (128 << 20)) >> 20) from the TOP-LEFT pixel of each 2x2 block
// One thread per 2x2 block: the block's chroma pair is loaded (or computed) once and its chroma terms multiplied once.
// Frame sizes are even (cv2 rejects odd ones); plane pitches are even (the compositor's staging and output buffers are
// dense with an even width), so the two luma bytes of a block row travel as one 16-bit word.
#include "sb_launch.h"

namespace sb {
namespace {

#define YUV_BX 32
#define YUV_BY 8

__device__ __forceinline__ unsigned sat8(int v) { return (unsigned)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

// b | g << 8 | r << 16 of one pixel from its luma and the block's three chroma terms (which include the rounding half)
__device__ __forceinline__ unsigned yuv_pixel(unsigned Y, int rc, int gc, int bc)
{
    const int y = ((int)Y > 16 ? (int)Y - 16 : 0) * 1220542;
    return sat8((y + bc) >> 20) | (sat8((y + gc) >> 20) << 8) | (sat8((y + rc) >> 20) << 16);
}

// FMT: SB_PIX_NV12 (u = interleaved UV plane) or SB_PIX_I420 (u, v planes).  WORD: write the word-per-pixel source of the
// warp kernel (WarpJob::src4, the layout of k_repack_rgbx) instead of the packed 3-byte one (WarpJob::src).
template <int FMT, bool WORD>
__global__ void __launch_bounds__(YUV_BX *YUV_BY) k_yuv420_to_src(const YuvPlanes in, int w2, int h2, uint8_t *__restrict__ bgr,
                                                                  long long bgr_pitch, uint32_t *__restrict__ bgrx, long long bgrx_pitch)
{
    const int bx = blockIdx.x * YUV_BX + threadIdx.x, by = blockIdx.y * YUV_BY + threadIdx.y;
    if (bx >= w2 || by >= h2) return;
    int U, V;
    if (FMT == SB_PIX_NV12) {
        const unsigned uv = __ldg(reinterpret_cast<const uint16_t *>(in.u + (long long)by * in.upitch) + bx);
        U = (int)(uv & 255u);
        V = (int)(uv >> 8);
    } else {
        U = (int)__ldg(in.u + (long long)by * in.upitch + bx);
        V = (int)__ldg(in.v + (long long)by * in.vpitch + bx);
    }
    const int u = U - 128, v = V - 128, H = 1 << 19;
    const int rc = H + 1673527 * v, gc = H - 852492 * v - 409993 * u, bc = H + 2116026 * u;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const long long y = 2ll * by + r;
        const unsigned yy = __ldg(reinterpret_cast<const uint16_t *>(in.y + y * in.ypitch) + bx);
        const unsigned p0 = yuv_pixel(yy & 255u, rc, gc, bc), p1 = yuv_pixel(yy >> 8, rc, gc, bc);
        if (WORD) {
            *reinterpret_cast<uint2 *>(bgrx + y * bgrx_pitch + 2 * bx) = make_uint2(p0, p1);  // pitch and x even: 8-byte aligned
        } else {
            // six bytes b0 g0 r0 b1 g1 r1 at an even offset: three 16-bit stores
            uint16_t *d = reinterpret_cast<uint16_t *>(bgr + y * bgr_pitch + 6ll * bx);
            d[0] = (uint16_t)(p0 & 0xffffu);
            d[1] = (uint16_t)((p0 >> 16) | ((p1 & 255u) << 8));
            d[2] = (uint16_t)(p1 >> 8);
        }
    }
}

__device__ __forceinline__ unsigned luma(unsigned b, unsigned g, unsigned r)
{
    return sat8((int)(269484 * r + 528482 * g + 102760 * b + (1u << 19) + (16u << 20)) >> 20);
}

template <int FMT>
__global__ void __launch_bounds__(YUV_BX *YUV_BY) k_bgr_to_yuv420(const uint8_t *__restrict__ bgr, long long bgr_pitch, int w2, int h2,
                                                                  YuvOut out)
{
    const int bx = blockIdx.x * YUV_BX + threadIdx.x, by = blockIdx.y * YUV_BY + threadIdx.y;
    if (bx >= w2 || by >= h2) return;
    const int H = 1 << 19;
    int U = 0, V = 0;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const long long y = 2ll * by + r;
        const uint8_t *p = bgr + y * bgr_pitch + 6ll * bx;
        const unsigned b0 = __ldg(p), g0 = __ldg(p + 1), r0 = __ldg(p + 2), b1 = __ldg(p + 3), g1 = __ldg(p + 4), r1 = __ldg(p + 5);
        *reinterpret_cast<uint16_t *>(out.y + y * out.ypitch + 2ll * bx) = (uint16_t)(luma(b0, g0, r0) | (luma(b1, g1, r1) << 8));
        if (r == 0) {
            const int R = (int)r0, G = (int)g0, B = (int)b0;
            U = (int)sat8((-155188 * R - 305135 * G + 460324 * B + H + (128 << 20)) >> 20);
            V = (int)sat8((460324 * R - 385875 * G - 74448 * B + H + (128 << 20)) >> 20);
        }
    }
    if (FMT == SB_PIX_NV12) {
        *reinterpret_cast<uint16_t *>(out.u + (long long)by * out.upitch + 2ll * bx) = (uint16_t)(U | (V << 8));
    } else {
        out.u[(long long)by * out.upitch + bx] = (uint8_t)U;
        out.v[(long long)by * out.vpitch + bx] = (uint8_t)V;
    }
}

}  // namespace

int launch_yuv420_to_src(int fmt, const YuvPlanes &in, int w, int h, uint8_t *bgr, long long bgr_pitch, uint32_t *bgrx,
                         long long bgrx_pitch, cudaStream_t s)
{
    const int w2 = w / 2, h2 = h / 2;
    if (w2 <= 0 || h2 <= 0) return SB_OK;
    const dim3 block(YUV_BX, YUV_BY), grid(div_up(w2, YUV_BX), div_up(h2, YUV_BY));
    if (fmt == SB_PIX_NV12) {
        if (bgrx)
            launch(k_yuv420_to_src<SB_PIX_NV12, true>, grid, block, 0, s, in, w2, h2, bgr, bgr_pitch, bgrx, bgrx_pitch);
        else
            launch(k_yuv420_to_src<SB_PIX_NV12, false>, grid, block, 0, s, in, w2, h2, bgr, bgr_pitch, bgrx, bgrx_pitch);
    } else {
        if (bgrx)
            launch(k_yuv420_to_src<SB_PIX_I420, true>, grid, block, 0, s, in, w2, h2, bgr, bgr_pitch, bgrx, bgrx_pitch);
        else
            launch(k_yuv420_to_src<SB_PIX_I420, false>, grid, block, 0, s, in, w2, h2, bgr, bgr_pitch, bgrx, bgrx_pitch);
    }
    return launch_check("k_yuv420_to_src");
}

int launch_bgr_to_yuv420(int fmt, const uint8_t *bgr, long long bgr_pitch, int w, int h, const YuvOut &out, cudaStream_t s)
{
    const int w2 = w / 2, h2 = h / 2;
    if (w2 <= 0 || h2 <= 0) return SB_OK;
    const dim3 block(YUV_BX, YUV_BY), grid(div_up(w2, YUV_BX), div_up(h2, YUV_BY));
    if (fmt == SB_PIX_NV12)
        launch(k_bgr_to_yuv420<SB_PIX_NV12>, grid, block, 0, s, bgr, bgr_pitch, w2, h2, out);
    else
        launch(k_bgr_to_yuv420<SB_PIX_I420>, grid, block, 0, s, bgr, bgr_pitch, w2, h2, out);
    return launch_check("k_bgr_to_yuv420");
}

}  // namespace sb
