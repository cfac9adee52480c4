// fd_resize.cuh — cv::resize(INTER_LINEAR), 8UC3, OpenCV's fixed-point scheme (imgproc/resize.cpp: 11-bit coefficients,
// int32 horizontal pass, ((b*(T>>4))>>16 ... +2)>>2 vertical pass) as device helpers shared by the preprocess kernels
// (face_detection.rs:156), the model preprocessors (face_extraction.rs:38-77) and the FaceAlignment bbox-crop fallback
// (face_alignment.rs:98-105).
#pragma once
#include "fd_internal.cuh"

namespace fd {

// horizontal + vertical fixed-point taps for one channel
__device__ __forceinline__ int resize_px(const uint8_t *r0, const uint8_t *r1, int x0, int x1, int a0, int a1, int b0, int b1) {
    int t0 = r0[x0] * a0 + r0[x1] * a1;
    int v = (b0 * (t0 >> 4)) >> 16;
    if (b1 != 0) {
        int t1 = r1[x0] * a0 + r1[x1] * a1;
        v += (b1 * (t1 >> 4)) >> 16;
    }
    return (v + 2) >> 2;
}

__device__ __forceinline__ short sat_short_rn(float v) {
    int r = __float2int_rn(v);  // round-half-even, as cvRound
    return (short)max(-32768, min(32767, r));
}

// x tap table for one destination column (cv::resize, INTER_LINEAR): byte offsets of the two taps and their weights
__device__ __forceinline__ void x_taps(int dx, double scale_x, int sw, int *o0, int *o1, short *a0, short *a1) {
    float fx = (float)(((double)dx + 0.5) * scale_x - 0.5);
    int sx = (int)floorf(fx);
    fx = __fsub_rn(fx, (float)sx);
    if (sx < 0) { fx = 0.0f; sx = 0; }
    if (sx >= sw - 1) { fx = 0.0f; sx = sw - 1; }
    *o0 = sx * 3;
    *o1 = min(sx + 1, sw - 1) * 3;
    *a0 = sat_short_rn(__fmul_rn(__fsub_rn(1.0f, fx), 2048.0f));
    *a1 = sat_short_rn(__fmul_rn(fx, 2048.0f));
}
__device__ __forceinline__ void y_taps(int dy, double scale_y, int sh, int *y0, int *y1, int *b0, int *b1) {
    float fy = (float)(((double)dy + 0.5) * scale_y - 0.5);
    int sy = (int)floorf(fy);
    fy = __fsub_rn(fy, (float)sy);
    *b0 = sat_short_rn(__fmul_rn(__fsub_rn(1.0f, fy), 2048.0f));
    *b1 = sat_short_rn(__fmul_rn(fy, 2048.0f));
    *y0 = min(max(sy, 0), sh - 1);
    *y1 = min(max(sy + 1, 0), sh - 1);
}

// FaceAlignment::call's fallback ROI (face_alignment.rs:64-93) when estimateAffinePartial2D returns an empty matrix:
//   det = bbox, or (W/16, H/16, W - W/16, H - H/16) when bbox is None (:66-74);  margin 44 (:76)
//   bb = (max(det0-22, 0), max(det1-22, 0), max(det2+22, W), max(det[1]+22, H))   -- `max` and det[1] as written (:78-81)
//   Rect(x0, y0, x1-x0, y1-y0) with `as i32` casts (:83-90), Mat::roi (:92), cv::resize to the crop size (:98-105).
// Mat::roi accepts the rectangle only if it lies inside the image and cv::resize needs a non-empty source, so the
// reference returns an image iff x1 == W, y1 == H, x0 < W, y0 < H (then the ROI is (x0,y0)..(W,H)); otherwise Err.
// f32::max ignores a NaN operand like fmaxf; `as i32` saturates and maps NaN to 0 like __float2int_rz.
__device__ __forceinline__ bool fallback_roi(const float *bbox, int W, int H, int *x0, int *y0) {
    float d0, d1, d2;
    const float Wf = (float)W, Hf = (float)H;
    if (bbox) {
        d0 = bbox[0]; d1 = bbox[1]; d2 = bbox[2];
    } else {
        d0 = __fmul_rn(Wf, 0.0625f);
        d1 = __fmul_rn(Hf, 0.0625f);
        d2 = __fsub_rn(Wf, d0);
    }
    const int ix0 = __float2int_rz(fmaxf(__fsub_rn(d0, 22.0f), 0.0f));
    const int iy0 = __float2int_rz(fmaxf(__fsub_rn(d1, 22.0f), 0.0f));
    const int ix1 = __float2int_rz(fmaxf(__fadd_rn(d2, 22.0f), Wf));
    const int iy1 = __float2int_rz(fmaxf(__fadd_rn(d1, 22.0f), Hf));
    *x0 = ix0;
    *y0 = iy0;
    return ix1 == W && iy1 == H && ix0 < W && iy0 < H;
}

// one output pixel (b | g << 8 | r << 16) of cv::resize(src ROI (rw x rh) -> (ow x oh), INTER_LINEAR)
__device__ __forceinline__ unsigned resize_pixel24(const uint8_t *roi, int pitch, int rw, int rh, int ow, int oh, int x, int y) {
    if (rw == ow && rh == oh) {   // cv::resize copies when the size is unchanged
        const uint8_t *p = roi + (size_t)y * pitch + (size_t)x * 3;
        return (unsigned)p[0] | ((unsigned)p[1] << 8) | ((unsigned)p[2] << 16);
    }
    const double scale_x = 1.0 / ((double)ow / rw), scale_y = 1.0 / ((double)oh / rh);
    int o0, o1, y0, y1, b0, b1;
    short a0, a1;
    x_taps(x, scale_x, rw, &o0, &o1, &a0, &a1);
    y_taps(y, scale_y, rh, &y0, &y1, &b0, &b1);
    const uint8_t *r0 = roi + (size_t)y0 * pitch, *r1 = roi + (size_t)y1 * pitch;
    const unsigned pb = (unsigned)resize_px(r0, r1, o0, o1, a0, a1, b0, b1);
    const unsigned pg = (unsigned)resize_px(r0, r1, o0 + 1, o1 + 1, a0, a1, b0, b1);
    const unsigned pr = (unsigned)resize_px(r0, r1, o0 + 2, o1 + 2, a0, a1, b0, b1);
    return pb | (pg << 8) | (pr << 16);
}

// ---- 4:2:0 sources: every tap is converted as cv::cvtColor(COLOR_YUV2BGR_*) would have converted the whole frame ------
// OpenCV's BT.601 limited-range conversion (imgproc color_yuv: 20-bit fixed point, round half up, saturate), restated in
// int32 and equal to cv2 4.13 on all 2^24 (Y,U,V) triples.  Returns b | g << 8 | r << 16.
__device__ __forceinline__ unsigned yuv_bgr24(int Y, int U, int V) {
    const int y = max(Y - 16, 0) * 1220542 + (1 << 19), u = U - 128, v = V - 128;
    const int r = (y + 1673527 * v) >> 20, g = (y - 852492 * v - 409993 * u) >> 20, b = (y + 2116026 * u) >> 20;
    return (unsigned)min(max(b, 0), 255) | ((unsigned)min(max(g, 0), 255) << 8) | ((unsigned)min(max(r, 0), 255) << 16);
}
// pixel x of a 4:2:0 row (FMT: SRC_NV12, SRC_NV21 or SRC_PLANAR): its own Y and the chroma of its 2x2 block.  crow is the
// chroma row y/2: interleaved U,V (NV12) or V,U (NV21), or the U row, whose V row is vrow (planar; unused otherwise).
template <int FMT>
__device__ __forceinline__ unsigned yuv_px24(const uint8_t *yrow, const uint8_t *crow, const uint8_t *vrow, int x) {
    if (FMT == SRC_PLANAR) return yuv_bgr24(yrow[x], crow[x >> 1], vrow[x >> 1]);
    if (FMT == SRC_NV21) return yuv_bgr24(yrow[x], crow[x | 1], crow[x & ~1]);
    return yuv_bgr24(yrow[x], crow[x & ~1], crow[x | 1]);
}

// resize_px on the three channels of packed pixels: taps (p00, p01) of the first row, (p10, p11) of the second (read only
// when b1 != 0)
__device__ __forceinline__ unsigned resize_px24(unsigned p00, unsigned p01, unsigned p10, unsigned p11, int a0, int a1, int b0, int b1) {
    unsigned out = 0;
#pragma unroll
    for (int c = 0; c < 24; c += 8) {
        const int t0 = (int)((p00 >> c) & 255u) * a0 + (int)((p01 >> c) & 255u) * a1;
        int v = (b0 * (t0 >> 4)) >> 16;
        if (b1 != 0) {
            const int t1 = (int)((p10 >> c) & 255u) * a0 + (int)((p11 >> c) & 255u) * a1;
            v += (b1 * (t1 >> 4)) >> 16;
        }
        out |= (unsigned)((v + 2) >> 2) << c;
    }
    return out;
}

// resize_pixel24 of the ROI (rx0, ry0)..(rx0 + rw, ry0 + rh) of a 4:2:0 frame (chroma plane uvp, and vp the V plane when
// planar): taps in ROI coordinates, chroma of the frame's own 2x2 blocks (rx0, ry0 may be odd)
// (The V pointers are formed only for the planar format: vp is null otherwise.)
template <int FMT>
__device__ __forceinline__ unsigned resize_pixel24_yuv(const uint8_t *yp, int pitch, const uint8_t *uvp, const uint8_t *vp, int pitch_uv,
                                                       int rx0, int ry0, int rw, int rh, int ow, int oh, int x, int y) {
    if (rw == ow && rh == oh) {
        const int sy = ry0 + y;
        if constexpr (FMT == SRC_PLANAR) {
            const size_t oc = (size_t)(sy >> 1) * pitch_uv;
            return yuv_px24<FMT>(yp + (size_t)sy * pitch, uvp + oc, vp + oc, rx0 + x);
        } else {
            return yuv_px24<FMT>(yp + (size_t)sy * pitch, uvp + (size_t)(sy >> 1) * pitch_uv, nullptr, rx0 + x);
        }
    }
    const double scale_x = 1.0 / ((double)ow / rw), scale_y = 1.0 / ((double)oh / rh);
    int o0, o1, y0, y1, b0, b1;
    short a0, a1;
    x_taps(x, scale_x, rw, &o0, &o1, &a0, &a1);
    y_taps(y, scale_y, rh, &y0, &y1, &b0, &b1);
    const int x0 = rx0 + o0 / 3, x1 = rx0 + o1 / 3, sy0 = ry0 + y0, sy1 = ry0 + y1;
    const uint8_t *r0 = yp + (size_t)sy0 * pitch, *c0 = uvp + (size_t)(sy0 >> 1) * pitch_uv;
    const uint8_t *r1 = yp + (size_t)sy1 * pitch, *c1 = uvp + (size_t)(sy1 >> 1) * pitch_uv;
    const uint8_t *v0 = nullptr, *v1 = nullptr;
    if constexpr (FMT == SRC_PLANAR) {
        v0 = vp + (size_t)(sy0 >> 1) * pitch_uv;
        v1 = vp + (size_t)(sy1 >> 1) * pitch_uv;
    }
    const unsigned p10 = b1 != 0 ? yuv_px24<FMT>(r1, c1, v1, x0) : 0u, p11 = b1 != 0 ? yuv_px24<FMT>(r1, c1, v1, x1) : 0u;
    return resize_px24(yuv_px24<FMT>(r0, c0, v0, x0), yuv_px24<FMT>(r0, c0, v0, x1), p10, p11, a0, a1, b0, b1);
}

// ---- packed 4:2:2 sources (YUY2, UYVY, YVYU): pixel x takes its own Y and the U, V of its pair x & ~1 ------------------
// A row is w/2 macropixels of 4 bytes.  sel is the __byte_perm selector that reorders a macropixel to Y0 U Y1 V (nibble k:
// the source byte that lands in byte k): YUY2 0x3210, UYVY 0x2301, YVYU 0x1230.
// pixel x of a macropixel n already reordered to Y0 U Y1 V
__device__ __forceinline__ unsigned packed_bgr24(unsigned n, int x) {
    return yuv_bgr24((x & 1) ? (n >> 16) & 255u : n & 255u, (n >> 8) & 255u, n >> 24);
}
// pixel x of a packed row at any alignment: three byte reads
__device__ __forceinline__ unsigned packed_px24(const uint8_t *row, unsigned sel, int x) {
    const uint8_t *m = row + 4 * (x >> 1);
    return yuv_bgr24(m[(sel >> ((x & 1) ? 8 : 0)) & 3u], m[(sel >> 4) & 3u], m[(sel >> 12) & 3u]);
}
// resize_pixel24 of the ROI (rx0, ry0)..(rx0 + rw, ry0 + rh) of a packed frame: taps in ROI coordinates, chroma of the
// frame's own pairs (rx0 may be odd)
__device__ __forceinline__ unsigned resize_pixel24_packed(const uint8_t *data, int pitch, unsigned sel, int rx0, int ry0, int rw, int rh,
                                                          int ow, int oh, int x, int y) {
    if (rw == ow && rh == oh) return packed_px24(data + (size_t)(ry0 + y) * pitch, sel, rx0 + x);
    const double scale_x = 1.0 / ((double)ow / rw), scale_y = 1.0 / ((double)oh / rh);
    int o0, o1, y0, y1, b0, b1;
    short a0, a1;
    x_taps(x, scale_x, rw, &o0, &o1, &a0, &a1);
    y_taps(y, scale_y, rh, &y0, &y1, &b0, &b1);
    const int x0 = rx0 + o0 / 3, x1 = rx0 + o1 / 3;
    const uint8_t *r0 = data + (size_t)(ry0 + y0) * pitch, *r1 = data + (size_t)(ry0 + y1) * pitch;
    const unsigned p10 = b1 != 0 ? packed_px24(r1, sel, x0) : 0u, p11 = b1 != 0 ? packed_px24(r1, sel, x1) : 0u;
    return resize_px24(packed_px24(r0, sel, x0), packed_px24(r0, sel, x1), p10, p11, a0, a1, b0, b1);
}

// ---- interleaved RGB-family sources: each tap is the pixel cv::cvtColor(COLOR_RGB2BGR / RGBA2BGR / BGRA2BGR / GRAY2BGR)
// would have made, and the resize arithmetic is the BGR one ---------------------------------------------------------------
// b | g << 8 | r << 16 of a packed pixel read as b, g, r (RGB24: channels 0 and 2 exchanged)
__device__ __forceinline__ unsigned swap_rb24(unsigned p) { return __byte_perm(p, 0u, 0x3012); }
// pixel x of a 4-byte row (RGBA / BGRA) at any alignment: three byte reads; sel reorders a pixel word to B,G,R,x (nibble k:
// the source byte that lands in byte k): RGBA 0x3012, BGRA 0x3210
__device__ __forceinline__ unsigned px32_px24(const uint8_t *row, unsigned sel, int x) {
    const uint8_t *p = row + 4 * x;
    return (unsigned)p[sel & 3u] | ((unsigned)p[(sel >> 4) & 3u] << 8) | ((unsigned)p[(sel >> 8) & 3u] << 16);
}
// pixel x of a GRAY8 row as BGR
__device__ __forceinline__ unsigned gray_px24(const uint8_t *row, int x) { return (unsigned)row[x] * 0x010101u; }
// resize_pixel24 of the ROI (rx0, ry0)..(rx0 + rw, ry0 + rh) of an RGBA / BGRA (FMT = SRC_PX32) or GRAY8 frame.  A GRAY8
// pixel is resized once: the three channels of its BGR image are equal.
template <int FMT>
__device__ __forceinline__ unsigned resize_pixel24_rgb(const uint8_t *data, int pitch, unsigned sel, int rx0, int ry0, int rw, int rh, int ow,
                                                       int oh, int x, int y) {
    if (rw == ow && rh == oh) {
        const uint8_t *row = data + (size_t)(ry0 + y) * pitch;
        return FMT == SRC_GRAY8 ? gray_px24(row, rx0 + x) : px32_px24(row, sel, rx0 + x);
    }
    const double scale_x = 1.0 / ((double)ow / rw), scale_y = 1.0 / ((double)oh / rh);
    int o0, o1, y0, y1, b0, b1;
    short a0, a1;
    x_taps(x, scale_x, rw, &o0, &o1, &a0, &a1);
    y_taps(y, scale_y, rh, &y0, &y1, &b0, &b1);
    const int x0 = rx0 + o0 / 3, x1 = rx0 + o1 / 3;
    const uint8_t *r0 = data + (size_t)(ry0 + y0) * pitch, *r1 = data + (size_t)(ry0 + y1) * pitch;
    if constexpr (FMT == SRC_GRAY8) return (unsigned)resize_px(r0, r1, x0, x1, a0, a1, b0, b1) * 0x010101u;
    const unsigned p10 = b1 != 0 ? px32_px24(r1, sel, x0) : 0u, p11 = b1 != 0 ? px32_px24(r1, sel, x1) : 0u;
    return resize_px24(px32_px24(r0, sel, x0), px32_px24(r0, sel, x1), p10, p11, a0, a1, b0, b1);
}

}  // namespace fd
