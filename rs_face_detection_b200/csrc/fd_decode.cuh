// fd_decode.cuh — RetinaFace head decode arithmetic as device code (shared by decode_kernel in fd_decode.cu and the fused
// post-CNN kernel in fd_detect_fused.cu).  Every operation is rounded separately, in the reference's order.
#pragma once
#include "fd_internal.cuh"

namespace fd {

typedef unsigned long long u64;

struct HeadPtrs {
    const float *p[3 * FD_MAX_STRIDES];
};

constexpr int CAND_REC = 12;  // floats per candidate record: 10 landmarks, score, pad

#ifdef __CUDACC__
// stride index of a position in the 32|16|8 concatenation
__device__ __forceinline__ int stride_of_pos(const DecodeCfg &c, int pos) {
    int s = 0;
#pragma unroll
    for (int k = 1; k < FD_MAX_STRIDES; ++k)
        if (k < c.n_strides && pos >= c.pos_off[k]) s = k;
    return s;
}
// (stride, local position, anchor) of a global anchor id (concat order 32|16|8, then (h,w,a) — face_detection.rs:410)
__device__ __forceinline__ void split_anchor_id(const DecodeCfg &c, int id, int &s, int &local, int &a) {
    s = 0;
#pragma unroll
    for (int k = 1; k < FD_MAX_STRIDES; ++k)
        if (k < c.n_strides && id >= c.anchor_off[k]) s = k;
    const int r = id - c.anchor_off[s];
    local = r / c.A;
    a = r - local * c.A;
}

struct AnchorGeo {
    float aw, ah, cx, cy;
};
// anchor = base + (w*stride, h*stride, w*stride, h*stride) (anchors.rs:8-16); width/height/centre as face_detection.rs:522-525
__device__ __forceinline__ AnchorGeo anchor_geo(const DecodeCfg &c, int s, int local, int a) {
    const int fw = c.fw[s];
    const int h = local / fw, w = local - h * fw;
    const float sw = (float)(w * c.stride[s]), sh = (float)(h * c.stride[s]);
    const float ax1 = __fadd_rn(c.base[s][a][0], sw), ay1 = __fadd_rn(c.base[s][a][1], sh);
    const float ax2 = __fadd_rn(c.base[s][a][2], sw), ay2 = __fadd_rn(c.base[s][a][3], sh);
    AnchorGeo g;
    g.aw = __fadd_rn(__fsub_rn(ax2, ax1), 1.0f);
    g.ah = __fadd_rn(__fsub_rn(ay2, ay1), 1.0f);
    g.cx = __fadd_rn(ax1, __fmul_rn(0.5f, __fsub_rn(g.aw, 1.0f)));
    g.cy = __fadd_rn(ay1, __fmul_rn(0.5f, __fsub_rn(g.ah, 1.0f)));
    return g;
}
// bbox_pred (face_detection.rs:516-549) + clip_boxes to the padded detector image (:373, bbox_transform.rs:36-42) from the
// anchor's 4 raw box deltas
__device__ __forceinline__ float4 decode_box(const DecodeCfg &c, const float *raw4, const AnchorGeo &g) {
    const float dx = __fmul_rn(raw4[0], c.bbox_stds[0]);  // :366-371
    const float dy = __fmul_rn(raw4[1], c.bbox_stds[1]);
    const float dw = __fmul_rn(raw4[2], c.bbox_stds[2]);
    const float dh = __fmul_rn(raw4[3], c.bbox_stds[3]);
    // :532-535.  exp through fp64 is correctly rounded to <=0.5 ulp; the reference's f32::exp is the platform expf.
    const float pcx = __fadd_rn(__fmul_rn(dx, g.aw), g.cx), pcy = __fadd_rn(__fmul_rn(dy, g.ah), g.cy);
    const float pw = __fmul_rn((float)exp((double)dw), g.aw), ph = __fmul_rn((float)exp((double)dh), g.ah);
    // :539-542
    const float hwx = __fmul_rn(0.5f, __fsub_rn(pw, 1.0f)), hwy = __fmul_rn(0.5f, __fsub_rn(ph, 1.0f));
    float4 box;
    box.x = fmaxf(fminf(__fsub_rn(pcx, hwx), c.clip_w), 0.0f);
    box.y = fmaxf(fminf(__fsub_rn(pcy, hwy), c.clip_h), 0.0f);
    box.z = fmaxf(fminf(__fadd_rn(pcx, hwx), c.clip_w), 0.0f);
    box.w = fmaxf(fminf(__fadd_rn(pcy, hwy), c.clip_h), 0.0f);
    return box;
}
__device__ __forceinline__ float4 decode_box(const DecodeCfg &c, const HeadPtrs &hp, int b, int s, int local, int a, const AnchorGeo &g) {
    const int hw = c.fh[s] * c.fw[s];
    const float *bb = hp.p[3 * s + 1] + (size_t)b * 4 * c.A * hw;
    float raw[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) raw[k] = __ldg(bb + (size_t)(4 * a + k) * hw + local);
    return decode_box(c, raw, g);
}
// landmark_pred from the ANCHOR box, never clipped (face_detection.rs:399, :551-570), from the anchor's 10 raw deltas
__device__ __forceinline__ void decode_landmarks(const DecodeCfg &c, const float *lraw, const AnchorGeo &g, float *out10) {
#pragma unroll
    for (int p = 0; p < 5; ++p) {
        out10[2 * p] = __fadd_rn(__fmul_rn(__fmul_rn(lraw[2 * p], c.landmark_std), g.aw), g.cx);
        out10[2 * p + 1] = __fadd_rn(__fmul_rn(__fmul_rn(lraw[2 * p + 1], c.landmark_std), g.ah), g.cy);
    }
}
__device__ __forceinline__ void decode_landmarks(const DecodeCfg &c, const HeadPtrs &hp, int b, int s, int local, int a,
                                                 const AnchorGeo &g, float *out10) {
    const int hw = c.fh[s] * c.fw[s];
    const float *lm = hp.p[3 * s + 2] + (size_t)b * 10 * c.A * hw;
    float lraw[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) lraw[k] = __ldg(lm + (size_t)(10 * a + k) * hw + local);
    decode_landmarks(c, lraw, g, out10);
}
#endif  // __CUDACC__

}  // namespace fd
