// fd_align.cu — 5-point similarity estimate (LMedS) + fixed-point bilinear warp to the ArcFace crop, batched.
//
// Replaces FaceAlignment::call (face_alignment.rs:27-141): cv::estimateAffinePartial2D(landmarks, template, LMEDS,
// 3.0, 2000, 0.99, 10) (:50-59) and cv::warpAffine(img, M, (112,112), INTER_LINEAR, BORDER_CONSTANT, 0) (:119-126).
//
// estimate_kernel: 16 lanes per face, fp64 (device code in fd_estimate.cuh; the batched pipeline runs it inside the fused
// detect kernel instead): the operation order of OpenCV's calib3d/ptsetreg.cpp (RNG reseeded per call, 2-point exact
// similarity per LMedS iteration, float32 squared errors, median, inlier threshold) followed by the least-squares
// similarity over the inliers that OpenCV's LM refinement converges to.
// warp_fixed_kernel (112x112) / warp_kernel (any size): persistent, ticket-scheduled kernels evaluating OpenCV's
// imgwarp.cpp fixed-point scheme (inverse matrix in fp64, 10-bit coordinates, 5-bit sub-pixel position, 15-bit weights,
// per-tap BORDER_CONSTANT) so crops are bit-identical, not "within a few grey levels".
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cfloat>
#include <type_traits>
#include "fd_internal.cuh"
#include "fd_estimate.cuh"
#include "fd_resize.cuh"

namespace fd {

struct EstArgs {
    const float *from;     // (F,5,2)
    const float *to;       // (F,5,2) or nullptr -> template
    const int *count_dev;  // optional device-side F
    int F;
    EstConst ec;
    double *M12;           // (F,12): M (6) then inverse (6)
    double *M_out;         // optional (F,6)
    uint8_t *ok;           // (F)
    uint8_t *ok_out;       // optional (F)
};

__global__ void estimate_kernel(EstArgs a) {
    const int F = a.count_dev ? min(*a.count_dev, a.F) : a.F;
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int f = gt / EST_LANES, sub = gt % EST_LANES;
    const bool live = f < F;
    const int fc = live ? f : 0;
    float from[10], to[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) {
        from[k] = live ? a.from[(size_t)fc * 10 + k] : 0.0f;
        to[k] = a.to ? (live ? a.to[(size_t)fc * 10 + k] : 0.0f) : a.ec.tmpl[k];
    }
    double M[6], iM[6];
    bool ok;
    estimate_group(a.ec, from, to, live, sub, M, iM, ok);
    if (!live || sub != 0) return;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        a.M12[(size_t)f * 12 + k] = M[k];
        a.M12[(size_t)f * 12 + 6 + k] = iM[k];
        if (a.M_out) a.M_out[(size_t)f * 6 + k] = M[k];
    }
    a.ok[f] = ok ? 1 : 0;
    if (a.ok_out) a.ok_out[f] = ok ? 1 : 0;
}

// M given by the caller (fd_warp_affine): fill M12 with M and its inverse
__global__ void invert_kernel(const double *M, int F, double *M12, uint8_t *ok) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    double m[6], iM[6];
    for (int k = 0; k < 6; ++k) m[k] = M[(size_t)f * 6 + k];
    invert_affine(m, iM);
    for (int k = 0; k < 6; ++k) {
        M12[(size_t)f * 12 + k] = m[k];
        M12[(size_t)f * 12 + 6 + k] = iM[k];
    }
    ok[f] = 1;
}

constexpr int WARP_BAND = 16;      // output rows per work item
constexpr int WARP_THREADS = 256;

struct WarpArgs {
    const FrameDev *frames;
    const int *frame_idx;  // (F) or nullptr -> frame 0
    const double *M12;
    const uint8_t *ok;
    const int *count_dev;  // optional
    int F;
    uint8_t *crops;        // (F, ch, cw, 3)
    int cw, ch;
    int bands;             // ceil(ch / WARP_BAND)
    unsigned cw_magic;     // floor(2^32 / cw) + 1: p / cw == umulhi(p, cw_magic) for p < 2^20 (cw <= 4096)
    int *ticket;           // [0] next work item, [1] CTAs finished (both return to 0 when the launch ends)
    // FaceAlignment::call's bbox-crop fallback (face_alignment.rs:64-116) for faces whose estimate is empty (ok == 0)
    const float *bbox;     // rows of x1,y1,x2,y2,... (bbox_stride floats apart) or nullptr (bbox == None)
    int bbox_stride;
    const int *sel;        // optional (F,2) = {bbox row, key-point row} (fd_select_detections); key-point row < 0: landmarks == None
    uint8_t *mode_out;     // optional (F): 1 = similarity warp, 2 = bbox-crop fallback, 0 = the reference returns Err (zero crop)
    long long *dbg;        // FD_WARP_DBG=1: per-CTA timestamps {entry, first item start, first item end, exit, items, sum of item ns}
};
__device__ __forceinline__ long long warp_now() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Resolves the fallback of face f: returns true and the ROI origin when the reference would crop + resize, false when it
// returns Err (landmarks == None: cv::estimateAffinePartial2D asserts on the empty Mat; ROI outside the image: Mat::roi).
__device__ __forceinline__ bool warp_fallback_roi(const WarpArgs &a, int f, int fw, int fh, int *rx0, int *ry0) {
    const float *bb = nullptr;
    if (a.sel) {
        if (a.sel[2 * f + 1] < 0) return false;
        const int br = a.sel[2 * f];
        if (br >= 0 && a.bbox) bb = a.bbox + (size_t)br * a.bbox_stride;
    } else if (a.bbox) {
        bb = a.bbox + (size_t)f * a.bbox_stride;
    }
    return fallback_roi(bb, fw, fh, rx0, ry0);
}

// The 6 bytes of two horizontally adjacent BGR pixels at byte offset `off` of an 8-byte aligned base, extracted from the
// two aligned 64-bit words that cover them (lo = bytes 0..3, hi = bytes 4..5 in its low half).
__device__ __forceinline__ void extract6(uint2 q0, uint2 q1, unsigned off, unsigned &lo, unsigned &hi) {
    const bool up = (off & 4u) != 0;
    const unsigned a = up ? q0.y : q0.x, b = up ? q1.x : q0.y, c = up ? q1.y : q1.x;
    const unsigned sft = (off & 3u) * 8;
    lo = __funnelshift_r(a, b, sft);
    hi = __funnelshift_r(b, c, sft);
}
__device__ __forceinline__ void load6_fast(const uint8_t *p, unsigned &lo, unsigned &hi) {
    const uintptr_t ad = reinterpret_cast<uintptr_t>(p);
    const uint2 *al = reinterpret_cast<const uint2 *>(ad & ~(uintptr_t)7);
    extract6(__ldg(al), __ldg(al + 1), (unsigned)(ad & 7), lo, hi);
}
// guarded variant for the frame's first/last bytes and for single-column border taps
__device__ __forceinline__ void load6_safe(const uint8_t *p, const uint8_t *lo_lim, const uint8_t *hi_lim, unsigned &lo, unsigned &hi) {
    const uintptr_t ad = reinterpret_cast<uintptr_t>(p);
    const uint8_t *al = reinterpret_cast<const uint8_t *>(ad & ~(uintptr_t)7);
    if (al >= lo_lim && al + 16 <= hi_lim) {
        load6_fast(p, lo, hi);
        return;
    }
    lo = hi = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) lo |= (unsigned)__ldg(p + k) << (8 * k);
    hi = (unsigned)__ldg(p + 4) | ((unsigned)__ldg(p + 5) << 8);
}

// OpenCV: out = (sum_ij v_ij * W_ij + 2^14) >> 15 with W_ij = a_i * b_j * 32 (a = {32-ay, ay}, b = {32-ax, ax}; the
// 15-bit table entries are exact multiples of 32).  Integer arithmetic is exact, so the sum is evaluated separably:
// horizontal 2-tap dot products with 6-bit weights (dp4a on the packed byte pair), then the vertical pair; and
// (32*S + 2^14) >> 15 == (S + 512) >> 10.  Returns the pixel as b | g << 8 | r << 16.
// RB: the taps are R,G,B (RGB24), so channels 0 and 2 are taken the other way round.  Bytes 6 and 7 of [lo | hi] contribute
// nothing (their weights are 0), so a caller may leave them undefined.
template <bool RB = false>
__device__ __forceinline__ unsigned blend24(unsigned lo0, unsigned hi0, unsigned lo1, unsigned hi1, int ax, int ay) {
    constexpr unsigned SB = RB ? 0x7752 : 0x7730, SR = RB ? 0x7730 : 0x7752;
    const unsigned wx = (unsigned)(32 - ax) | ((unsigned)ax << 8);   // bytes: [32-ax, ax, 0, 0]
    const int wy0 = 32 - ay, wy1 = ay;
    // byte pairs (tap0, tap1) per channel: b = bytes (0,3), g = (1,4), r = (2,5) of [lo | hi]
    const int hb0 = (int)__dp4a(__byte_perm(lo0, hi0, SB), wx, 0u), hb1 = (int)__dp4a(__byte_perm(lo1, hi1, SB), wx, 0u);
    const int hg0 = (int)__dp4a(__byte_perm(lo0, hi0, 0x7741), wx, 0u), hg1 = (int)__dp4a(__byte_perm(lo1, hi1, 0x7741), wx, 0u);
    const int hr0 = (int)__dp4a(__byte_perm(lo0, hi0, SR), wx, 0u), hr1 = (int)__dp4a(__byte_perm(lo1, hi1, SR), wx, 0u);
    const unsigned ob = (unsigned)(hb0 * wy0 + hb1 * wy1 + 512) >> 10;
    const unsigned og = (unsigned)(hg0 * wy0 + hg1 * wy1 + 512) >> 10;
    const unsigned orr = (unsigned)(hr0 * wy0 + hr1 * wy1 + 512) >> 10;
    return ob | (og << 8) | (orr << 16);
}

// blend24 for the fixed-size kernel: ay6 = ay << 6, so each channel's sum lands in byte 2 of its word ((S + 512) << 6 < 2^24) and
// two byte permutes assemble the pixel instead of three shifts and two merges.  RB: as for blend24.
template <bool RB = false>
__device__ __forceinline__ unsigned blend24_scaled(unsigned lo0, unsigned hi0, unsigned lo1, unsigned hi1, int ax, int ay6) {
    constexpr unsigned SB = RB ? 0x7752 : 0x7730, SR = RB ? 0x7730 : 0x7752;
    const unsigned wx = (unsigned)(32 - ax) | ((unsigned)ax << 8);
    const int wy0 = 2048 - ay6, wy1 = ay6;
    const int hb0 = (int)__dp4a(__byte_perm(lo0, hi0, SB), wx, 0u), hb1 = (int)__dp4a(__byte_perm(lo1, hi1, SB), wx, 0u);
    const int hg0 = (int)__dp4a(__byte_perm(lo0, hi0, 0x7741), wx, 0u), hg1 = (int)__dp4a(__byte_perm(lo1, hi1, 0x7741), wx, 0u);
    const int hr0 = (int)__dp4a(__byte_perm(lo0, hi0, SR), wx, 0u), hr1 = (int)__dp4a(__byte_perm(lo1, hi1, SR), wx, 0u);
    const unsigned sb = (unsigned)(hb0 * wy0 + hb1 * wy1 + 32768);
    const unsigned sg = (unsigned)(hg0 * wy0 + hg1 * wy1 + 32768);
    const unsigned sr = (unsigned)(hr0 * wy0 + hr1 * wy1 + 32768);
    return __byte_perm(__byte_perm(sb, sg, 0x7762), sr, 0x7610);   // b | g << 8 | r << 16, byte 3 = 0
}

// blend24 / blend24_scaled of a GRAY8 tap square: the one channel is blended once and replicated.  g0, g1: the tap bytes
// (sx, sx+1) of rows sy, sy+1 in bytes 0 and 1.
__device__ __forceinline__ unsigned blend8(unsigned g0, unsigned g1, int ax, int ay) {
    const unsigned wx = (unsigned)(32 - ax) | ((unsigned)ax << 8);
    const int h0 = (int)__dp4a(g0, wx, 0u), h1 = (int)__dp4a(g1, wx, 0u);
    return ((unsigned)(h0 * (32 - ay) + h1 * ay + 512) >> 10) * 0x010101u;
}
__device__ __forceinline__ unsigned blend8_scaled(unsigned g0, unsigned g1, int ax, int ay6) {
    const unsigned wx = (unsigned)(32 - ax) | ((unsigned)ax << 8);
    const int h0 = (int)__dp4a(g0, wx, 0u), h1 = (int)__dp4a(g1, wx, 0u);
    return __byte_perm((unsigned)(h0 * (2048 - ay6) + h1 * ay6 + 32768), 0u, 0x4222);   // byte 2 thrice, byte 3 = 0
}

// One output pixel with per-tap BORDER_CONSTANT(0) tests; X, Y are the 5-bit sub-pixel fixed-point source coordinates.
// RB: an RGB24 frame (blend24<true>).
template <bool RB = false>
__device__ __forceinline__ unsigned border_tap_blend(const uint8_t *data, int w, int h, int pitch, const uint8_t *lo_lim,
                                                     const uint8_t *hi_lim, int X, int Y) {
    unsigned lo0 = 0, hi0 = 0, lo1 = 0, hi1 = 0;
    const int sx = max(-32768, min(32767, X >> 5)), sy = max(-32768, min(32767, Y >> 5));   // saturate_cast<short>
    const bool inx0 = sx >= 0 && sx < w, inx1 = sx + 1 >= 0 && sx + 1 < w;
    const bool iny0 = sy >= 0 && sy < h, iny1 = sy + 1 >= 0 && sy + 1 < h;
    if (inx0 && inx1) {
        const uint8_t *t0 = data + (ptrdiff_t)sy * pitch + (ptrdiff_t)sx * 3;
        if (iny0) load6_safe(t0, lo_lim, hi_lim, lo0, hi0);
        if (iny1) load6_safe(t0 + pitch, lo_lim, hi_lim, lo1, hi1);
    } else if (inx0 || inx1) {  // one tap column outside the image
        const int sxv = inx0 ? sx : sx + 1;
        unsigned t0 = 0, t1 = 0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            if (iny0) t0 |= (unsigned)__ldg(data + (ptrdiff_t)sy * pitch + sxv * 3 + c) << (8 * c);
            if (iny1) t1 |= (unsigned)__ldg(data + (ptrdiff_t)(sy + 1) * pitch + sxv * 3 + c) << (8 * c);
        }
        if (inx0) { lo0 = t0; lo1 = t1; }              // tap 0 valid, tap 1 (bytes 3..5) zero
        else { lo0 = t0 << 24; hi0 = t0 >> 8; lo1 = t1 << 24; hi1 = t1 >> 8; }  // tap 1 valid
    }
    return blend24<RB>(lo0, hi0, lo1, hi1, X & 31, Y & 31);
}

// ---- 4:2:0 sources: the four taps are converted to BGR (yuv_bgr24) and blended with the same arithmetic --------------
// Two horizontally adjacent packed pixels p0, p1 as the (lo, hi) byte pair blend24 takes: bytes b0 g0 r0 b1 | g1 r1.
__device__ __forceinline__ void pack6(unsigned p0, unsigned p1, unsigned &lo, unsigned &hi) {
    lo = p0 | (p1 << 24);
    hi = p1 >> 8;
}
// Interior tap square (sx, sy)..(sx+1, sy+1) of an NV12/NV21 frame whose planes and pitches are 4-byte aligned: four bytes
// at sx of each Y row and at sx & ~1 of each tap row's chroma row (the chroma pairs of both columns: one pair when sx is
// even, two when it is odd; both rows read the same chroma row when sy is even), each cut from the two aligned words that
// cover it.
struct Nv12Quad {
    unsigned y0[2], y1[2], c0[2], c1[2];
    unsigned sy_sh, sc_sh;   // byte phase of the Y and of the UV reads (the two rows of a plane share it)
    bool odd;
};
__device__ __forceinline__ void nv12_quad_load(const uint8_t *yp, unsigned py, const uint8_t *uvp, unsigned puv, int sx, int sy, Nv12Quad &q) {
    const unsigned oy = (unsigned)sy * py + (unsigned)sx, xc = (unsigned)(sx & ~1);
    const unsigned oc0 = (unsigned)(sy >> 1) * puv + xc, oc1 = (unsigned)((sy + 1) >> 1) * puv + xc;
    const unsigned *ry0 = reinterpret_cast<const unsigned *>(yp + (oy & ~3u));
    const unsigned *ry1 = reinterpret_cast<const unsigned *>(yp + ((oy + py) & ~3u));
    const unsigned *rc0 = reinterpret_cast<const unsigned *>(uvp + (oc0 & ~3u));
    const unsigned *rc1 = reinterpret_cast<const unsigned *>(uvp + (oc1 & ~3u));
    q.y0[0] = __ldg(ry0); q.y0[1] = __ldg(ry0 + 1);
    q.y1[0] = __ldg(ry1); q.y1[1] = __ldg(ry1 + 1);
    q.c0[0] = __ldg(rc0); q.c0[1] = __ldg(rc0 + 1);
    q.c1[0] = __ldg(rc1); q.c1[1] = __ldg(rc1 + 1);
    q.sy_sh = (oy & 3u) * 8;
    q.sc_sh = (oc0 & 3u) * 8;
    q.odd = (sx & 1) != 0;
}
// FMT: SRC_NV12 (chroma bytes U,V) or SRC_NV21 (V,U)
template <int FMT>
__device__ __forceinline__ void nv12_row_taps(unsigned yw, unsigned cw, bool odd, unsigned &lo, unsigned &hi) {
    const unsigned e1 = odd ? (cw >> 16) & 255u : cw & 255u, o1 = odd ? cw >> 24 : (cw >> 8) & 255u;   // chroma pair of column sx+1
    if (FMT == SRC_NV21) pack6(yuv_bgr24(yw & 255u, (cw >> 8) & 255u, cw & 255u), yuv_bgr24((yw >> 8) & 255u, o1, e1), lo, hi);
    else pack6(yuv_bgr24(yw & 255u, cw & 255u, (cw >> 8) & 255u), yuv_bgr24((yw >> 8) & 255u, e1, o1), lo, hi);
}
template <int FMT>
__device__ __forceinline__ void nv12_quad_taps(const Nv12Quad &q, unsigned &lo0, unsigned &hi0, unsigned &lo1, unsigned &hi1) {
    nv12_row_taps<FMT>(__funnelshift_r(q.y0[0], q.y0[1], q.sy_sh), __funnelshift_r(q.c0[0], q.c0[1], q.sc_sh), q.odd, lo0, hi0);
    nv12_row_taps<FMT>(__funnelshift_r(q.y1[0], q.y1[1], q.sy_sh), __funnelshift_r(q.c1[0], q.c1[1], q.sc_sh), q.odd, lo1, hi1);
}
// The same square of a planar (I420/YV12) frame: four bytes at sx of each Y row, and at sx >> 1 of each tap row's U and V
// rows (byte 0: the chroma of column sx; byte 1: that of column sx+1 when sx is odd).  The U and V planes share the pitch
// and the 4-byte phase.
struct PlanarQuad {
    unsigned y0[2], y1[2], u0[2], v0[2], u1[2], v1[2];
    unsigned sy_sh, sc_sh;
    bool odd;
};
__device__ __forceinline__ void planar_quad_load(const uint8_t *yp, unsigned py, const uint8_t *up, const uint8_t *vp, unsigned puv, int sx,
                                                 int sy, PlanarQuad &q) {
    const unsigned oy = (unsigned)sy * py + (unsigned)sx, xc = (unsigned)(sx >> 1);
    const unsigned oc0 = (unsigned)(sy >> 1) * puv + xc, oc1 = (unsigned)((sy + 1) >> 1) * puv + xc;
    const unsigned *ry0 = reinterpret_cast<const unsigned *>(yp + (oy & ~3u));
    const unsigned *ry1 = reinterpret_cast<const unsigned *>(yp + ((oy + py) & ~3u));
    const unsigned *ru0 = reinterpret_cast<const unsigned *>(up + (oc0 & ~3u)), *rv0 = reinterpret_cast<const unsigned *>(vp + (oc0 & ~3u));
    const unsigned *ru1 = reinterpret_cast<const unsigned *>(up + (oc1 & ~3u)), *rv1 = reinterpret_cast<const unsigned *>(vp + (oc1 & ~3u));
    q.y0[0] = __ldg(ry0); q.y0[1] = __ldg(ry0 + 1);
    q.y1[0] = __ldg(ry1); q.y1[1] = __ldg(ry1 + 1);
    q.u0[0] = __ldg(ru0); q.u0[1] = __ldg(ru0 + 1);
    q.v0[0] = __ldg(rv0); q.v0[1] = __ldg(rv0 + 1);
    q.u1[0] = __ldg(ru1); q.u1[1] = __ldg(ru1 + 1);
    q.v1[0] = __ldg(rv1); q.v1[1] = __ldg(rv1 + 1);
    q.sy_sh = (oy & 3u) * 8;
    q.sc_sh = (oc0 & 3u) * 8;
    q.odd = (sx & 1) != 0;
}
__device__ __forceinline__ void planar_row_taps(unsigned yw, unsigned uw, unsigned vw, bool odd, unsigned &lo, unsigned &hi) {
    const unsigned u1 = odd ? (uw >> 8) & 255u : uw & 255u, v1 = odd ? (vw >> 8) & 255u : vw & 255u;
    pack6(yuv_bgr24(yw & 255u, uw & 255u, vw & 255u), yuv_bgr24((yw >> 8) & 255u, u1, v1), lo, hi);
}
__device__ __forceinline__ void planar_quad_taps(const PlanarQuad &q, unsigned &lo0, unsigned &hi0, unsigned &lo1, unsigned &hi1) {
    planar_row_taps(__funnelshift_r(q.y0[0], q.y0[1], q.sy_sh), __funnelshift_r(q.u0[0], q.u0[1], q.sc_sh),
                    __funnelshift_r(q.v0[0], q.v0[1], q.sc_sh), q.odd, lo0, hi0);
    planar_row_taps(__funnelshift_r(q.y1[0], q.y1[1], q.sy_sh), __funnelshift_r(q.u1[0], q.u1[1], q.sc_sh),
                    __funnelshift_r(q.v1[0], q.v1[1], q.sc_sh), q.odd, lo1, hi1);
}
// The same square of a packed 4:2:2 frame (data and pitch 4-byte aligned): per tap row, the aligned macropixel word of
// column sx and, when sx is odd, that of column sx+1 (for an even sx both columns share one word).  No byte past the words
// of the two columns is read.  sel reorders a word to Y0 U Y1 V.
struct PackedQuad {
    unsigned r0[2], r1[2];   // words of columns sx, sx+1 in tap rows sy, sy+1
    unsigned sel;
    bool odd;
};
__device__ __forceinline__ void packed_quad_load(const uint8_t *p, unsigned pitch, unsigned sel, int sx, int sy, PackedQuad &q) {
    const unsigned o = (unsigned)sy * pitch + 2u * (unsigned)(sx & ~1);
    const unsigned *w0 = reinterpret_cast<const unsigned *>(p + o), *w1 = reinterpret_cast<const unsigned *>(p + o + pitch);
    q.odd = (sx & 1) != 0;
    q.r0[0] = __ldg(w0); q.r1[0] = __ldg(w1);
    q.r0[1] = q.odd ? __ldg(w0 + 1) : q.r0[0];
    q.r1[1] = q.odd ? __ldg(w1 + 1) : q.r1[0];
    q.sel = sel;
}
__device__ __forceinline__ void packed_row_taps(unsigned a, unsigned b, unsigned sel, bool odd, unsigned &lo, unsigned &hi) {
    a = __byte_perm(a, 0u, sel);
    b = __byte_perm(b, 0u, sel);
    pack6(packed_bgr24(a, odd ? 1 : 0), packed_bgr24(b, odd ? 0 : 1), lo, hi);
}
// The same square of an RGBA / BGRA frame (data and pitch 4-byte aligned): per tap row, the words of pixels sx and sx+1
// (8 bytes at 4-byte alignment).  No byte outside the four tap pixels is read.  sel reorders a word to B,G,R,x.
struct Px32Quad {
    unsigned r0[2], r1[2];   // words of columns sx, sx+1 in tap rows sy, sy+1
    unsigned sel;
};
__device__ __forceinline__ void px32_quad_load(const uint8_t *p, unsigned pitch, unsigned sel, int sx, int sy, Px32Quad &q) {
    const unsigned o = (unsigned)sy * pitch + 4u * (unsigned)sx;
    const unsigned *w0 = reinterpret_cast<const unsigned *>(p + o), *w1 = reinterpret_cast<const unsigned *>(p + o + pitch);
    q.r0[0] = __ldg(w0); q.r0[1] = __ldg(w0 + 1);
    q.r1[0] = __ldg(w1); q.r1[1] = __ldg(w1 + 1);
    q.sel = sel;
}
// blend24's (lo, hi) from the words a, b of two adjacent pixels: lo = B0 G0 R0 B1, hi = G1 R1 and two unused bytes
__device__ __forceinline__ void px32_row_taps(unsigned a, unsigned b, unsigned sel, unsigned &lo, unsigned &hi) {
    lo = __byte_perm(a, b, (sel & 0xfffu) | ((4u + (sel & 3u)) << 12));
    hi = __byte_perm(b, 0u, sel >> 4);
}
// The same square of a GRAY8 frame: the four tap bytes, one byte load each (any alignment; nothing else is read).
struct GrayQuad {
    unsigned r0, r1;   // bytes (sx, sx+1) of tap rows sy, sy+1 in bytes 0 and 1
};
__device__ __forceinline__ void gray_quad_load(const uint8_t *p, unsigned pitch, int sx, int sy, GrayQuad &q) {
    const uint8_t *t0 = p + (unsigned)sy * pitch + (unsigned)sx, *t1 = t0 + pitch;
    q.r0 = (unsigned)__ldg(t0) | ((unsigned)__ldg(t0 + 1) << 8);
    q.r1 = (unsigned)__ldg(t1) | ((unsigned)__ldg(t1 + 1) << 8);
}
// the tap square of a format whose taps are converted before the blend (FMT: SRC_NV12, SRC_NV21, SRC_PLANAR, SRC_PACKED422,
// SRC_PX32 or SRC_GRAY8); sel: packed 4:2:2 and RGBA / BGRA only
template <int FMT>
using YuvQuad = typename std::conditional<
    FMT == SRC_PLANAR, PlanarQuad,
    typename std::conditional<FMT == SRC_PACKED422, PackedQuad,
                              typename std::conditional<FMT == SRC_PX32, Px32Quad,
                                                        typename std::conditional<FMT == SRC_GRAY8, GrayQuad, Nv12Quad>::type>::type>::type>::type;
template <int FMT>
__device__ __forceinline__ void yuv_quad_load(const uint8_t *yp, unsigned py, const uint8_t *uvp, const uint8_t *vp, unsigned puv, unsigned sel,
                                              int sx, int sy, YuvQuad<FMT> &q) {
    if constexpr (FMT == SRC_PLANAR) planar_quad_load(yp, py, uvp, vp, puv, sx, sy, q);
    else if constexpr (FMT == SRC_PACKED422) packed_quad_load(yp, py, sel, sx, sy, q);
    else if constexpr (FMT == SRC_PX32) px32_quad_load(yp, py, sel, sx, sy, q);
    else if constexpr (FMT == SRC_GRAY8) gray_quad_load(yp, py, sx, sy, q);
    else nv12_quad_load(yp, py, uvp, puv, sx, sy, q);
}
template <int FMT>
__device__ __forceinline__ void yuv_quad_taps(const YuvQuad<FMT> &q, unsigned &lo0, unsigned &hi0, unsigned &lo1, unsigned &hi1) {
    if constexpr (FMT == SRC_PLANAR) {
        planar_quad_taps(q, lo0, hi0, lo1, hi1);
    } else if constexpr (FMT == SRC_PACKED422) {
        packed_row_taps(q.r0[0], q.r0[1], q.sel, q.odd, lo0, hi0);
        packed_row_taps(q.r1[0], q.r1[1], q.sel, q.odd, lo1, hi1);
    } else if constexpr (FMT == SRC_PX32) {
        px32_row_taps(q.r0[0], q.r0[1], q.sel, lo0, hi0);
        px32_row_taps(q.r1[0], q.r1[1], q.sel, lo1, hi1);
    } else {
        nv12_quad_taps<FMT>(q, lo0, hi0, lo1, hi1);
    }
}
// pixel (xx, yy) of a converted-tap frame inside it (vp: the V plane, planar only; sel: packed 4:2:2 and RGBA / BGRA only)
template <int FMT>
__device__ __forceinline__ unsigned yuv_tap(const uint8_t *yp, int py, const uint8_t *uvp, const uint8_t *vp, int puv, unsigned sel, int xx, int yy) {
    if constexpr (FMT == SRC_PX32)
        return px32_px24(yp + (ptrdiff_t)yy * py, sel, xx);
    else if constexpr (FMT == SRC_GRAY8)
        return (unsigned)__ldg(yp + (ptrdiff_t)yy * py + xx) * 0x010101u;
    else if constexpr (FMT == SRC_PACKED422)
        return packed_px24(yp + (ptrdiff_t)yy * py, sel, xx);
    else if constexpr (FMT == SRC_PLANAR)
        return yuv_bgr24(__ldg(yp + (ptrdiff_t)yy * py + xx), __ldg(uvp + (ptrdiff_t)(yy >> 1) * puv + (xx >> 1)),
                         __ldg(vp + (ptrdiff_t)(yy >> 1) * puv + (xx >> 1)));
    else if constexpr (FMT == SRC_NV21)
        return yuv_bgr24(__ldg(yp + (ptrdiff_t)yy * py + xx), __ldg(uvp + (ptrdiff_t)(yy >> 1) * puv + (xx | 1)),
                         __ldg(uvp + (ptrdiff_t)(yy >> 1) * puv + (xx & ~1)));
    else
        return yuv_bgr24(__ldg(yp + (ptrdiff_t)yy * py + xx), __ldg(uvp + (ptrdiff_t)(yy >> 1) * puv + (xx & ~1)),
                         __ldg(uvp + (ptrdiff_t)(yy >> 1) * puv + (xx | 1)));
}
// border_tap_blend for a converted-tap frame: BORDER_CONSTANT(0) applies to the BGR image, so a tap outside the frame is BGR
// (0,0,0).  Reads only the bytes of the taps inside the frame (RGBA / BGRA: three bytes of a pixel; GRAY8: one).
template <int FMT>
__device__ __forceinline__ unsigned border_tap_blend_yuv(const uint8_t *yp, int py, const uint8_t *uvp, const uint8_t *vp, int puv, unsigned sel,
                                                         int w, int h, int X, int Y) {
    const int sx = max(-32768, min(32767, X >> 5)), sy = max(-32768, min(32767, Y >> 5));   // saturate_cast<short>
    unsigned p[2][2];
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int xx = sx + i, yy = sy + j;
            p[j][i] = xx >= 0 && xx < w && yy >= 0 && yy < h ? yuv_tap<FMT>(yp, py, uvp, vp, puv, sel, xx, yy) : 0u;
        }
    unsigned lo0, hi0, lo1, hi1;
    pack6(p[0][0], p[0][1], lo0, hi0);
    pack6(p[1][0], p[1][1], lo1, hi1);
    return blend24(lo0, hi0, lo1, hi1, X & 31, Y & 31);
}
// The warp kernels read a 4:2:0 frame's interior taps with yuv_quad_load when its planes and pitches are 4-byte aligned
// and its offsets fit 32 bits; the reads run up to 7 bytes past a tap, so the interior also keeps two rows from the bottom
// (the last chroma row is then never read there: the over-read of a chroma row stays in the next row, pitch_uv >= 8).
__device__ __forceinline__ bool nv12_interior_ok(const FrameDev &f) {
    return ((reinterpret_cast<uintptr_t>(f.data) | reinterpret_cast<uintptr_t>(f.uv)) & 3) == 0 && (f.pitch & 3) == 0 && (f.pitch_uv & 3) == 0 &&
           f.pitch >= 8 && f.pitch_uv >= 8 && (size_t)f.h * f.pitch < 0x7fffffffull && (size_t)f.h * f.pitch_uv < 0x7fffffffull;
}
// A packed frame's interior reads stay inside the two tap columns' words (W is even, so a macropixel never straddles the
// end of a row): only the 4-byte alignment and 32-bit offsets are needed.  The same holds for an RGBA / BGRA frame, whose
// interior reads are the four tap pixels' words, and a GRAY8 frame's interior reads are the four tap bytes (no alignment).
template <int FMT>
__device__ __forceinline__ bool yuv_interior_ok(const FrameDev &f) {
    if constexpr (FMT == SRC_PLANAR) return nv12_interior_ok(f) && (f.v_off & 3) == 0;   // the V plane too
    else if constexpr (FMT == SRC_PACKED422 || FMT == SRC_PX32)
        return ((reinterpret_cast<uintptr_t>(f.data) | (uintptr_t)f.pitch) & 3) == 0 && (size_t)f.h * f.pitch < 0x7fffffffull;
    else if constexpr (FMT == SRC_GRAY8) return (size_t)f.h * f.pitch < 0x7fffffffull;
    else return nv12_interior_ok(f);
}

// Stores the 24-bit pixels of a warp's 32 consecutive output pixels.  packed: the 4 pixels of a lane quad (12 bytes) leave
// as three aligned 32-bit words (one shuffle to fetch the neighbour's pixel), i.e. 96 contiguous bytes per warp
// instruction instead of 96 single-byte stores.  Every lane of the warp must call this (shuffle), valid or not.
__device__ __forceinline__ void store_px(uint8_t *band_out, int p, unsigned v, bool valid, bool packed) {
    const unsigned nv = __shfl_down_sync(0xffffffffu, v, 1);
    if (packed) {
        const unsigned q = (unsigned)p & 3u;
        const unsigned lo = __byte_perm(v, nv, 0x4210), hi = nv >> 8;     // 48-bit concat v | nv << 24
        const unsigned word = __funnelshift_r(lo, hi, 8 * q);
        if (valid && q < 3u) reinterpret_cast<unsigned *>(band_out)[3 * (p >> 2) + q] = word;
    } else if (valid) {
        uint8_t *o = band_out + (size_t)p * 3;
        o[0] = (uint8_t)v; o[1] = (uint8_t)(v >> 8); o[2] = (uint8_t)(v >> 16);
    }
}

struct WarpItem {
    const uint8_t *data;
    int w, h, pitch;
    const uint8_t *lo_lim, *hi_lim;
    const uint8_t *uv;   // 4:2:0 only
    int pitch_uv;
    const uint8_t *v;    // planar only
    unsigned sel;        // packed 4:2:2 and RGBA / BGRA only
};

// N rounds of WARP_THREADS consecutive output pixels starting at p0: all 4N aligned 64-bit loads of a thread are issued
// before any is consumed (interior items: no border test anywhere in the band).
template <int FMT, int N>
__device__ __forceinline__ void warp_rounds_interior_yuv(const WarpItem &it, const int2 *__restrict__ dxy, const int2 *__restrict__ xy0,
                                                         int cw, unsigned cw_magic, int p0, int npix, uint8_t *band_out, bool packed) {
    YuvQuad<FMT> q[N];
    int axy[N];
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const int p = min(p0 + u * WARP_THREADS, npix - 1);
        const int row = cw_magic ? (int)__umulhi((unsigned)p, cw_magic) : p, x = p - row * cw;
        const int2 d = dxy[x], r0 = xy0[row];
        const int X = (int)((unsigned)r0.x + (unsigned)d.x) >> 5, Y = (int)((unsigned)r0.y + (unsigned)d.y) >> 5;
        axy[u] = (X & 31) | ((Y & 31) << 8);
        yuv_quad_load<FMT>(it.data, (unsigned)it.pitch, it.uv, it.v, (unsigned)it.pitch_uv, it.sel, X >> 5, Y >> 5, q[u]);
    }
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const int p = p0 + u * WARP_THREADS;
        unsigned v;
        if constexpr (FMT == SRC_GRAY8) {
            v = blend8(q[u].r0, q[u].r1, axy[u] & 31, axy[u] >> 8);
        } else {
            unsigned lo0, hi0, lo1, hi1;
            yuv_quad_taps<FMT>(q[u], lo0, hi0, lo1, hi1);
            v = blend24(lo0, hi0, lo1, hi1, axy[u] & 31, axy[u] >> 8);
        }
        store_px(band_out, p, v, p < npix, packed);
    }
}

// RB: an RGB24 frame (blend24<true>)
template <int N, bool RB = false>
__device__ __forceinline__ void warp_rounds_interior(const WarpItem &it, const int2 *__restrict__ dxy, const int2 *__restrict__ xy0,
                                                     int cw, unsigned cw_magic, int p0, int npix, uint8_t *band_out, bool packed) {
    uint2 q[N][4];
    unsigned off[N];
    int axy[N];
    const unsigned pitch = (unsigned)it.pitch;
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const int p = min(p0 + u * WARP_THREADS, npix - 1);
        const int row = cw_magic ? (int)__umulhi((unsigned)p, cw_magic) : p, x = p - row * cw;
        const int2 d = dxy[x], r0 = xy0[row];
        const int X = (int)((unsigned)r0.x + (unsigned)d.x) >> 5, Y = (int)((unsigned)r0.y + (unsigned)d.y) >> 5;
        axy[u] = (X & 31) | ((Y & 31) << 8);
        off[u] = (unsigned)(Y >> 5) * pitch + (unsigned)(X >> 5) * 3u;
        const uint2 *r0p = reinterpret_cast<const uint2 *>(it.data + (off[u] & ~7u));
        const uint2 *r1p = reinterpret_cast<const uint2 *>(it.data + ((off[u] + pitch) & ~7u));
        q[u][0] = __ldg(r0p); q[u][1] = __ldg(r0p + 1);
        q[u][2] = __ldg(r1p); q[u][3] = __ldg(r1p + 1);
    }
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const int p = p0 + u * WARP_THREADS;
        unsigned lo0, hi0, lo1, hi1;
        extract6(q[u][0], q[u][1], off[u], lo0, hi0);
        extract6(q[u][2], q[u][3], off[u] + pitch, lo1, hi1);
        const unsigned v = blend24<RB>(lo0, hi0, lo1, hi1, axy[u] & 31, axy[u] >> 8);
        store_px(band_out, p, v, p < npix, packed);
    }
}

// one round with per-tap BORDER_CONSTANT tests (items that touch the frame border, unaligned or > 2 GB frames)
template <int FMT>
__device__ __forceinline__ void warp_round_border(const WarpItem &it, const int2 *__restrict__ dxy, const int2 *__restrict__ xy0, int cw,
                                                  unsigned cw_magic, int p0, int npix, uint8_t *band_out, bool packed) {
    const int p = min(p0, npix - 1);
    const int row = cw_magic ? (int)__umulhi((unsigned)p, cw_magic) : p, x = p - row * cw;
    const int2 d = dxy[x], r0 = xy0[row];
    const int X = (int)((unsigned)r0.x + (unsigned)d.x) >> 5, Y = (int)((unsigned)r0.y + (unsigned)d.y) >> 5;
    const unsigned v = FMT != SRC_BGR && FMT != SRC_RGB24
                           ? border_tap_blend_yuv<FMT>(it.data, it.pitch, it.uv, it.v, it.pitch_uv, it.sel, it.w, it.h, X, Y)
                           : border_tap_blend<FMT == SRC_RGB24>(it.data, it.w, it.h, it.pitch, it.lo_lim, it.hi_lim, X, Y);
    store_px(band_out, p0, v, p0 < npix, packed);
}

// Persistent kernel: the grid fills the GPU once; work items (face, band of 16 output rows) are handed out through an
// atomic ticket so big faces (more DRAM per item) do not leave a tail.  The next ticket is fetched while the current
// item is being processed.  Lanes = consecutive output pixels of the band (row-major), so one load instruction's lanes
// share cache lines and one store instruction writes 96 contiguous bytes.
// FMT: the source format of the frames (SrcFmt)
template <int FMT>
__global__ void __launch_bounds__(WARP_THREADS, 4) warp_kernel(WarpArgs a) {
    constexpr bool NV = FMT == SRC_NV12 || FMT == SRC_NV21 || FMT == SRC_PLANAR, PK = FMT == SRC_PACKED422;   // NV: 4:2:0
    constexpr bool RG = FMT == SRC_RGB24, P4 = FMT == SRC_PX32, G1 = FMT == SRC_GRAY8;
    constexpr bool CV = NV || PK || P4 || G1;   // taps converted to BGR before the blend (the others: 3-byte pixels)
    extern __shared__ int2 wsm[];
    int2 *dxy = wsm;             // [cw]  (adelta, bdelta)
    int2 *xy0 = dxy + a.cw;      // [WARP_BAND]  (X0, Y0) per row
    __shared__ int s_item[2];
    const int tid = threadIdx.x;
    pdl_wait();
    const int F = a.count_dev ? min(*a.count_dev, a.F) : a.F;
    const int n_items = F * a.bands;
    if (tid == 0) s_item[0] = atomicAdd(a.ticket, 1);
    __syncthreads();
    for (int par = 0;; par ^= 1) {
        const int item = s_item[par];
        if (item >= n_items) {
            pdl_trigger();   // out of tickets: the next step kernel may take this CTA's place
            break;
        }
        if (tid == 0) s_item[par ^ 1] = atomicAdd(a.ticket, 1);
        const int f = item / a.bands, band_y0 = (item - f * a.bands) * WARP_BAND;
        const int rows = min(WARP_BAND, a.ch - band_y0);
        const int npix = rows * a.cw;
        uint8_t *band_out = a.crops + ((size_t)f * a.ch + band_y0) * a.cw * 3;
        const bool packed = (reinterpret_cast<uintptr_t>(band_out) & 3) == 0 && (npix & 3) == 0;
        const FrameDev fr = a.frames[a.frame_idx ? a.frame_idx[f] : 0];
        if (!a.ok[f]) {   // estimation failed (uniform over the CTA): bbox-crop fallback, or a zero crop where the reference errs
            int rx0 = 0, ry0 = 0;
            const bool valid = warp_fallback_roi(a, f, fr.w, fr.h, &rx0, &ry0);
            if (tid == 0 && band_y0 == 0 && a.mode_out) a.mode_out[f] = valid ? 2 : 0;
            if (valid) {
                const uint8_t *roi = fr.data + (size_t)ry0 * fr.pitch + (size_t)rx0 * 3;
                for (int p = tid; p < npix; p += WARP_THREADS) {
                    const int row = p / a.cw, x = p - row * a.cw;
                    const unsigned v = NV ? resize_pixel24_yuv<FMT>(fr.data, fr.pitch, fr.uv, fr.v_plane(), fr.pitch_uv, rx0, ry0, fr.w - rx0, fr.h - ry0, a.cw,
                                                                    a.ch, x, band_y0 + row)
                                       : PK ? resize_pixel24_packed(fr.data, fr.pitch, (unsigned)fr.v_off, rx0, ry0, fr.w - rx0, fr.h - ry0, a.cw, a.ch, x,
                                                                    band_y0 + row)
                                       : P4 || G1 ? resize_pixel24_rgb<FMT>(fr.data, fr.pitch, (unsigned)fr.v_off, rx0, ry0, fr.w - rx0, fr.h - ry0, a.cw,
                                                                            a.ch, x, band_y0 + row)
                                       : RG ? swap_rb24(resize_pixel24(roi, fr.pitch, fr.w - rx0, fr.h - ry0, a.cw, a.ch, x, band_y0 + row))
                                          : resize_pixel24(roi, fr.pitch, fr.w - rx0, fr.h - ry0, a.cw, a.ch, x, band_y0 + row);
                    band_out[3 * p] = (uint8_t)v; band_out[3 * p + 1] = (uint8_t)(v >> 8); band_out[3 * p + 2] = (uint8_t)(v >> 16);
                }
            } else {
                for (int p = tid; p < npix * 3; p += WARP_THREADS) band_out[p] = 0;
            }
            __syncthreads();
            continue;
        }
        if (tid == 0 && band_y0 == 0 && a.mode_out) a.mode_out[f] = 1;
        const double *iM = a.M12 + (size_t)f * 12 + 6;
        const double i0 = iM[0], i1 = iM[1], i2 = iM[2], i3 = iM[3], i4 = iM[4], i5 = iM[5];
        for (int x = tid; x < a.cw; x += WARP_THREADS)   // saturate_cast<int>(M[0]*x*AB_SCALE), AB_SCALE = 1024
            dxy[x] = make_int2(__double2int_rn(i0 * x * 1024), __double2int_rn(i3 * x * 1024));
        if (tid >= WARP_THREADS - WARP_BAND) {
            const int r = tid - (WARP_THREADS - WARP_BAND), y = band_y0 + min(r, rows - 1);
            xy0[r] = make_int2(__double2int_rn((i1 * y + i2) * 1024) + 16, __double2int_rn((i4 * y + i5) * 1024) + 16);  // + round_delta
        }
        __syncthreads();
        // The map is affine, so the tap coordinates of the band are extremal at its 4 corners: if all 4 corner taps
        // (and their +1 neighbours) are interior, no pixel of the band needs a border test.
        bool interior = CV ? yuv_interior_ok<FMT>(fr)
                           : (reinterpret_cast<uintptr_t>(fr.data) & 7) == 0 && (fr.pitch & 7) == 0 && fr.pitch >= 16 &&
                                 (size_t)fr.h * fr.pitch < 0x7fffffffull;
        const int bottom = NV ? 2 : CV ? 0 : 1;   // rows kept from the bottom: the loads over-read past the last tap row
        {
            const int xs[2] = {0, a.cw - 1}, ys[2] = {0, rows - 1};
#pragma unroll
            for (int cy = 0; cy < 2; ++cy)
#pragma unroll
                for (int cx = 0; cx < 2; ++cx) {
                    const long long Xl = (long long)xy0[ys[cy]].x + dxy[xs[cx]].x, Yl = (long long)xy0[ys[cy]].y + dxy[xs[cx]].y;
                    const long long sx = Xl >> 10, sy = Yl >> 10;
                    interior = interior && sx >= 0 && sx + 1 < fr.w && sy >= 0 && sy + 1 < fr.h - bottom;  // over-read stays in the frame
                }
        }
        WarpItem it;
        it.data = fr.data; it.w = fr.w; it.h = fr.h; it.pitch = fr.pitch;
        it.lo_lim = fr.data;
        it.hi_lim = fr.data + (size_t)(fr.h - 1) * fr.pitch + (size_t)fr.w * 3;  // end of valid pixel bytes
        it.uv = fr.uv; it.pitch_uv = fr.pitch_uv;
        if constexpr (FMT == SRC_PLANAR) it.v = fr.v_plane();
        it.sel = PK || P4 ? (unsigned)fr.v_off : 0u;
        int p0 = tid;
        if (CV && interior) {
            for (int rounds = (npix + WARP_THREADS - 1) / WARP_THREADS; rounds > 0; rounds -= 2, p0 += 2 * WARP_THREADS) {
                if (rounds >= 2) warp_rounds_interior_yuv<FMT, 2>(it, dxy, xy0, a.cw, a.cw_magic, p0, npix, band_out, packed);
                else warp_rounds_interior_yuv<FMT, 1>(it, dxy, xy0, a.cw, a.cw_magic, p0, npix, band_out, packed);
            }
        } else if (interior) {
            int rounds = (npix + WARP_THREADS - 1) / WARP_THREADS;
            while (rounds > 0) {
                if (rounds >= 4) { warp_rounds_interior<4, RG>(it, dxy, xy0, a.cw, a.cw_magic, p0, npix, band_out, packed); rounds -= 4; p0 += 4 * WARP_THREADS; }
                else if (rounds == 3) { warp_rounds_interior<3, RG>(it, dxy, xy0, a.cw, a.cw_magic, p0, npix, band_out, packed); rounds = 0; }
                else if (rounds == 2) { warp_rounds_interior<2, RG>(it, dxy, xy0, a.cw, a.cw_magic, p0, npix, band_out, packed); rounds = 0; }
                else { warp_rounds_interior<1, RG>(it, dxy, xy0, a.cw, a.cw_magic, p0, npix, band_out, packed); rounds = 0; }
            }
        } else {
            for (; p0 - tid < npix; p0 += WARP_THREADS) warp_round_border<FMT>(it, dxy, xy0, a.cw, a.cw_magic, p0, npix, band_out, packed);
        }
        __syncthreads();  // tables and s_item[par] are free again
    }
    if (tid == 0) {  // the last CTA to leave re-arms the ticket for the next launch on this ctx
        __threadfence();
        if (atomicAdd(a.ticket + 1, 1) == (int)gridDim.x - 1) {
            a.ticket[0] = 0;
            a.ticket[1] = 0;
            __threadfence();
        }
    }
}

// ---- fixed-size fast path (the reference's 112x112 ArcFace crop, config.rs:45) --------------------------------------
// Same persistent/ticket structure; a CTA is 2 output rows x CW columns, so a thread keeps ONE column for the whole item:
// its (adelta, bdelta) live in registers, no index division, and the packed-store word address advances by a constant.
// An item is IR output rows (IR/2 rounds per thread); the per-row (X0, Y0) table is double-buffered so one barrier per
// item is enough, and that barrier also carries the band's interior vote (4 threads evaluate the 4 corners).
#ifdef WARP_LDCG
#define WARP_LD(p) __ldcg(p)
#else
#define WARP_LD(p) __ldg(p)
#endif
// pack_sel: the byte permute that cuts this lane's word out of (its pixel, the next lane's pixel): lanes 0..2 of a quad store
// bytes 0-3, 4-7, 8-11 of the quad's 12.  RB: an RGB24 frame (blend24_scaled<true>).
template <int CW, int N, bool RB = false>
__device__ __forceinline__ void fixed_rounds_interior(const uint8_t *__restrict__ data, unsigned pitch, int2 d, const int2 *__restrict__ xy,
                                                      unsigned *__restrict__ outw, bool store, unsigned pack_sel) {
    uint2 q[N][4];
    unsigned off[N];
    int axy[N];
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const int2 r0 = xy[2 * u];
        const int X = (int)((unsigned)r0.x + (unsigned)d.x) >> 5, Y = (int)((unsigned)r0.y + (unsigned)d.y) >> 5;
        axy[u] = (X & 31) | ((Y & 31) << 14);   // ax | ay << 6 << 8
        off[u] = (unsigned)(Y >> 5) * pitch + (unsigned)(X >> 5) * 3u;
        const uint2 *r0p = reinterpret_cast<const uint2 *>(data + (off[u] & ~7u));
        const uint2 *r1p = reinterpret_cast<const uint2 *>(reinterpret_cast<const uint8_t *>(r0p) + pitch);   // pitch % 8 == 0
        q[u][0] = WARP_LD(r0p); q[u][1] = WARP_LD(r0p + 1);
        q[u][2] = WARP_LD(r1p); q[u][3] = WARP_LD(r1p + 1);
    }
#pragma unroll
    for (int u = 0; u < N; ++u) {
        // both rows share the byte phase (pitch % 8 == 0)
        const bool up = (off[u] & 4u) != 0;
        const unsigned sft = (off[u] & 3u) * 8;
        const unsigned a0 = up ? q[u][0].y : q[u][0].x, b0 = up ? q[u][1].x : q[u][0].y, c0 = up ? q[u][1].y : q[u][1].x;
        const unsigned a1 = up ? q[u][2].y : q[u][2].x, b1 = up ? q[u][3].x : q[u][2].y, c1 = up ? q[u][3].y : q[u][3].x;
        const unsigned v = blend24_scaled<RB>(__funnelshift_r(a0, b0, sft), __funnelshift_r(b0, c0, sft), __funnelshift_r(a1, b1, sft),
                                          __funnelshift_r(b1, c1, sft), axy[u] & 31, axy[u] >> 8);
        const unsigned nv = __shfl_down_sync(0xffffffffu, v, 1);
        if (store) outw[u * (2 * CW * 3 / 4)] = __byte_perm(v, nv, pack_sel);
    }
}

template <int CW, int N, int FMT>
__device__ __forceinline__ void fixed_rounds_interior_yuv(const uint8_t *__restrict__ yp, unsigned py, const uint8_t *__restrict__ uvp,
                                                          const uint8_t *__restrict__ vp, unsigned puv, unsigned sel, int2 d,
                                                          const int2 *__restrict__ xy, unsigned *__restrict__ outw, bool store, unsigned pack_sel) {
    YuvQuad<FMT> q[N];
    int axy[N];
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const int2 r0 = xy[2 * u];
        const int X = (int)((unsigned)r0.x + (unsigned)d.x) >> 5, Y = (int)((unsigned)r0.y + (unsigned)d.y) >> 5;
        axy[u] = (X & 31) | ((Y & 31) << 14);   // ax | ay << 6 << 8
        yuv_quad_load<FMT>(yp, py, uvp, vp, puv, sel, X >> 5, Y >> 5, q[u]);
    }
#pragma unroll
    for (int u = 0; u < N; ++u) {
        unsigned v;
        if constexpr (FMT == SRC_GRAY8) {
            v = blend8_scaled(q[u].r0, q[u].r1, axy[u] & 31, axy[u] >> 8);
        } else {
            unsigned lo0, hi0, lo1, hi1;
            yuv_quad_taps<FMT>(q[u], lo0, hi0, lo1, hi1);
            v = blend24_scaled(lo0, hi0, lo1, hi1, axy[u] & 31, axy[u] >> 8);
        }
        const unsigned nv = __shfl_down_sync(0xffffffffu, v, 1);
        if (store) outw[u * (2 * CW * 3 / 4)] = __byte_perm(v, nv, pack_sel);
    }
}

// FMT: the source format of the frames (SrcFmt)
template <int CW, int CH, int IR, int UN, int FMT>
__global__ void __launch_bounds__(2 * CW) warp_fixed_kernel(WarpArgs a) {
    constexpr bool NV = FMT == SRC_NV12 || FMT == SRC_NV21 || FMT == SRC_PLANAR, PK = FMT == SRC_PACKED422;   // NV: 4:2:0
    constexpr bool RG = FMT == SRC_RGB24, P4 = FMT == SRC_PX32, G1 = FMT == SRC_GRAY8;
    constexpr bool CV = NV || PK || P4 || G1;   // taps converted to BGR before the blend (the others: 3-byte pixels)
    constexpr int T = 2 * CW, ITEMS = CH / IR, ROUNDS = IR / 2;
    static_assert(CH % IR == 0 && IR % 2 == 0 && T % 32 == 0 && (2 * CW * 3) % 4 == 0 && (IR * CW * 3) % 4 == 0, "fixed warp geometry");
    __shared__ int2 xy0[2][IR];
    __shared__ int s_item[2];
    const int tid = threadIdx.x;
    const int r = tid / CW, x = tid - r * CW;
    pdl_wait();
    const int F = a.count_dev ? min(*a.count_dev, a.F) : a.F;
    const int n_items = F * ITEMS;
    long long t_entry = 0, t_prev = 0, t_sum = 0;
    int n_done = 0;
    if (a.dbg && tid == 0) t_entry = warp_now();
    if (tid == 0) s_item[0] = atomicAdd(a.ticket, 1);
    __syncthreads();
    if (a.dbg && tid == 0) { t_prev = warp_now(); a.dbg[blockIdx.x * 8 + 1] = t_prev; }
    for (int par = 0;; par ^= 1) {
        const int item = s_item[par];
        if (a.dbg && tid == 0 && par == 1 && n_done == 1) a.dbg[blockIdx.x * 8 + 2] = warp_now();
        if (a.dbg && tid == 0) { const long long t = warp_now(); if (n_done) t_sum += t - t_prev; t_prev = t; ++n_done; }
        if (item >= n_items) {
            pdl_trigger();   // out of tickets: the next step kernel may take this CTA's place
            break;
        }
        if (tid == 0) s_item[par ^ 1] = atomicAdd(a.ticket, 1);
        const int f = item / ITEMS, y0 = (item - f * ITEMS) * IR;
        uint8_t *band_out = a.crops + ((size_t)f * CH + y0) * CW * 3;
        const bool okf = a.ok[f] != 0;
        const FrameDev *frp = a.frames + (a.frame_idx ? a.frame_idx[f] : 0);
        const uint8_t *data = frp->data;
        const int fw = frp->w, fh = frp->h, pitch = frp->pitch;
        const uint8_t *uvp = NV ? frp->uv : nullptr;
        const int pitch_uv = NV ? frp->pitch_uv : 0;
        const uint8_t *vp = nullptr;   // planar only
        if constexpr (FMT == SRC_PLANAR) vp = frp->v_plane();
        const unsigned sel = PK || P4 ? (unsigned)frp->v_off : 0u;
        int2 d = make_int2(0, 0);
        bool vote = true;
        if (okf) {
            const double *iM = a.M12 + (size_t)f * 12 + 6;
            const double i0 = iM[0], i3 = iM[3];
            d = make_int2(__double2int_rn(i0 * x * 1024), __double2int_rn(i3 * x * 1024));   // adelta[x], bdelta[x]
            if (tid < IR || tid >= T - 4) {
                const double i1 = iM[1], i2 = iM[2], i4 = iM[4], i5 = iM[5];
                if (tid < IR) {
                    const int y = y0 + tid;
                    xy0[par][tid] = make_int2(__double2int_rn((i1 * y + i2) * 1024) + 16, __double2int_rn((i4 * y + i5) * 1024) + 16);
                } else {   // one corner of the item each: the affine map's tap coordinates are extremal there
                    const int c = tid - (T - 4), cx = (c & 1) ? CW - 1 : 0, y = y0 + ((c & 2) ? IR - 1 : 0);
                    const long long Xl = (long long)(__double2int_rn((i1 * y + i2) * 1024) + 16) + __double2int_rn(i0 * cx * 1024);
                    const long long Yl = (long long)(__double2int_rn((i4 * y + i5) * 1024) + 16) + __double2int_rn(i3 * cx * 1024);
                    const long long sx = Xl >> 10, sy = Yl >> 10;
                    vote = sx >= 0 && sx + 1 < fw && sy >= 0 && sy + 1 < fh - (NV ? 2 : CV ? 0 : 1);   // the over-read stays in the frame
                }
            }
        }
        const bool interior = __syncthreads_and(vote) && (CV ? yuv_interior_ok<FMT>(*frp)
                                                             : (reinterpret_cast<uintptr_t>(data) & 7) == 0 && (pitch & 7) == 0 && pitch >= 16 &&
                                                                   (size_t)fh * pitch < 0x7fffffffull);
        const bool store = (tid & 3) != 3;
        unsigned *outw = reinterpret_cast<unsigned *>(band_out) + 3 * (tid >> 2) + (tid & 3);
        if (!okf) {   // estimation failed: bbox-crop fallback (face_alignment.rs:64-116), or a zero crop where the reference errs
            int rx0 = 0, ry0 = 0;
            const bool valid = warp_fallback_roi(a, f, fw, fh, &rx0, &ry0);
            if (tid == 0 && y0 == 0 && a.mode_out) a.mode_out[f] = valid ? 2 : 0;
            if (valid) {
                const uint8_t *roi = data + (size_t)ry0 * pitch + (size_t)rx0 * 3;
                for (int u = 0; u < ROUNDS; ++u) {
                    const unsigned v = NV ? resize_pixel24_yuv<FMT>(data, pitch, uvp, vp, pitch_uv, rx0, ry0, fw - rx0, fh - ry0, CW, CH, x, y0 + r + 2 * u)
                                       : PK ? resize_pixel24_packed(data, pitch, sel, rx0, ry0, fw - rx0, fh - ry0, CW, CH, x, y0 + r + 2 * u)
                                       : P4 || G1 ? resize_pixel24_rgb<FMT>(data, pitch, sel, rx0, ry0, fw - rx0, fh - ry0, CW, CH, x, y0 + r + 2 * u)
                                       : RG ? swap_rb24(resize_pixel24(roi, pitch, fw - rx0, fh - ry0, CW, CH, x, y0 + r + 2 * u))
                                          : resize_pixel24(roi, pitch, fw - rx0, fh - ry0, CW, CH, x, y0 + r + 2 * u);
                    const unsigned nv = __shfl_down_sync(0xffffffffu, v, 1);
                    const unsigned word = __funnelshift_r(__byte_perm(v, nv, 0x4210), nv >> 8, 8 * (tid & 3u));
                    if (store) outw[u * (T * 3 / 4)] = word;
                }
            } else {
                for (int p = tid; p < IR * CW * 3 / 4; p += T) reinterpret_cast<unsigned *>(band_out)[p] = 0u;
            }
            continue;
        }
        if (tid == 0 && y0 == 0 && a.mode_out) a.mode_out[f] = 1;
        const int2 *xy = &xy0[par][r];
        if (interior) {
            const unsigned pack_sel = (tid & 3) == 0 ? 0x4210u : ((tid & 3) == 1 ? 0x5421u : 0x6542u);
            int u = 0;
            constexpr int REM = ROUNDS % UN;
            if (CV) {
#pragma unroll 1
                for (; u + UN <= ROUNDS; u += UN)
                    fixed_rounds_interior_yuv<CW, UN, FMT>(data, (unsigned)pitch, uvp, vp, (unsigned)pitch_uv, sel, d, xy + 2 * u,
                                                           outw + u * (T * 3 / 4), store, pack_sel);
                if (REM) fixed_rounds_interior_yuv<CW, REM ? REM : 1, FMT>(data, (unsigned)pitch, uvp, vp, (unsigned)pitch_uv, sel, d,
                                                                           xy + 2 * (ROUNDS - REM), outw + (ROUNDS - REM) * (T * 3 / 4), store, pack_sel);
            } else {
#pragma unroll 1
                for (; u + UN <= ROUNDS; u += UN)
                    fixed_rounds_interior<CW, UN, RG>(data, (unsigned)pitch, d, xy + 2 * u, outw + u * (T * 3 / 4), store, pack_sel);
                if (REM) fixed_rounds_interior<CW, REM ? REM : 1, RG>(data, (unsigned)pitch, d, xy + 2 * (ROUNDS - REM), outw + (ROUNDS - REM) * (T * 3 / 4), store, pack_sel);
            }
        } else {
            const uint8_t *lo_lim = data, *hi_lim = data + (size_t)(fh - 1) * pitch + (size_t)fw * 3;  // end of valid pixel bytes
            for (int u = 0; u < ROUNDS; ++u) {
                const int2 r0 = xy[2 * u];
                const int X = (int)((unsigned)r0.x + (unsigned)d.x) >> 5, Y = (int)((unsigned)r0.y + (unsigned)d.y) >> 5;
                const unsigned v = CV ? border_tap_blend_yuv<FMT>(data, pitch, uvp, vp, pitch_uv, sel, fw, fh, X, Y)
                                      : border_tap_blend<RG>(data, fw, fh, pitch, lo_lim, hi_lim, X, Y);
                const unsigned nv = __shfl_down_sync(0xffffffffu, v, 1);
                const unsigned word = __funnelshift_r(__byte_perm(v, nv, 0x4210), nv >> 8, 8 * (tid & 3u));
                if (store) outw[u * (T * 3 / 4)] = word;
            }
        }
    }
    if (a.dbg && tid == 0) {
        a.dbg[blockIdx.x * 8 + 0] = t_entry;
        a.dbg[blockIdx.x * 8 + 3] = warp_now();
        a.dbg[blockIdx.x * 8 + 4] = n_done - 1;
        a.dbg[blockIdx.x * 8 + 5] = t_sum;
    }
    if (tid == 0) {  // the last CTA to leave re-arms the ticket for the next launch on this ctx
        __threadfence();
        if (atomicAdd(a.ticket + 1, 1) == (int)gridDim.x - 1) {
            a.ticket[0] = 0;
            a.ticket[1] = 0;
            __threadfence();
        }
    }
}

static int lmeds_niters(double p, double ep, int modelPoints, int maxIters) {  // RANSACUpdateNumIters
    p = std::max(p, 0.); p = std::min(p, 1.);
    ep = std::max(ep, 0.); ep = std::min(ep, 1.);
    double num = std::max(1. - p, DBL_MIN);
    double denom = 1. - std::pow(1. - ep, modelPoints);
    if (denom < DBL_MIN) return 0;
    num = std::log(num);
    denom = std::log(denom);
    return denom >= 0 || -num >= maxIters * (-denom) ? maxIters : (int)std::lrint(num / denom);
}

int make_est_const(const fd_ctx *ctx, EstConst *out) {
    for (int i = 0; i < 10; ++i) out->tmpl[i] = (&ctx->cfg.template_landmarks[0][0])[i];
    out->niters = std::max(lmeds_niters(0.99, 0.45, 2, 2000), 3);
    if (out->niters > EST_LANES) return fail(FD_ERR_INVALID, "estimate: LMedS iteration count exceeds the lane group");
    // cv::RNG(-1): state = (uint32)state * 4164903690 + (state >> 32); uniform(0,n) = next() % n
    unsigned long long st = 0xFFFFFFFFFFFFFFFFull;
    auto next = [&]() { st = (unsigned long long)(unsigned)st * 4164903690ull + (unsigned)(st >> 32); return (unsigned)st; };
    for (int it = 0; it < 16; ++it) {
        int i0 = (int)(next() % 5u), i1;
        do { i1 = (int)(next() % 5u); } while (i1 == i0);
        out->pair0[it] = (int8_t)i0;
        out->pair1[it] = (int8_t)i1;
    }
    return FD_OK;
}

// zero-initialised work tickets of the persistent kernels (each launch leaves them at zero again)
int ticket_buffer(fd_ctx *ctx) {
    if (ctx->tickets.p) return FD_OK;
    FD_TRY(ctx->tickets.reserve(sizeof(int) * 16));
    FD_CUDA(cudaMemsetAsync(ctx->tickets.p, 0, sizeof(int) * 16, ctx->stream));
    return FD_OK;
}

// from_dev (F,10); to_dev (F,10) or nullptr (ctx template).  count_dev optional device-side face count (<= F_cap).
int estimate_launch(fd_ctx *ctx, const float *from_dev, const float *to_dev, const int *count_dev, int F_cap,
                    double *M12_dev, double *M_out_dev, uint8_t *ok_dev, uint8_t *ok_out_dev) {
    if (F_cap <= 0) return FD_OK;
    EstArgs a;
    a.from = from_dev;
    a.to = to_dev;
    a.count_dev = count_dev;
    a.F = F_cap;
    FD_TRY(make_est_const(ctx, &a.ec));
    a.M12 = M12_dev;
    a.M_out = M_out_dev;
    a.ok = ok_dev;
    a.ok_out = ok_out_dev;
    estimate_kernel<<<(F_cap * EST_LANES + 127) / 128, 128, 0, ctx->stream>>>(a);
    FD_LAUNCH_CHECK_NAMED(ctx, "estimate_kernel");
    return FD_OK;
}

int invert_launch(fd_ctx *ctx, const double *M_dev, int F, double *M12_dev, uint8_t *ok_dev) {
    if (F <= 0) return FD_OK;
    invert_kernel<<<(F + 127) / 128, 128, 0, ctx->stream>>>(M_dev, F, M12_dev, ok_dev);
    FD_LAUNCH_CHECK(ctx);
    return FD_OK;
}

// Planar frames keep 2 rounds in flight (12 words a round instead of NV12's 8): with 4 the kernel needs 99 registers and
// fits 2 CTAs per SM instead of 4.
template <int IR>
static void (*fixed_kernel_for(int fmt))(WarpArgs) {
    return fmt == SRC_NV12 ? warp_fixed_kernel<112, 112, IR, 4, SRC_NV12>
           : fmt == SRC_NV21 ? warp_fixed_kernel<112, 112, IR, 4, SRC_NV21>
           : fmt == SRC_PLANAR ? warp_fixed_kernel<112, 112, IR, 2, SRC_PLANAR>
           : fmt == SRC_PACKED422 ? warp_fixed_kernel<112, 112, IR, 4, SRC_PACKED422>
           : fmt == SRC_RGB24 ? warp_fixed_kernel<112, 112, IR, 4, SRC_RGB24>
           : fmt == SRC_PX32 ? warp_fixed_kernel<112, 112, IR, 4, SRC_PX32>
           : fmt == SRC_GRAY8 ? warp_fixed_kernel<112, 112, IR, 4, SRC_GRAY8> : warp_fixed_kernel<112, 112, IR, 4, SRC_BGR>;
}
// launch names by source format (I420 and YV12 share the planar instantiations, YUY2, UYVY and YVYU the packed ones, RGBA
// and BGRA the 4-byte ones)
static const char *const FIXED_NAMES[SRC_FMT_COUNT] = {"warp_fixed_kernel",       "warp_fixed_kernel_nv12",   "warp_fixed_kernel_nv21",
                                                       "warp_fixed_kernel_i420",  "warp_fixed_kernel_yuv422", "warp_fixed_kernel_rgb24",
                                                       "warp_fixed_kernel_rgba",  "warp_fixed_kernel_gray8"};
static const char *const WARP_NAMES[SRC_FMT_COUNT] = {"warp_kernel",      "warp_kernel_nv12",   "warp_kernel_nv21", "warp_kernel_i420",
                                                      "warp_kernel_yuv422", "warp_kernel_rgb24", "warp_kernel_rgba", "warp_kernel_gray8"};

// fmt: the source format of frames_dev (SrcFmt)
int warp_launch(fd_ctx *ctx, const FrameDev *frames_dev, const int32_t *frame_idx_dev, const double *M12_dev,
                const uint8_t *ok_dev, const int *count_dev, int F_cap, uint8_t *crops_dev, int cw, int ch, const WarpFallback &fb,
                int fmt) {
    if (F_cap <= 0) return FD_OK;
    WarpArgs a;
    a.bbox = fb.bbox;
    a.bbox_stride = fb.bbox_stride;
    a.sel = fb.sel;
    a.mode_out = fb.mode_out;
    a.frames = frames_dev;
    a.frame_idx = frame_idx_dev;
    a.M12 = M12_dev;
    a.ok = ok_dev;
    a.count_dev = count_dev;
    a.F = F_cap;
    a.crops = crops_dev;
    a.cw = cw;
    a.ch = ch;
    a.bands = (ch + WARP_BAND - 1) / WARP_BAND;
    a.cw_magic = cw > 1 ? (unsigned)((1ull << 32) / (unsigned)cw + 1ull) : 0u;
    FD_TRY(ticket_buffer(ctx));
    a.ticket = ctx->tickets.as<int>();
    a.dbg = nullptr;
    static const bool dbg_on = getenv("FD_WARP_DBG") != nullptr;
    static long long *dbg_dev = nullptr;
    if (dbg_on) {
        if (!dbg_dev) FD_CUDA(cudaMalloc(&dbg_dev, sizeof(long long) * 8 * 4096));
        FD_CUDA(cudaMemsetAsync(dbg_dev, 0, sizeof(long long) * 8 * 4096, ctx->stream));
        a.dbg = dbg_dev;
    }
    if (cw == 112 && ch == 112 && (reinterpret_cast<uintptr_t>(crops_dev) & 3) == 0) {
        // 14-row items (8 per face, 7 rounds per thread as 4 + 3): small enough that the last items of a launch leave
        // no long tail (28 rows: +10 % time), large enough to amortise the per-item setup (8 rows: same time, 4: +8 %).
        // 4 rounds in flight per thread (72 registers, 4 CTAs/SM); 2, 3 measure the same, 7 (104 registers) is 35 % slower.
        static const int ir_env = getenv("FD_WARP_IR") ? atoi(getenv("FD_WARP_IR")) : 14;   // A/B: 16-row items (7 per face, 8 rounds as 4 + 4): 82.0 vs 78.8 us on C2
        const int IR = ir_env == 16 ? 16 : 14;
        void (*kern)(WarpArgs) = IR == 16 ? fixed_kernel_for<16>(fmt) : fixed_kernel_for<14>(fmt);
        static int per_sm_fixed[SRC_FMT_COUNT] = {};
        int &per_sm_k = per_sm_fixed[fmt];
        if (!per_sm_k) FD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_k, kern, 224, 0));
        const long long items = (long long)F_cap * (112 / IR);
        const int grid = (int)std::min<long long>(items, (long long)ctx->num_sms * std::max(per_sm_k, 1));
        FD_TRY(launch_pdl(ctx, kern, dim3(grid), dim3(224), 0, a));
        FD_LAUNCH_CHECK_NAMED(ctx, FIXED_NAMES[fmt]);
        if (dbg_on) {   // in-kernel timeline (globaltimer): where a launch's time goes beyond the per-item work
            std::vector<long long> h(8 * (size_t)std::min(grid, 4096));
            cudaStreamSynchronize(ctx->stream);
            cudaMemcpy(h.data(), dbg_dev, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost);
            long long t0 = h[0], t1 = h[3], first_sum = 0, item_sum = 0, items_n = 0, entry_max = h[0], tick_sum = 0;
            const int n = (int)h.size() / 8;
            for (int b = 0; b < n; ++b) {
                t0 = std::min(t0, h[8 * b]); t1 = std::max(t1, h[8 * b + 3]); entry_max = std::max(entry_max, h[8 * b]);
                tick_sum += h[8 * b + 1] - h[8 * b];
                if (h[8 * b + 2]) first_sum += h[8 * b + 2] - h[8 * b + 1];
                item_sum += h[8 * b + 5]; items_n += h[8 * b + 4];
            }
            fprintf(stderr, "[warp dbg] F=%d grid=%d span %.2f us; CTA entry spread %.2f us; first ticket %.2f us; first item %.2f us; mean item %.2f us over %lld items\n",
                    F_cap, grid, (t1 - t0) * 1e-3, (entry_max - t0) * 1e-3, tick_sum * 1e-3 / n, first_sum * 1e-3 / n, items_n ? item_sum * 1e-3 / items_n : 0.0, items_n);
        }
        return FD_OK;
    }
    const size_t smem = sizeof(int2) * ((size_t)cw + WARP_BAND);
    int per_sm = 0;
    void (*kern)(WarpArgs) = fmt == SRC_NV12 ? warp_kernel<SRC_NV12>
                             : fmt == SRC_NV21 ? warp_kernel<SRC_NV21>
                             : fmt == SRC_PLANAR ? warp_kernel<SRC_PLANAR>
                             : fmt == SRC_PACKED422 ? warp_kernel<SRC_PACKED422>
                             : fmt == SRC_RGB24 ? warp_kernel<SRC_RGB24>
                             : fmt == SRC_PX32 ? warp_kernel<SRC_PX32>
                             : fmt == SRC_GRAY8 ? warp_kernel<SRC_GRAY8> : warp_kernel<SRC_BGR>;
    FD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARP_THREADS, smem));
    const long long items = (long long)F_cap * a.bands;
    const int grid = (int)std::min<long long>(items, (long long)ctx->num_sms * std::max(per_sm, 1));
    FD_TRY(launch_pdl(ctx, kern, dim3(grid), dim3(WARP_THREADS), smem, a));
    FD_LAUNCH_CHECK_NAMED(ctx, WARP_NAMES[fmt]);
    return FD_OK;
}

}  // namespace fd
