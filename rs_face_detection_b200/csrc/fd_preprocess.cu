// fd_preprocess.cu — letterbox resize + zero pad + BGR->RGB + normalise + HWC->NCHW fp32, one launch per batch.
//
// Replaces RetinaFaceDetection::_preprocess (face_detection.rs:131-198: cv::resize INTER_LINEAR into the top-left
// corner of a zero canvas) and the per-pixel tensor loop (face_detection.rs:220-230).  The resize reproduces OpenCV's
// 8UC3 fixed-point scheme bit for bit (imgproc/resize.cpp: 11-bit coefficients, int32 horizontal pass,
// ((b*(T>>4))>>16 ... +2)>>2 vertical pass); a float bilinear would be off by up to 6 grey levels.
//
// Data movement: a CTA owns a band of output rows of one image.  The (one or two) source rows an output row needs are
// staged into shared memory with 128-bit coalesced loads — the second row is skipped when its vertical weight is zero
// (exact integer down-scales, e.g. 1080p -> 640x360 reads one source row in three) — the taps are then gathered from
// shared memory, and each thread writes 4 consecutive pixels of the three channel planes as 128-bit stores.
// Normalisation is a 3x256-entry table of the reference's exact (p/scale - mean)/std expression (two IEEE divides per
// entry instead of per pixel).
#include <algorithm>
#include "fd_internal.cuh"
#include "fd_resize.cuh"

namespace fd {

constexpr int PRE_ROWS = 8;  // output rows per CTA

struct PreArgs {
    const FrameDev *frames;
    float *out;
    int out_w, out_h;
    float pixel_scale, means[3], stds[3];
    int row_buf_bytes;  // per staged row (multiple of 16, >= max(w*3)+32)
    int vec_store;      // out_w % 4 == 0
};

// stage nbytes of a source row into shared memory keeping the source's 16-byte phase; returns the pointer to byte 0
__device__ __forceinline__ const uint8_t *stage_row(uint8_t *buf, const uint8_t *__restrict__ src, int nbytes) {
    const int mis = (int)(reinterpret_cast<uintptr_t>(src) & 15);
    uint8_t *dst = buf + mis;
    const int head = mis ? min(nbytes, 16 - mis) : 0;
    for (int i = threadIdx.x; i < head; i += blockDim.x) dst[i] = __ldg(src + i);
    const int nvec = (nbytes - head) >> 4;
    const int4 *s4 = reinterpret_cast<const int4 *>(src + head);
    int4 *d4 = reinterpret_cast<int4 *>(dst + head);
    for (int v = threadIdx.x; v < nvec; v += blockDim.x) d4[v] = __ldg(s4 + v);
    const int done = head + (nvec << 4);
    for (int i = done + threadIdx.x; i < nbytes; i += blockDim.x) dst[i] = __ldg(src + i);
    return dst;
}

// FMT: the source format (SrcFmt).  A YUV frame's taps are converted to BGR (yuv_bgr24) before the resize arithmetic.  A
// 4:2:0 frame's staged rows are the Y rows and the chroma row(s) of the taps; a planar chroma row is staged as its U half and,
// row_buf_bytes / 2 further, its V half.  A packed 4:2:2 frame stages its tap rows (2w bytes) as a BGR frame does, and so
// do the RGB-family frames (RGB24 3w, RGBA / BGRA 4w, GRAY8 w bytes).  Rows staged here keep the source's 16-byte phase, so
// a 4-byte pixel is read as three bytes at any frame alignment.
template <int FMT>
__global__ void preprocess_kernel(PreArgs a) {
    constexpr bool NV = FMT == SRC_NV12 || FMT == SRC_NV21 || FMT == SRC_PLANAR, PL = FMT == SRC_PLANAR;   // NV: 4:2:0
    constexpr bool PK = FMT == SRC_PACKED422;
    constexpr bool RG = FMT == SRC_RGB24, P4 = FMT == SRC_PX32, G1 = FMT == SRC_GRAY8;
    extern __shared__ __align__(16) unsigned char smem[];
    const int ow = a.out_w;
    float *lut = reinterpret_cast<float *>(smem);                  // [3][256], indexed by BGR channel
    int *xo0 = reinterpret_cast<int *>(lut + 768);                 // [ow]
    int *xo1 = xo0 + ow;                                           // [ow]
    short *xa0 = reinterpret_cast<short *>(xo1 + ow);              // [ow]
    short *xa1 = xa0 + ow;                                         // [ow]
    size_t tab_bytes = 768 * 4 + (size_t)ow * 12;
    tab_bytes = (tab_bytes + 15) & ~(size_t)15;
    uint8_t *rowbuf0 = smem + tab_bytes;
    uint8_t *rowbuf1 = rowbuf0 + a.row_buf_bytes;
    uint8_t *rowbuf2 = rowbuf1 + a.row_buf_bytes, *rowbuf3 = rowbuf2 + a.row_buf_bytes;   // NV: chroma rows
    const int half = a.row_buf_bytes >> 1;                                                // PL: V half of a chroma row

    for (int i = threadIdx.x; i < 768; i += blockDim.x) {
        int c = i >> 8, v = i & 255;
        lut[i] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)v, a.pixel_scale), a.means[c]), a.stds[c]);  // face_detection.rs:227
    }
    pdl_wait();   // (no early trigger: the detect kernel's CTAs would take SMs this grid still needs)
    const FrameDev f = a.frames[blockIdx.y];
    for (int x = threadIdx.x; x < f.new_w; x += blockDim.x) {
        x_taps(x, f.scale_x, f.w, &xo0[x], &xo1[x], &xa0[x], &xa1[x]);
        if (NV || PK || P4 || G1) { xo0[x] /= 3; xo1[x] /= 3; }   // pixel, not byte, offsets
    }
    __syncthreads();
    const float pad_r = lut[2 * 256], pad_g = lut[1 * 256], pad_b = lut[0];
    const size_t plane = (size_t)a.out_h * ow;
    float *out_img = a.out + (size_t)blockIdx.y * 3 * plane;
    const int ngroups = (ow + 3) >> 2;
    const int row_begin = blockIdx.x * PRE_ROWS;
    const int row_end = min(row_begin + PRE_ROWS, a.out_h);
    const int src_row_bytes = NV || G1 ? f.w : PK ? 2 * f.w : P4 ? 4 * f.w : f.w * 3;
    const unsigned sel = PK || P4 ? (unsigned)f.v_off : 0u;

    for (int dy = row_begin; dy < row_end; ++dy) {
        float *o_r = out_img + (size_t)dy * ow;  // plane 0 = R (BGR channel 2), face_detection.rs:226-227
        float *o_g = o_r + plane;
        float *o_b = o_g + plane;
        const bool content = dy < f.new_h;
        const uint8_t *r0 = nullptr, *r1 = nullptr, *c0 = nullptr, *c1 = nullptr, *v0 = nullptr, *v1 = nullptr;
        int b0 = 0, b1 = 0;
        if (content) {
            int y0, y1;
            y_taps(dy, f.scale_y, f.h, &y0, &y1, &b0, &b1);
            r0 = stage_row(rowbuf0, f.data + (size_t)y0 * f.pitch, src_row_bytes);
            r1 = b1 != 0 ? stage_row(rowbuf1, f.data + (size_t)y1 * f.pitch, src_row_bytes) : r0;
            if (PL) {   // U and V halves of one chroma row when both taps share it (or the second tap has weight 0)
                const int cb = f.w >> 1;
                const size_t oc0 = (size_t)(y0 >> 1) * f.pitch_uv, oc1 = (size_t)(y1 >> 1) * f.pitch_uv;
                c0 = stage_row(rowbuf2, f.uv + oc0, cb);
                v0 = stage_row(rowbuf2 + half, f.v_plane() + oc0, cb);
                const bool two = b1 != 0 && (y1 >> 1) != (y0 >> 1);
                c1 = two ? stage_row(rowbuf3, f.uv + oc1, cb) : c0;
                v1 = two ? stage_row(rowbuf3 + half, f.v_plane() + oc1, cb) : v0;
            } else if (NV) {   // one UV row when both taps share it (or the second tap has weight 0)
                c0 = stage_row(rowbuf2, f.uv + (size_t)(y0 >> 1) * f.pitch_uv, src_row_bytes);
                c1 = b1 != 0 && (y1 >> 1) != (y0 >> 1) ? stage_row(rowbuf3, f.uv + (size_t)(y1 >> 1) * f.pitch_uv, src_row_bytes) : c0;
            }
            __syncthreads();
        }
        for (int g = threadIdx.x; g < ngroups; g += blockDim.x) {
            float vr[4], vg[4], vb[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int x = 4 * g + j;
                if (content && x < f.new_w) {
                    const int x0 = xo0[x], x1 = xo1[x], a0 = xa0[x], a1 = xa1[x];
                    if (PK) {
                        const unsigned p = resize_px24(packed_px24(r0, sel, x0), packed_px24(r0, sel, x1),
                                                       b1 != 0 ? packed_px24(r1, sel, x0) : 0u, b1 != 0 ? packed_px24(r1, sel, x1) : 0u,
                                                       a0, a1, b0, b1);
                        vb[j] = lut[p & 255u];
                        vg[j] = lut[256 + ((p >> 8) & 255u)];
                        vr[j] = lut[512 + (p >> 16)];
                    } else if (NV) {
                        const unsigned p = resize_px24(yuv_px24<FMT>(r0, c0, v0, x0), yuv_px24<FMT>(r0, c0, v0, x1),
                                                       b1 != 0 ? yuv_px24<FMT>(r1, c1, v1, x0) : 0u, b1 != 0 ? yuv_px24<FMT>(r1, c1, v1, x1) : 0u,
                                                       a0, a1, b0, b1);
                        vb[j] = lut[p & 255u];
                        vg[j] = lut[256 + ((p >> 8) & 255u)];
                        vr[j] = lut[512 + (p >> 16)];
                    } else if (P4) {
                        const unsigned p = resize_px24(px32_px24(r0, sel, x0), px32_px24(r0, sel, x1),
                                                       b1 != 0 ? px32_px24(r1, sel, x0) : 0u, b1 != 0 ? px32_px24(r1, sel, x1) : 0u,
                                                       a0, a1, b0, b1);
                        vb[j] = lut[p & 255u];
                        vg[j] = lut[256 + ((p >> 8) & 255u)];
                        vr[j] = lut[512 + (p >> 16)];
                    } else if (G1) {   // one resize indexes the three planes
                        const int p = resize_px(r0, r1, x0, x1, a0, a1, b0, b1);
                        vb[j] = lut[p];
                        vg[j] = lut[256 + p];
                        vr[j] = lut[512 + p];
                    } else {   // BGR, or RGB24 with channels 0 and 2 exchanged
                        vb[j] = lut[resize_px(r0, r1, x0 + (RG ? 2 : 0), x1 + (RG ? 2 : 0), a0, a1, b0, b1)];
                        vg[j] = lut[256 + resize_px(r0, r1, x0 + 1, x1 + 1, a0, a1, b0, b1)];
                        vr[j] = lut[512 + resize_px(r0, r1, x0 + (RG ? 0 : 2), x1 + (RG ? 0 : 2), a0, a1, b0, b1)];
                    }
                } else {
                    vb[j] = pad_b; vg[j] = pad_g; vr[j] = pad_r;
                }
            }
            if (a.vec_store) {
                *reinterpret_cast<float4 *>(o_r + 4 * g) = make_float4(vr[0], vr[1], vr[2], vr[3]);
                *reinterpret_cast<float4 *>(o_g + 4 * g) = make_float4(vg[0], vg[1], vg[2], vg[3]);
                *reinterpret_cast<float4 *>(o_b + 4 * g) = make_float4(vb[0], vb[1], vb[2], vb[3]);
            } else {
                for (int j = 0; j < 4 && 4 * g + j < ow; ++j) {
                    o_r[4 * g + j] = vr[j];
                    o_g[4 * g + j] = vg[j];
                    o_b[4 * g + j] = vb[j];
                }
            }
        }
        if (content) __syncthreads();  // row buffers are overwritten by the next row
    }
}

// ---- v2: bulk-TMA staged variant ------------------------------------------------------------------------------------
// Same arithmetic, different data movement: source rows are brought into shared memory by the TMA engine
// (cp.async.bulk global->shared, completion on an mbarrier) in a PRE2_STAGES-deep ring, so no thread spends issue
// slots on staging; each thread keeps the x taps of its 4 pixels in registers; rows whose taps are all single-pixel
// (exact integer scales such as 1080p -> 640x360: scale 3, fractions 0) reduce to byte gathers; identity normalisation
// skips the table.  Requires 16-byte aligned rows (base, pitch) — otherwise the v1 kernel above is used.
constexpr int PRE2_STAGES = 4;
// RGBA / BGRA rows are a third longer than BGR ones: with three stages a 4K frame's ring (94 KB) still leaves room for two
// CTAs per SM, which four stages (123 KB) do not.
template <int FMT> constexpr int PRE2_STAGES_OF = FMT == SRC_PX32 ? 3 : PRE2_STAGES;
constexpr int PRE2_ROWS = 16;

// pixel x of a packed 4:2:2 row staged at a 4-byte aligned address: its macropixel as one aligned word
__device__ __forceinline__ unsigned packed_tap(const uint8_t *row, unsigned sel, int x) {
    return packed_bgr24(__byte_perm(*reinterpret_cast<const unsigned *>(row + 4 * (x >> 1)), 0u, sel), x);
}
// pixel x of an RGBA / BGRA row staged at a 4-byte aligned address: one aligned word reordered to B,G,R,x (byte 3 is then
// the alpha, which the callers mask off)
__device__ __forceinline__ unsigned px32_tap(const uint8_t *row, unsigned sel, int x) {
    return __byte_perm(*reinterpret_cast<const unsigned *>(row + 4 * x), 0u, sel);
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// FMT: the source format (SrcFmt).  4:2:0: a stage holds the Y rows of the taps and their chroma row(s) — one when both
// taps map to the same chroma row (4K -> 640x360: rows 6y+2 and 6y+3 both read chroma row 3y+1).  A planar chroma row
// fills its slot as the U half and, row_buf_bytes / 2 further, the V half: bulk copies of round16(w/2) bytes each.
// Packed 4:2:2: a stage holds the packed tap rows (2w bytes each), and a tap reads its macropixel as one aligned word.
// RGB family: a stage holds the tap rows (RGB24 3w, RGBA / BGRA 4w, GRAY8 w bytes); a 4-byte tap is one aligned word, and a
// GRAY8 tap is resized once and indexes the three planes.
template <bool IDENT, int FMT>
__global__ void __launch_bounds__(256) preprocess_tma_kernel(PreArgs a) {
    constexpr bool NV = FMT == SRC_NV12 || FMT == SRC_NV21 || FMT == SRC_PLANAR, PL = FMT == SRC_PLANAR;   // NV: 4:2:0
    constexpr bool PK = FMT == SRC_PACKED422;
    constexpr bool RG = FMT == SRC_RGB24, P4 = FMT == SRC_PX32, G1 = FMT == SRC_GRAY8;
    constexpr bool PXO = NV || PK || P4 || G1;   // taps in pixels, not bytes
    constexpr int STAGES = PRE2_STAGES_OF<FMT>;
    constexpr int SLOTS = NV ? 4 : 2;                           // rows per stage: Y0, Y1 (BGR: row 0, row 1), UV0, UV1
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem);        // [STAGES]
    float *lut = reinterpret_cast<float *>(smem + 64);          // [3][256]
    uint8_t *bufs = smem + 64 + 3072;                           // [STAGES][SLOTS][row_buf_bytes]
    const int tid = threadIdx.x;
    const int ow = a.out_w;
    const int rb = a.row_buf_bytes;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (!IDENT) {
        for (int i = tid; i < 768; i += blockDim.x) {
            int c = i >> 8, v = i & 255;
            lut[i] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)v, a.pixel_scale), a.means[c]), a.stds[c]);
        }
    }
    pdl_wait();   // (no early trigger: the detect kernel's CTAs would take SMs this grid still needs)
    const FrameDev f = a.frames[blockIdx.y];
    // x taps of this thread's 4 pixels, in registers
    int x0[4];
    short wa0[4], wa1[4];
    bool point = true;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int x = 4 * tid + j;
        x0[j] = -1;
        wa0[j] = 0;
        wa1[j] = 0;
        if (x < f.new_w) {
            int o1;
            x_taps(x, f.scale_x, f.w, &x0[j], &o1, &wa0[j], &wa1[j]);
            if (PXO) x0[j] /= 3;   // pixel, not byte, offset
            point &= (wa1[j] == 0);
        }
    }
    const bool hpoint = __syncthreads_and(point);  // also publishes the barrier init and the table

    const float pad_b = IDENT ? 0.0f : lut[0], pad_g = IDENT ? 0.0f : lut[256], pad_r = IDENT ? 0.0f : lut[512];
    const size_t plane = (size_t)a.out_h * ow;
    float *out_img = a.out + (size_t)blockIdx.y * 3 * plane;
    const int row_begin = blockIdx.x * PRE2_ROWS;
    const int row_end = min(row_begin + PRE2_ROWS, a.out_h);
    const int n_content = max(0, min(f.new_h, row_end) - row_begin);
    const uint32_t copy_bytes = (uint32_t)(((NV || G1 ? f.w : PK ? 2 * f.w : P4 ? 4 * f.w : f.w * 3) + 15) & ~15);
    const unsigned sel = PK || P4 ? (unsigned)f.v_off : 0u;
    const uint32_t half_bytes = (uint32_t)(((f.w >> 1) + 15) & ~15);   // PL: one U or V row
    const int half = rb >> 1;
    const bool active = 4 * tid < ow;

    auto issue = [&](int it) {
        int y0, y1, b0, b1;
        y_taps(row_begin + it, f.scale_y, f.h, &y0, &y1, &b0, &b1);
        const int st = it % STAGES;
        uint8_t *dst = bufs + (size_t)st * SLOTS * rb;
        const bool uv1 = NV && b1 != 0 && (y1 >> 1) != (y0 >> 1);
        if (PL) mbar_expect_tx(&full[st], copy_bytes * (b1 != 0 ? 2 : 1) + half_bytes * (uv1 ? 4 : 2));
        else mbar_expect_tx(&full[st], copy_bytes * ((b1 != 0 ? 2 : 1) + (NV ? 1 : 0) + (uv1 ? 1 : 0)));
        bulk_g2s(dst, f.data + (size_t)y0 * f.pitch, copy_bytes, &full[st]);
        if (b1 != 0) bulk_g2s(dst + rb, f.data + (size_t)y1 * f.pitch, copy_bytes, &full[st]);
        if (PL) {
            const size_t oc0 = (size_t)(y0 >> 1) * f.pitch_uv, oc1 = (size_t)(y1 >> 1) * f.pitch_uv;
            bulk_g2s(dst + 2 * rb, f.uv + oc0, half_bytes, &full[st]);
            bulk_g2s(dst + 2 * rb + half, f.v_plane() + oc0, half_bytes, &full[st]);
            if (uv1) {
                bulk_g2s(dst + 3 * rb, f.uv + oc1, half_bytes, &full[st]);
                bulk_g2s(dst + 3 * rb + half, f.v_plane() + oc1, half_bytes, &full[st]);
            }
        } else {
            if (NV) bulk_g2s(dst + 2 * rb, f.uv + (size_t)(y0 >> 1) * f.pitch_uv, copy_bytes, &full[st]);
            if (uv1) bulk_g2s(dst + 3 * rb, f.uv + (size_t)(y1 >> 1) * f.pitch_uv, copy_bytes, &full[st]);
        }
    };
    if (tid == 0)
        for (int it = 0; it < STAGES - 1 && it < n_content; ++it) issue(it);

    for (int it = 0; it < n_content; ++it) {
        if (tid == 0 && it + STAGES - 1 < n_content) issue(it + STAGES - 1);
        const int dy = row_begin + it;
        int y0, y1, b0, b1;
        y_taps(dy, f.scale_y, f.h, &y0, &y1, &b0, &b1);
        const int st = it % STAGES;
        const uint8_t *r0 = bufs + (size_t)st * SLOTS * rb;
        const uint8_t *r1 = b1 != 0 ? r0 + rb : r0;
        const uint8_t *c0 = r0 + 2 * rb, *c1 = b1 != 0 && (y1 >> 1) != (y0 >> 1) ? r0 + 3 * rb : c0;   // NV only
        const uint8_t *v0 = c0 + half, *v1 = c1 + half;                                               // PL only
        mbar_wait(&full[st], (uint32_t)((it / STAGES) & 1));
        if (active) {
            float vr[4], vg[4], vb[4];
            if (hpoint && b1 == 0) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (x0[j] >= 0) {
                        int pb, pg, pr;
                        if (PK) {
                            const unsigned p = packed_tap(r0, sel, x0[j]);
                            pb = p & 255u; pg = (p >> 8) & 255u; pr = p >> 16;
                        } else if (NV) {
                            const unsigned p = yuv_px24<FMT>(r0, c0, v0, x0[j]);
                            pb = p & 255u; pg = (p >> 8) & 255u; pr = p >> 16;
                        } else if (P4) {
                            const unsigned p = px32_tap(r0, sel, x0[j]);
                            pb = p & 255u; pg = (p >> 8) & 255u; pr = (p >> 16) & 255u;
                        } else if (G1) {
                            pb = pg = pr = r0[x0[j]];
                        } else {   // BGR, or RGB24 with channels 0 and 2 exchanged
                            const uint8_t *p = r0 + x0[j];
                            pb = p[RG ? 2 : 0]; pg = p[1]; pr = p[RG ? 0 : 2];
                        }
                        vb[j] = IDENT ? (float)pb : lut[pb];
                        vg[j] = IDENT ? (float)pg : lut[256 + pg];
                        vr[j] = IDENT ? (float)pr : lut[512 + pr];
                    } else {
                        vb[j] = pad_b; vg[j] = pad_g; vr[j] = pad_r;
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (x0[j] >= 0) {
                        const int o0 = x0[j], o1 = x0[j] + (wa1[j] != 0 ? (PXO ? 1 : 3) : 0), q0 = wa0[j], q1 = wa1[j];
                        int pb, pg, pr;
                        if (PK) {
                            const unsigned p = resize_px24(packed_tap(r0, sel, o0), packed_tap(r0, sel, o1),
                                                           b1 != 0 ? packed_tap(r1, sel, o0) : 0u, b1 != 0 ? packed_tap(r1, sel, o1) : 0u,
                                                           q0, q1, b0, b1);
                            pb = p & 255u; pg = (p >> 8) & 255u; pr = p >> 16;
                        } else if (NV) {
                            const unsigned p = resize_px24(yuv_px24<FMT>(r0, c0, v0, o0), yuv_px24<FMT>(r0, c0, v0, o1),
                                                           b1 != 0 ? yuv_px24<FMT>(r1, c1, v1, o0) : 0u,
                                                           b1 != 0 ? yuv_px24<FMT>(r1, c1, v1, o1) : 0u, q0, q1, b0, b1);
                            pb = p & 255u; pg = (p >> 8) & 255u; pr = p >> 16;
                        } else if (P4) {   // resize_px24 keeps only bytes 0..2 of the taps: the alpha byte drops out
                            const unsigned p = resize_px24(px32_tap(r0, sel, o0), px32_tap(r0, sel, o1),
                                                           b1 != 0 ? px32_tap(r1, sel, o0) : 0u, b1 != 0 ? px32_tap(r1, sel, o1) : 0u,
                                                           q0, q1, b0, b1);
                            pb = p & 255u; pg = (p >> 8) & 255u; pr = p >> 16;
                        } else if (G1) {
                            pb = pg = pr = resize_px(r0, r1, o0, o1, q0, q1, b0, b1);
                        } else {   // BGR, or RGB24 with channels 0 and 2 exchanged
                            pb = resize_px(r0, r1, o0 + (RG ? 2 : 0), o1 + (RG ? 2 : 0), q0, q1, b0, b1);
                            pg = resize_px(r0, r1, o0 + 1, o1 + 1, q0, q1, b0, b1);
                            pr = resize_px(r0, r1, o0 + (RG ? 0 : 2), o1 + (RG ? 0 : 2), q0, q1, b0, b1);
                        }
                        vb[j] = IDENT ? (float)pb : lut[pb];
                        vg[j] = IDENT ? (float)pg : lut[256 + pg];
                        vr[j] = IDENT ? (float)pr : lut[512 + pr];
                    } else {
                        vb[j] = pad_b; vg[j] = pad_g; vr[j] = pad_r;
                    }
                }
            }
            float *o_r = out_img + (size_t)dy * ow + 4 * tid;
            __stcs(reinterpret_cast<float4 *>(o_r), make_float4(vr[0], vr[1], vr[2], vr[3]));
            __stcs(reinterpret_cast<float4 *>(o_r + plane), make_float4(vg[0], vg[1], vg[2], vg[3]));
            __stcs(reinterpret_cast<float4 *>(o_r + 2 * plane), make_float4(vb[0], vb[1], vb[2], vb[3]));
        }
        __syncthreads();  // every thread is done with this stage before thread 0 refills it
    }
    if (active) {
        const float4 zr = make_float4(pad_r, pad_r, pad_r, pad_r), zg = make_float4(pad_g, pad_g, pad_g, pad_g),
                     zb = make_float4(pad_b, pad_b, pad_b, pad_b);
        for (int dy = row_begin + n_content; dy < row_end; ++dy) {
            float *o_r = out_img + (size_t)dy * ow + 4 * tid;
            __stcs(reinterpret_cast<float4 *>(o_r), zr);
            __stcs(reinterpret_cast<float4 *>(o_r + plane), zg);
            __stcs(reinterpret_cast<float4 *>(o_r + 2 * plane), zb);
        }
    }
}

// plain cv::resize to u8 HWC (face_detection.rs:156 on its own; also the FaceAlignment fallback :98-105)
__global__ void resize_u8_kernel(FrameDev f, uint8_t *__restrict__ out, int out_h, int out_w) {
    const int dy = blockIdx.y;
    int y0, y1, b0, b1;
    y_taps(dy, f.scale_y, f.h, &y0, &y1, &b0, &b1);
    const uint8_t *r0 = f.data + (size_t)y0 * f.pitch, *r1 = f.data + (size_t)y1 * f.pitch;
    for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < out_w; x += gridDim.x * blockDim.x) {
        int x0, x1;
        short a0, a1;
        x_taps(x, f.scale_x, f.w, &x0, &x1, &a0, &a1);
        uint8_t *o = out + ((size_t)dy * out_w + x) * 3;
        if (f.h == out_h && f.w == out_w) {  // cv::resize copies when the size is unchanged
            o[0] = r0[x * 3]; o[1] = r0[x * 3 + 1]; o[2] = r0[x * 3 + 2];
        } else {
            o[0] = (uint8_t)resize_px(r0, r1, x0, x1, a0, a1, b0, b1);
            o[1] = (uint8_t)resize_px(r0, r1, x0 + 1, x1 + 1, a0, a1, b0, b1);
            o[2] = (uint8_t)resize_px(r0, r1, x0 + 2, x1 + 2, a0, a1, b0, b1);
        }
    }
}

// N1 (SURVEY 8f): post-align model preprocessors fused onto the warp output — FaceExtraction::_preprocess
// (face_extraction.rs:38-77), FaceQuality::call (face_quality.rs:43-101), FaceQualityAssessment::call
// (face_quality_assessment.rs:48-88): cv::resize INTER_LINEAR to the model input, BGR->RGB, (p - mean[i]) * mul[i], NCHW.
// crops (F, in_h, in_w, 3) u8 dense; out (F, 3, out_h, out_w).  4 pixels per thread, 128-bit stores per plane.
struct CropArgs {
    const uint8_t *crops;
    const int *count_dev;
    int F, in_h, in_w, out_h, out_w;
    float mean[3], mul[3];  // RGB order
    float *out;
};
__global__ void __launch_bounds__(256) crops_to_tensor_kernel(CropArgs a) {
    const int F = a.count_dev ? min(*a.count_dev, a.F) : a.F;
    const int groups_per_row = (a.out_w + 3) >> 2;
    const int groups = a.out_h * groups_per_row;
    const bool same = a.in_h == a.out_h && a.in_w == a.out_w;   // cv::resize copies when the size is unchanged
    const double scale_x = 1.0 / ((double)a.out_w / a.in_w), scale_y = 1.0 / ((double)a.out_h / a.in_h);
    const size_t plane = (size_t)a.out_h * a.out_w;
    for (int f = blockIdx.y; f < F; f += gridDim.y) {
        const uint8_t *src = a.crops + (size_t)f * a.in_h * a.in_w * 3;
        float *o = a.out + (size_t)f * 3 * plane;
        for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += gridDim.x * blockDim.x) {
            const int y = g / groups_per_row, x4 = (g - y * groups_per_row) * 4;
            float v[3][4];
            int y0 = y, y1 = y, b0 = 2048, b1 = 0;
            if (!same) y_taps(y, scale_y, a.in_h, &y0, &y1, &b0, &b1);
            const uint8_t *r0 = src + (size_t)y0 * a.in_w * 3, *r1 = src + (size_t)y1 * a.in_w * 3;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int x = min(x4 + j, a.out_w - 1);
                int bgr[3];
                if (same) {
                    bgr[0] = r0[x * 3]; bgr[1] = r0[x * 3 + 1]; bgr[2] = r0[x * 3 + 2];
                } else {
                    int o0, o1;
                    short q0, q1;
                    x_taps(x, scale_x, a.in_w, &o0, &o1, &q0, &q1);
#pragma unroll
                    for (int c = 0; c < 3; ++c) bgr[c] = resize_px(r0, r1, o0 + c, o1 + c, q0, q1, b0, b1);
                }
#pragma unroll
                for (int i = 0; i < 3; ++i) v[i][j] = __fmul_rn(__fsub_rn((float)bgr[2 - i], a.mean[i]), a.mul[i]);
            }
            float *dst = o + (size_t)y * a.out_w + x4;
            if (x4 + 3 < a.out_w && (a.out_w & 3) == 0) {
#pragma unroll
                for (int i = 0; i < 3; ++i) __stcs(reinterpret_cast<float4 *>(dst + i * plane), make_float4(v[i][0], v[i][1], v[i][2], v[i][3]));
            } else {
                for (int j = 0; j < 4 && x4 + j < a.out_w; ++j)
                    for (int i = 0; i < 3; ++i) dst[i * plane + j] = v[i][j];
            }
        }
    }
}

int crops_to_tensor_launch(fd_ctx *ctx, const uint8_t *crops_dev, const int *count_dev, int F, int in_h, int in_w, int out_h,
                           int out_w, const float *mean_rgb, const float *mul_rgb, float *out_dev) {
    if (F <= 0) return FD_OK;
    CropArgs a;
    a.crops = crops_dev;
    a.count_dev = count_dev;
    a.F = F; a.in_h = in_h; a.in_w = in_w; a.out_h = out_h; a.out_w = out_w;
    for (int i = 0; i < 3; ++i) { a.mean[i] = mean_rgb[i]; a.mul[i] = mul_rgb[i]; }
    a.out = out_dev;
    const int groups = out_h * ((out_w + 3) / 4);
    dim3 grid(std::max(1, std::min(16, (groups + 255) / 256)), std::min(F, 65535));
    if (count_dev) grid.y = std::min(F, std::max(1, ctx->num_sms * 8 / (int)grid.x));
    crops_to_tensor_kernel<<<grid, 256, 0, ctx->stream>>>(a);
    FD_LAUNCH_CHECK_NAMED(ctx, "crops_to_tensor_kernel");
    return FD_OK;
}

// launch names by source format (I420 and YV12 share the planar instantiations, YUY2, UYVY and YVYU the packed ones, RGBA
// and BGRA the 4-byte ones)
static const char *const TMA_NAMES[SRC_FMT_COUNT] = {"preprocess_tma_kernel",      "preprocess_tma_kernel_nv12",  "preprocess_tma_kernel_nv21",
                                                     "preprocess_tma_kernel_i420", "preprocess_tma_kernel_yuv422", "preprocess_tma_kernel_rgb24",
                                                     "preprocess_tma_kernel_rgba", "preprocess_tma_kernel_gray8"};
static const char *const PRE_NAMES[SRC_FMT_COUNT] = {"preprocess_kernel",      "preprocess_kernel_nv12",   "preprocess_kernel_nv21",
                                                     "preprocess_kernel_i420", "preprocess_kernel_yuv422", "preprocess_kernel_rgb24",
                                                     "preprocess_kernel_rgba", "preprocess_kernel_gray8"};

template <bool IDENT>
static void (*tma_kernel_for(int fmt))(PreArgs) {
    return fmt == SRC_NV12 ? preprocess_tma_kernel<IDENT, SRC_NV12>
           : fmt == SRC_NV21 ? preprocess_tma_kernel<IDENT, SRC_NV21>
           : fmt == SRC_PLANAR ? preprocess_tma_kernel<IDENT, SRC_PLANAR>
           : fmt == SRC_PACKED422 ? preprocess_tma_kernel<IDENT, SRC_PACKED422>
           : fmt == SRC_RGB24 ? preprocess_tma_kernel<IDENT, SRC_RGB24>
           : fmt == SRC_PX32 ? preprocess_tma_kernel<IDENT, SRC_PX32>
           : fmt == SRC_GRAY8 ? preprocess_tma_kernel<IDENT, SRC_GRAY8> : preprocess_tma_kernel<IDENT, SRC_BGR>;
}

// max_row_bytes: widest staged row (BGR and RGB24: 3w, NV12/NV21: w, planar: 2 round16(w/2), a U half and a V half, packed
// 4:2:2: 2w, RGBA / BGRA: 4w, GRAY8: w); fmt: the source format of frames_dev (SrcFmt).  A row too wide for the bulk-copy
// ring (PRE2_STAGES_OF x 2 rows: a 4K RGBA row of 15 360 B fits, an 8K one does not) takes the row-staging kernel.
int preprocess_launch(fd_ctx *ctx, const FrameDev *frames_dev, int B, float *out_nchw_dev, int max_row_bytes, bool rows_aligned16,
                      int fmt) {
    constexpr int SLOTS_NV = 4;
    const bool nv = fmt == SRC_NV12 || fmt == SRC_NV21 || fmt == SRC_PLANAR;   // 4:2:0: two more row slots for the chroma
    PreArgs a;
    a.frames = frames_dev;
    a.out = out_nchw_dev;
    a.out_w = ctx->cfg.image_w;
    a.out_h = ctx->cfg.image_h;
    a.pixel_scale = ctx->cfg.pixel_scale;
    bool ident = a.pixel_scale == 1.0f;
    for (int i = 0; i < 3; ++i) {
        a.means[i] = ctx->cfg.pixel_means[i];
        a.stds[i] = ctx->cfg.pixel_stds[i];
        ident = ident && a.means[i] == 0.0f && a.stds[i] == 1.0f;
    }
    a.row_buf_bytes = ((max_row_bytes + 32) + 15) & ~15;
    a.vec_store = (a.out_w % 4 == 0) && ((reinterpret_cast<uintptr_t>(out_nchw_dev) & 15) == 0);
    const int ngroups = (a.out_w + 3) / 4;
    // v2 (bulk-TMA staging): 16-byte aligned source rows, vector stores, one 4-pixel group per thread
    if (rows_aligned16 && a.vec_store && ngroups <= 256) {
        a.row_buf_bytes = (max_row_bytes + 15) & ~15;
        const int stages = fmt == SRC_PX32 ? PRE2_STAGES_OF<SRC_PX32> : PRE2_STAGES;
        size_t smem = 64 + 3072 + (size_t)stages * (nv ? SLOTS_NV : 2) * a.row_buf_bytes;
        if (smem <= (size_t)ctx->max_smem_optin) {
            int threads = std::max(32, ((ngroups + 31) / 32) * 32);
            dim3 grid((a.out_h + PRE2_ROWS - 1) / PRE2_ROWS, B);
            void (*kern)(PreArgs) = ident ? tma_kernel_for<true>(fmt) : tma_kernel_for<false>(fmt);
            FD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            FD_TRY(launch_pdl(ctx, kern, grid, dim3(threads), smem, a));
            FD_LAUNCH_CHECK_NAMED(ctx, TMA_NAMES[fmt]);
            return FD_OK;
        }
    }
    size_t tab_bytes = 768 * 4 + (size_t)a.out_w * 12;
    tab_bytes = (tab_bytes + 15) & ~(size_t)15;
    size_t smem = tab_bytes + (nv ? SLOTS_NV : 2) * (size_t)a.row_buf_bytes;
    if (smem > (size_t)ctx->max_smem_optin) return fail(FD_ERR_INVALID, "fd_preprocess: source row too wide for shared-memory staging");
    void (*kern)(PreArgs) = fmt == SRC_NV12 ? preprocess_kernel<SRC_NV12>
                            : fmt == SRC_NV21 ? preprocess_kernel<SRC_NV21>
                            : fmt == SRC_PLANAR ? preprocess_kernel<SRC_PLANAR>
                            : fmt == SRC_PACKED422 ? preprocess_kernel<SRC_PACKED422>
                            : fmt == SRC_RGB24 ? preprocess_kernel<SRC_RGB24>
                            : fmt == SRC_PX32 ? preprocess_kernel<SRC_PX32>
                            : fmt == SRC_GRAY8 ? preprocess_kernel<SRC_GRAY8> : preprocess_kernel<SRC_BGR>;
    FD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int threads = std::min(1024, std::max(64, ((ngroups + 31) / 32) * 32));
    dim3 grid((a.out_h + PRE_ROWS - 1) / PRE_ROWS, B);
    FD_TRY(launch_pdl(ctx, kern, grid, dim3(threads), smem, a));
    FD_LAUNCH_CHECK_NAMED(ctx, PRE_NAMES[fmt]);
    return FD_OK;
}

int resize_launch(fd_ctx *ctx, const FrameDev &frame, uint8_t *out_dev, int out_h, int out_w) {
    dim3 grid(std::max(1, std::min(64, (out_w + 127) / 128)), out_h);
    resize_u8_kernel<<<grid, 128, 0, ctx->stream>>>(frame, out_dev, out_h, out_w);
    FD_LAUNCH_CHECK(ctx);
    return FD_OK;
}

}  // namespace fd
