// fd_pipeline.cu — batched device-resident pipeline entry points, single-image host wrappers and the
// host-buffer end-to-end call.  Mirrors RetinaFaceDetection::call (face_detection.rs:496-513) and
// FaceAlignment::call (face_alignment.rs:27-141) at batch granularity.
#include <algorithm>
#include <cmath>
#include <climits>
#include <cstdlib>
#include <cstddef>
#include <cstring>
#include "fd_internal.cuh"

namespace fd {

// Waits for the ctx stream.  In blocking mode (set by fd_pipeline_host: several host threads / processes each drive a ctx and
// sleep through multi-millisecond PCIe transfers) the wait is an OS-level block on an event created with
// cudaEventBlockingSync instead of a spin on the CPU, so N ranks x L lanes do not burn N*L host cores.
static int wait_stream(fd_ctx *ctx) {
    if (ctx->blocking_sync && ctx->ev_block) {
        FD_CUDA(cudaEventRecord(ctx->ev_block, ctx->stream));
        FD_CUDA(cudaEventSynchronize(ctx->ev_block));
    } else {
        FD_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return FD_OK;
}

// RetinaFaceDetection::_preprocess geometry (face_detection.rs:140-153): f32 arithmetic, `as i32` truncation
static void letterbox(int h, int w, int size_w, int size_h, int *new_w, int *new_h, float *det_scale) {
    volatile float im_ratio = (float)h / (float)w;
    volatile float model_ratio = (float)size_h / (float)size_w;
    if (im_ratio > model_ratio) {
        *new_h = size_h;
        volatile float q = (float)(*new_h) / im_ratio;
        *new_w = (int)q;
    } else {
        *new_w = size_w;
        volatile float q = (float)(*new_w) * im_ratio;
        *new_h = (int)q;
    }
    volatile float ds = (float)(*new_h) / (float)h;
    *det_scale = ds;
}

// letterbox geometry of an h x w frame (out->h, out->w, new_w, new_h, scales)
static int fill_geometry(const fd_ctx *ctx, int height, int width, FrameDev *out, float *det_scale) {
    out->h = height;
    out->w = width;
    float ds;
    letterbox(height, width, ctx->cfg.image_w, ctx->cfg.image_h, &out->new_w, &out->new_h, &ds);
    // cv::resize rejects an empty destination size (the reference returns Err, face_detection.rs:156-159)
    FD_REQUIRE(out->new_w > 0 && out->new_h > 0, "frame: letterbox size is empty (extreme aspect ratio)");
    out->new_w = std::min(out->new_w, ctx->cfg.image_w);
    out->new_h = std::min(out->new_h, ctx->cfg.image_h);
    out->scale_x = 1.0 / ((double)out->new_w / width);
    out->scale_y = 1.0 / ((double)out->new_h / height);
    if (det_scale) *det_scale = ds;
    return FD_OK;
}

static int fill_frame(const fd_ctx *ctx, const fd_frame &fr, const uint8_t *data_dev, FrameDev *out, float *det_scale) {
    FD_REQUIRE(fr.height > 0 && fr.width > 0 && fr.pitch >= fr.width * 3, "frame: bad geometry");
    out->data = data_dev;
    out->pitch = fr.pitch;
    return fill_geometry(ctx, fr.height, fr.width, out, det_scale);
}

// the kernels' source format of an FD_YUV420_* layout, or -1
static int yuv420_format(int32_t layout) {
    switch (layout) {
    case FD_YUV420_NV12: return SRC_NV12;
    case FD_YUV420_NV21: return SRC_NV21;
    case FD_YUV420_I420:
    case FD_YUV420_YV12: return SRC_PLANAR;
    default: return -1;
    }
}

// cv::cvtColor(COLOR_YUV2BGR_NV12 / _NV21 / _I420 / _YV12) accepts even sizes only.  The planar layouts' second chroma
// plane starts (height/2) * pitch_uv bytes after the first: V after U for I420, U after V for YV12.
static int fill_frame_yuv420(const fd_ctx *ctx, const fd_frame_nv12 &fr, int32_t layout, FrameDev *out, float *det_scale) {
    const bool planar = yuv420_format(layout) == SRC_PLANAR;
    FD_REQUIRE(fr.y && fr.uv, "frame (YUV 4:2:0): null plane");
    FD_REQUIRE(fr.height > 0 && fr.width > 0 && fr.height % 2 == 0 && fr.width % 2 == 0 && fr.pitch_y >= fr.width &&
                   fr.pitch_uv >= (planar ? fr.width / 2 : fr.width),
               "frame (YUV 4:2:0): bad geometry (width and height must be even, pitches at least the width, or half of it for "
               "the planar chroma)");
    out->data = fr.y;
    out->pitch = fr.pitch_y;
    out->uv = fr.uv;
    out->pitch_uv = fr.pitch_uv;
    if (planar) {   // V - U fits the table's 32-bit offset
        const size_t plane = (size_t)(fr.height / 2) * fr.pitch_uv;
        FD_REQUIRE(plane <= 0x7fffffffull, "frame (YUV 4:2:0): chroma plane of 2 GB or more");
        out->v_off = layout == FD_YUV420_I420 ? (int)plane : -(int)plane;
        if (layout == FD_YUV420_YV12) out->uv = fr.uv + plane;
    }
    return fill_geometry(ctx, fr.height, fr.width, out, det_scale);
}

// __byte_perm selector that reorders a macropixel of an FD_YUV422_* layout to Y0 U Y1 V, or -1
static int yuv422_selector(int32_t layout) {
    switch (layout) {
    case FD_YUV422_YUY2: return 0x3210;
    case FD_YUV422_UYVY: return 0x2301;   // U Y0 V Y1
    case FD_YUV422_YVYU: return 0x1230;   // Y0 V Y1 U
    default: return -1;
    }
}

// cv::cvtColor(COLOR_YUV2BGR_YUY2 / _UYVY / _YVYU) accepts even widths and any height.
static int fill_frame_yuv422(const fd_ctx *ctx, const fd_frame &fr, int32_t layout, FrameDev *out, float *det_scale) {
    FD_REQUIRE(fr.data, "frame (YUV 4:2:2): null data");
    FD_REQUIRE(fr.height > 0 && fr.width > 0 && fr.width % 2 == 0 && (int64_t)fr.pitch >= 2 * (int64_t)fr.width,
               "frame (YUV 4:2:2): bad geometry (width must be even, pitch at least twice the width)");
    out->data = fr.data;
    out->pitch = fr.pitch;
    out->v_off = yuv422_selector(layout);
    return fill_geometry(ctx, fr.height, fr.width, out, det_scale);
}

// the kernels' source format of an FD_RGB_* layout, or -1
static int rgb_format(int32_t layout) {
    switch (layout) {
    case FD_RGB_RGB24: return SRC_RGB24;
    case FD_RGB_RGBA:
    case FD_RGB_BGRA: return SRC_PX32;
    case FD_RGB_GRAY8: return SRC_GRAY8;
    default: return -1;
    }
}

// bytes per pixel of a known FD_RGB_* layout
static int rgb_bpp(int32_t layout) { return layout == FD_RGB_RGB24 ? 3 : layout == FD_RGB_GRAY8 ? 1 : 4; }

// cv::cvtColor(COLOR_RGB2BGR / RGBA2BGR / BGRA2BGR / GRAY2BGR) accepts any size.  An RGBA / BGRA frame carries the
// __byte_perm selector that reorders its pixel word to B,G,R,x.
static int fill_frame_rgb(const fd_ctx *ctx, const fd_frame &fr, int32_t layout, FrameDev *out, float *det_scale) {
    FD_REQUIRE(fr.data, "frame (RGB): null data");
    FD_REQUIRE(fr.height > 0 && fr.width > 0 && (int64_t)fr.pitch >= rgb_bpp(layout) * (int64_t)fr.width,
               "frame (RGB): bad geometry (pitch at least the bytes per pixel times the width)");
    out->data = fr.data;
    out->pitch = fr.pitch;
    out->v_off = layout == FD_RGB_RGBA ? 0x3012 : layout == FD_RGB_BGRA ? 0x3210 : 0;
    return fill_geometry(ctx, fr.height, fr.width, out, det_scale);
}

// The frames of a batched call, device pointers: BGR (bgr), 4:2:0 (yuv, in the FD_YUV420_* layout `layout`), packed 4:2:2
// (packed, in the FD_YUV422_* layout `layout`) or interleaved RGB-family (rgb, in the FD_RGB_* layout `layout`); exactly one
// is set.
struct FrameList {
    const fd_frame *bgr = nullptr;
    const fd_frame_nv12 *yuv = nullptr;
    const fd_frame *packed = nullptr;
    const fd_frame *rgb = nullptr;
    int32_t layout = FD_YUV420_NV12;
    bool any() const { return bgr || yuv || packed || rgb; }
};

// the FrameList of a *_yuv420 call; an unknown layout is rejected here, before any call can return early
static int yuv420_frames(const fd_frame_nv12 *frames, int32_t layout, FrameList *fl) {
    FD_REQUIRE(yuv420_format(layout) >= 0, "frame (YUV 4:2:0): unknown layout");
    fl->yuv = frames;
    fl->layout = layout;
    return FD_OK;
}

// the FrameList of a *_yuv422 call; an unknown layout is rejected here, before any call can return early
static int yuv422_frames(const fd_frame *frames, int32_t layout, FrameList *fl) {
    FD_REQUIRE(yuv422_selector(layout) >= 0, "frame (YUV 4:2:2): unknown layout");
    fl->packed = frames;
    fl->layout = layout;
    return FD_OK;
}

// the FrameList of an *_rgb call; an unknown layout is rejected here, before any call can return early
static int rgb_frames(const fd_frame *frames, int32_t layout, FrameList *fl) {
    FD_REQUIRE(rgb_format(layout) >= 0, "frame (RGB): unknown layout");
    fl->rgb = frames;
    fl->layout = layout;
    return FD_OK;
}

// the kernels' source format of a FrameList whose layout is known (yuv420_frames, yuv422_frames, rgb_frames)
static int frames_format(const FrameList &frames) {
    return frames.rgb ? rgb_format(frames.layout) : frames.packed ? SRC_PACKED422 : frames.yuv ? yuv420_format(frames.layout) : SRC_BGR;
}

// validates frame i of `frames` and fills its table entry; *row_bytes: the staged source row of the frame in bytes (BGR and
// RGB24: 3w, NV12/NV21: w, planar: a U and a V half of round16(w/2) bytes each, packed 4:2:2: 2w, RGBA / BGRA: 4w, GRAY8: w)
static int fill_frame_of(const fd_ctx *ctx, const FrameList &frames, int i, FrameDev *out, float *ds, int *row_bytes) {
    memset(out, 0, sizeof(FrameDev));
    if (frames.yuv) {
        const int w = frames.yuv[i].width;
        FD_TRY(fill_frame_yuv420(ctx, frames.yuv[i], frames.layout, out, ds));
        *row_bytes = yuv420_format(frames.layout) == SRC_PLANAR ? 2 * ((w / 2 + 15) & ~15) : w;
    } else if (frames.packed) {
        FD_TRY(fill_frame_yuv422(ctx, frames.packed[i], frames.layout, out, ds));
        *row_bytes = 2 * frames.packed[i].width;
    } else if (frames.rgb) {
        FD_TRY(fill_frame_rgb(ctx, frames.rgb[i], frames.layout, out, ds));
        *row_bytes = rgb_bpp(frames.layout) * frames.rgb[i].width;
    } else {
        FD_REQUIRE(frames.bgr[i].data != nullptr, "frame: null data");
        FD_TRY(fill_frame(ctx, frames.bgr[i], frames.bgr[i].data, out, ds));
        *row_bytes = frames.bgr[i].width * 3;
    }
    return FD_OK;
}

// uploads B descriptors and records their source format in ctx->frames_fmt (the same buffers described as BGR and as RGB24
// give byte-identical tables: only the format tells them apart); returns the widest staged source row in bytes
static int upload_frame_table(fd_ctx *ctx, FrameList frames, int B, float *det_scale_host, int *max_row_bytes) {
    const int fmt = frames_format(frames);
    std::vector<FrameDev> tab(B);
    int mrb = 0;
    for (int i = 0; i < B; ++i) {
        float ds;
        int rb;
        FD_TRY(fill_frame_of(ctx, frames, i, &tab[i], &ds, &rb));
        mrb = std::max(mrb, rb);
        if (det_scale_host) det_scale_host[i] = ds;
    }
    if (max_row_bytes) *max_row_bytes = mrb;
    ctx->frames_fmt = fmt;
    const size_t bytes = sizeof(FrameDev) * (size_t)B;
    // the table already on the device is reused when nothing changed (steady-state streaming over a frame ring)
    if (ctx->frames_shadow.size() == bytes && memcmp(ctx->frames_shadow.data(), tab.data(), bytes) == 0) return FD_OK;
    FD_TRY(ctx->pinned[0].reserve(bytes));
    FD_TRY(ctx->frames_dev.reserve(bytes));
    FD_CUDA(cudaEventSynchronize(ctx->ev[0]));  // the pinned staging copy may still be in flight
    memcpy(ctx->pinned[0].p, tab.data(), bytes);
    FD_CUDA(cudaMemcpyAsync(ctx->frames_dev.p, ctx->pinned[0].p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    FD_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    ctx->frames_shadow.assign(reinterpret_cast<unsigned char *>(tab.data()), reinterpret_cast<unsigned char *>(tab.data()) + bytes);
    return FD_OK;
}

// from_detect: the faces are the detections of the last fd_detect_batch; when the fused detect kernel already estimated
// their transforms (ctx->est_valid) and they all fit, the estimate launch is skipped.
// fb: the bbox rows / selection of the fallback (face_alignment.rs:64-116); ok_dev receives the per-face mode (0/1/2).
// The frames are those of the table in ctx->frames_dev, in its format (ctx->frames_fmt).
static int align_enqueue(fd_ctx *ctx, const float *lmk_dev, const int32_t *frame_idx_dev,
                         const int *count_dev, int F_cap, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev, bool from_detect,
                         WarpFallback fb) {
    if (F_cap <= 0) return FD_OK;
    ctx->align_cap_hint = std::max(ctx->align_cap_hint, F_cap);
    const bool reuse = from_detect && ctx->est_valid && F_cap <= ctx->est_cap && !M_dev;
    if (!reuse) {
        ctx->est_valid = false;
        FD_TRY(ctx->align_M.reserve(sizeof(double) * 12 * (size_t)F_cap));
        FD_TRY(ctx->align_ok.reserve((size_t)F_cap));
        FD_TRY(estimate_launch(ctx, lmk_dev, nullptr, count_dev, F_cap, ctx->align_M.as<double>(), M_dev, ctx->align_ok.as<uint8_t>(), nullptr));
    }
    fb.mode_out = ok_dev;
    FD_TRY(warp_launch(ctx, ctx->frames_dev.as<FrameDev>(), frame_idx_dev, ctx->align_M.as<double>(), ctx->align_ok.as<uint8_t>(), count_dev,
                       F_cap, crops_dev, ctx->cfg.crop_w, ctx->cfg.crop_h, fb, ctx->frames_fmt));
    return FD_OK;
}

// the detections of the last fd_detect_batch as fallback boxes: row f of out_det = x1,y1,x2,y2,score
static WarpFallback detect_fallback(fd_ctx *ctx) {
    WarpFallback fb;
    fb.bbox = ctx->out_det.as<float>();
    fb.bbox_stride = 5;
    return fb;
}

// completes a pending fd_detect_batch: runs the big path for images the detect kernel deferred (K > 4096)
static int detect_resolve(fd_ctx *ctx) {
    if (!ctx->detect_pending) return FD_OK;
    const int B = ctx->last_B;
    int st[4] = {0, 0, 0, 0};
    FD_CUDA(cudaMemcpyAsync(st, ctx->status(), sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    FD_TRY(wait_stream(ctx));
    ctx->detect_pending = false;
    if (st[1] > 0) {
        ctx->crowded = true;   // later fused launches keep images with up to 4096 candidates on the device
        std::vector<int> big(st[1]), counts(B);
        FD_CUDA(cudaMemcpy(big.data(), ctx->big_list.p, sizeof(int) * st[1], cudaMemcpyDeviceToHost));
        FD_CUDA(cudaMemcpy(counts.data(), ctx->cand_count.p, sizeof(int) * B, cudaMemcpyDeviceToHost));
        for (int b : big) {
            if (counts[b] <= 4096) FD_TRY(nms_batch_small_image(ctx, b, counts[b], ctx->last_iou));
            else FD_TRY(nms_batch_big_image(ctx, b, counts[b], ctx->last_iou));
        }
        FD_TRY(finalize_launch(ctx, B));
        ctx->est_valid = false;
        if (ctx->align_replay)  // the crops were produced from incomplete detections: align again (in the table's format)
            FD_TRY(align_enqueue(ctx, ctx->out_lmk.as<float>(), ctx->out_frame_idx.as<int32_t>(),
                                 ctx->status() + 2, ctx->align_cap, ctx->align_crops, ctx->align_M_out, ctx->align_ok_out, true,
                                 detect_fallback(ctx)));
        FD_TRY(wait_stream(ctx));
    }
    return FD_OK;
}

static int reserve_detect(fd_ctx *ctx, int B) {
    const size_t TA = (size_t)ctx->dcfg.total_anchors, n = TA * B;
    FD_TRY(ctx->det_scale_dev.reserve(sizeof(float) * B));
    FD_TRY(ctx->cand_count.reserve(sizeof(int) * B));
    FD_TRY(ctx->cand_keys.reserve(sizeof(unsigned long long) * n));
    FD_TRY(ctx->cand_box.reserve(sizeof(float4) * n));
    FD_TRY(ctx->cand_lmk.reserve(sizeof(float) * 12 * n));
    FD_TRY(ctx->keep_src.reserve(sizeof(int) * n));
    FD_TRY(ctx->keep_count.reserve(sizeof(int) * B));
    if (!ctx->status_dev.p) {   // both halves start at zero; afterwards every detect call leaves the OTHER half zeroed
        FD_TRY(ctx->status_dev.reserve(sizeof(int) * 16));
        FD_CUDA(cudaMemsetAsync(ctx->status_dev.p, 0, sizeof(int) * 16, ctx->stream));
    }
    FD_TRY(ctx->big_list.reserve(sizeof(int) * B));
    FD_TRY(ctx->out_offsets.reserve(sizeof(int) * (B + 1)));
    FD_TRY(ctx->out_det.reserve(sizeof(float) * 5 * n));
    FD_TRY(ctx->out_lmk.reserve(sizeof(float) * 10 * n));
    FD_TRY(ctx->out_frame_idx.reserve(sizeof(int) * n));
    // transforms of the detections, estimated inside the fused detect kernel for the align call that usually follows
    ctx->est_cap = (int)std::min<size_t>(n, (size_t)std::max(ctx->align_cap_hint, B * 64));
    FD_TRY(ctx->align_M.reserve(sizeof(double) * 12 * (size_t)ctx->est_cap));
    FD_TRY(ctx->align_ok.reserve((size_t)ctx->est_cap));
    return FD_OK;
}

static int detect_enqueue(fd_ctx *ctx, const float *const *heads_dev, int B, const float *det_scale_host, float conf_thr,
                          float iou_thr) {
    FD_TRY(reserve_detect(ctx, B));
    if (ctx->det_scale_shadow.size() != (size_t)B || memcmp(ctx->det_scale_shadow.data(), det_scale_host, sizeof(float) * (size_t)B) != 0) {
        FD_TRY(ctx->pinned[1].reserve(sizeof(float) * (size_t)B));
        FD_CUDA(cudaEventSynchronize(ctx->ev[1]));
        memcpy(ctx->pinned[1].p, det_scale_host, sizeof(float) * (size_t)B);
        FD_CUDA(cudaMemcpyAsync(ctx->det_scale_dev.p, ctx->pinned[1].p, sizeof(float) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
        FD_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
        ctx->det_scale_shadow.assign(det_scale_host, det_scale_host + B);
    }
    // status flags: the half the previous call did not use was zeroed by that call's kernel (no memset node on the stream)
    ctx->status_cur ^= 8;
    bool fused = false;
    FD_TRY(detect_fused_launch(ctx, heads_dev, B, conf_thr, iou_thr, ctx->est_cap, &fused));
    if (!fused) {
        FD_CUDA(cudaMemsetAsync(ctx->status_dev.p, 0, sizeof(int) * 16, ctx->stream));
        FD_CUDA(cudaMemsetAsync(ctx->cand_count.p, 0, sizeof(int) * (size_t)B, ctx->stream));
        FD_TRY(decode_launch(ctx, heads_dev, B, conf_thr));
        FD_TRY(nms_batch_launch(ctx, B, iou_thr));
        FD_TRY(finalize_launch(ctx, B));
    }
    ctx->est_valid = fused;
    ctx->last_fused = fused;
    ctx->last_B = B;
    ctx->last_iou = iou_thr;
    ctx->detect_pending = true;
    ctx->align_replay = false;
    return FD_OK;
}

}  // namespace fd

using namespace fd;

FD_EXPORT int fd_letterbox_geometry(const fd_ctx *ctx, int img_h, int img_w, int *new_w, int *new_h, float *det_scale) {
    FD_REQUIRE(ctx && img_h > 0 && img_w > 0 && new_w && new_h && det_scale, "fd_letterbox_geometry: bad arguments");
    letterbox(img_h, img_w, ctx->cfg.image_w, ctx->cfg.image_h, new_w, new_h, det_scale);
    return FD_OK;
}

static int preprocess_batch(fd_ctx *ctx, FrameList frames, int B, float *out_nchw_dev, float *det_scale_host) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(B >= 0 && (B == 0 || (frames.any() && out_nchw_dev)), "fd_preprocess_batch: bad arguments");
    if (B == 0) return FD_OK;
    int mrb = 0;
    FD_TRY(upload_frame_table(ctx, frames, B, det_scale_host, &mrb));
    bool aligned = true;  // bulk-TMA staging needs 16-byte aligned rows that can be over-read to a 16-byte multiple
    auto row_ok = [](const uint8_t *p, int pitch, int row_bytes) {
        return reinterpret_cast<uintptr_t>(p) % 16 == 0 && pitch % 16 == 0 && ((row_bytes + 15) & ~15) <= pitch;
    };
    for (int i = 0; i < B; ++i) {
        if (frames.yuv) {   // planar: the second chroma plane starts whole pitches after the first
            const fd_frame_nv12 &f = frames.yuv[i];
            const bool planar = ctx->frames_fmt == SRC_PLANAR;
            aligned = aligned && row_ok(f.y, f.pitch_y, f.width) && row_ok(f.uv, f.pitch_uv, planar ? f.width / 2 : f.width);
        } else if (frames.packed) {
            aligned = aligned && row_ok(frames.packed[i].data, frames.packed[i].pitch, 2 * frames.packed[i].width);
        } else if (frames.rgb) {
            aligned = aligned && row_ok(frames.rgb[i].data, frames.rgb[i].pitch, rgb_bpp(frames.layout) * frames.rgb[i].width);
        } else {
            aligned = aligned && row_ok(frames.bgr[i].data, frames.bgr[i].pitch, frames.bgr[i].width * 3);
        }
    }
    return preprocess_launch(ctx, ctx->frames_dev.as<FrameDev>(), B, out_nchw_dev, mrb, aligned, ctx->frames_fmt);
}

FD_EXPORT int fd_preprocess_batch(fd_ctx *ctx, const fd_frame *frames, int B, float *out_nchw_dev, float *det_scale_host) {
    FrameList fl;
    fl.bgr = frames;
    return preprocess_batch(ctx, fl, B, out_nchw_dev, det_scale_host);
}
FD_EXPORT int fd_preprocess_batch_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, float *out_nchw_dev, float *det_scale_host) {
    FrameList fl;
    FD_TRY(yuv420_frames(frames, layout, &fl));
    return preprocess_batch(ctx, fl, B, out_nchw_dev, det_scale_host);
}
FD_EXPORT int fd_preprocess_batch_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, float *out_nchw_dev, float *det_scale_host) {
    return fd_preprocess_batch_yuv420(ctx, frames, FD_YUV420_NV12, B, out_nchw_dev, det_scale_host);
}
FD_EXPORT int fd_preprocess_batch_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, float *out_nchw_dev, float *det_scale_host) {
    FrameList fl;
    FD_TRY(yuv422_frames(frames, layout, &fl));
    return preprocess_batch(ctx, fl, B, out_nchw_dev, det_scale_host);
}
FD_EXPORT int fd_preprocess_batch_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, float *out_nchw_dev, float *det_scale_host) {
    FrameList fl;
    FD_TRY(rgb_frames(frames, layout, &fl));
    return preprocess_batch(ctx, fl, B, out_nchw_dev, det_scale_host);
}

FD_EXPORT int fd_detect_batch(fd_ctx *ctx, const float *const *heads_dev, int n_heads, int B, const float *det_scale_host,
                              float conf_thr, float iou_thr) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(heads_dev && det_scale_host && B > 0, "fd_detect_batch: bad arguments");
    FD_REQUIRE(n_heads == 3 * ctx->dcfg.n_strides, "fd_detect_batch: n_heads must be 3 * n_strides");
    for (int i = 0; i < n_heads; ++i) FD_REQUIRE(heads_dev[i], "fd_detect_batch: null head tensor");
    return detect_enqueue(ctx, heads_dev, B, det_scale_host, conf_thr, iou_thr);
}

FD_EXPORT int fd_detect_fetch(fd_ctx *ctx, int32_t *counts, float *det, float *landmarks, int cap_rows, int *total) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(ctx->last_B > 0, "fd_detect_fetch: no fd_detect_batch results");
    FD_TRY(detect_resolve(ctx));
    const int B = ctx->last_B;
    std::vector<int> off(B + 1);
    FD_CUDA(cudaMemcpyAsync(off.data(), ctx->out_offsets.p, sizeof(int) * (B + 1), cudaMemcpyDeviceToHost, ctx->stream));
    FD_TRY(wait_stream(ctx));
    const int tot = off[B];
    if (total) *total = tot;
    if (counts)
        for (int i = 0; i < B; ++i) counts[i] = off[i + 1] - off[i];
    if (tot > cap_rows && (det || landmarks)) return fail(FD_ERR_CAPACITY, "fd_detect_fetch: cap_rows too small");
    if (det && tot) FD_CUDA(cudaMemcpyAsync(det, ctx->out_det.p, sizeof(float) * 5 * (size_t)tot, cudaMemcpyDeviceToHost, ctx->stream));
    if (landmarks && tot)
        FD_CUDA(cudaMemcpyAsync(landmarks, ctx->out_lmk.p, sizeof(float) * 10 * (size_t)tot, cudaMemcpyDeviceToHost, ctx->stream));
    FD_TRY(wait_stream(ctx));
    return FD_OK;
}

FD_EXPORT int fd_detect_view(fd_ctx *ctx, fd_det_view *out) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(out && ctx->last_B > 0, "fd_detect_view: no results");
    FD_TRY(detect_resolve(ctx));
    out->counts_dev = ctx->keep_count.as<int32_t>();
    out->offsets_dev = ctx->out_offsets.as<int32_t>();
    out->det_dev = ctx->out_det.as<float>();
    out->landmarks_dev = ctx->out_lmk.as<float>();
    out->frame_idx_dev = ctx->out_frame_idx.as<int32_t>();
    out->candidates_dev = ctx->cand_count.as<int32_t>();
    return FD_OK;
}

FD_EXPORT int fd_detect_last_stats(fd_ctx *ctx, int32_t *out) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(out && ctx->last_B > 0, "fd_detect_last_stats: no fd_detect_batch results");
    const int B = ctx->last_B;
    int st[4] = {0, 0, 0, 0};
    std::vector<int> counts(B);
    FD_CUDA(cudaMemcpyAsync(st, ctx->status(), sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaMemcpyAsync(counts.data(), ctx->cand_count.p, sizeof(int) * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
    FD_TRY(wait_stream(ctx));
    long long tot = 0;
    int mx = 0;
    for (int c : counts) { tot += c; mx = std::max(mx, c); }
    memset(out, 0, sizeof(int32_t) * 8);
    out[0] = ctx->detect_pending ? st[1] : 0;   // once resolved, nothing is pending any more
    out[1] = mx;
    out[2] = (int32_t)std::min<long long>(tot, INT_MAX);
    out[3] = st[2];
    out[4] = ctx->last_fused ? 1 : 0;
    out[5] = ctx->crowded ? 1 : 0;
    return FD_OK;
}

static int align_batch(fd_ctx *ctx, FrameList frames, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                       const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(B > 0 && frames.any() && F >= 0 && (F == 0 || (landmarks_dev && crops_dev)), "fd_align_batch: bad arguments");
    if (F == 0) return FD_OK;
    FD_TRY(upload_frame_table(ctx, frames, B, nullptr, nullptr));
    WarpFallback fb;
    fb.bbox = bbox_dev;
    fb.bbox_stride = 4;
    return align_enqueue(ctx, landmarks_dev, frame_idx_dev, nullptr, F, crops_dev, M_dev, ok_dev, false, fb);
}

FD_EXPORT int fd_align_batch(fd_ctx *ctx, const fd_frame *frames, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                             const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FrameList fl;
    fl.bgr = frames;
    return align_batch(ctx, fl, B, landmarks_dev, frame_idx_dev, bbox_dev, F, crops_dev, M_dev, ok_dev);
}
FD_EXPORT int fd_align_batch_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                                  const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(yuv420_frames(frames, layout, &fl));
    return align_batch(ctx, fl, B, landmarks_dev, frame_idx_dev, bbox_dev, F, crops_dev, M_dev, ok_dev);
}
FD_EXPORT int fd_align_batch_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                                  const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    return fd_align_batch_yuv420(ctx, frames, FD_YUV420_NV12, B, landmarks_dev, frame_idx_dev, bbox_dev, F, crops_dev, M_dev, ok_dev);
}
FD_EXPORT int fd_align_batch_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                                    const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(yuv422_frames(frames, layout, &fl));
    return align_batch(ctx, fl, B, landmarks_dev, frame_idx_dev, bbox_dev, F, crops_dev, M_dev, ok_dev);
}
FD_EXPORT int fd_align_batch_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                                 const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(rgb_frames(frames, layout, &fl));
    return align_batch(ctx, fl, B, landmarks_dev, frame_idx_dev, bbox_dev, F, crops_dev, M_dev, ok_dev);
}

static int align_detections(fd_ctx *ctx, FrameList frames, int B, uint8_t *crops_dev, int cap_faces, double *M_dev, uint8_t *ok_dev) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(B > 0 && frames.any() && B == ctx->last_B && crops_dev && cap_faces > 0, "fd_align_detections: bad arguments");
    // No host synchronisation here: images needing the big NMS path are detected lazily at
    // fd_detect_fetch / fd_detect_view / fd_ctx-level fetch, which replays this align if the detections changed.
    FD_TRY(upload_frame_table(ctx, frames, B, nullptr, nullptr));
    ctx->align_replay = true;
    ctx->align_crops = crops_dev;
    ctx->align_cap = cap_faces;
    ctx->align_M_out = M_dev;
    ctx->align_ok_out = ok_dev;
    return align_enqueue(ctx, ctx->out_lmk.as<float>(), ctx->out_frame_idx.as<int32_t>(), ctx->status() + 2, cap_faces, crops_dev, M_dev,
                         ok_dev, true, detect_fallback(ctx));
}

FD_EXPORT int fd_align_detections(fd_ctx *ctx, const fd_frame *frames, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                                  uint8_t *ok_dev) {
    FrameList fl;
    fl.bgr = frames;
    return align_detections(ctx, fl, B, crops_dev, cap_faces, M_dev, ok_dev);
}
FD_EXPORT int fd_align_detections_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                                       uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(yuv420_frames(frames, layout, &fl));
    return align_detections(ctx, fl, B, crops_dev, cap_faces, M_dev, ok_dev);
}
FD_EXPORT int fd_align_detections_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                                       uint8_t *ok_dev) {
    return fd_align_detections_yuv420(ctx, frames, FD_YUV420_NV12, B, crops_dev, cap_faces, M_dev, ok_dev);
}
FD_EXPORT int fd_align_detections_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                                         uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(yuv422_frames(frames, layout, &fl));
    return align_detections(ctx, fl, B, crops_dev, cap_faces, M_dev, ok_dev);
}
FD_EXPORT int fd_align_detections_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                                      uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(rgb_frames(frames, layout, &fl));
    return align_detections(ctx, fl, B, crops_dev, cap_faces, M_dev, ok_dev);
}

// ---- single-image host wrappers -----------------------------------------------------------------------------------
static int upload_image(fd_ctx *ctx, int slot, const uint8_t *img, int h, int w, int pitch, const uint8_t **dev, int *dev_pitch) {
    FD_REQUIRE(img && h > 0 && w > 0 && pitch >= w * 3, "image: bad geometry");
    const int dp = (w * 3 + 15) & ~15;
    FD_TRY(ctx->scratch[slot].reserve((size_t)dp * h));
    FD_CUDA(cudaMemcpy2DAsync(ctx->scratch[slot].p, dp, img, pitch, (size_t)w * 3, h, cudaMemcpyHostToDevice, ctx->stream));
    *dev = ctx->scratch[slot].as<uint8_t>();
    *dev_pitch = dp;
    return FD_OK;
}

FD_EXPORT int fd_preprocess(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, float *out_nchw, float *det_scale) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(out_nchw, "fd_preprocess: null output");
    const uint8_t *d_img;
    int dp;
    FD_TRY(upload_image(ctx, 3, img, h, w, pitch, &d_img, &dp));
    fd_frame fr{d_img, h, w, dp};
    const size_t n = (size_t)3 * ctx->cfg.image_h * ctx->cfg.image_w;
    FD_TRY(ctx->scratch[4].reserve(sizeof(float) * n));
    float ds = 0.f;
    FD_TRY(fd_preprocess_batch(ctx, &fr, 1, ctx->scratch[4].as<float>(), &ds));
    if (det_scale) *det_scale = ds;
    FD_CUDA(cudaMemcpyAsync(out_nchw, ctx->scratch[4].p, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaStreamSynchronize(ctx->stream));
    return FD_OK;
}

FD_EXPORT int fd_resize_linear(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, uint8_t *out, int out_h, int out_w) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(out && out_h > 0 && out_w > 0, "fd_resize_linear: bad output size");
    const uint8_t *d_img;
    int dp;
    FD_TRY(upload_image(ctx, 3, img, h, w, pitch, &d_img, &dp));
    FrameDev f{};
    f.data = d_img; f.h = h; f.w = w; f.pitch = dp; f.new_w = out_w; f.new_h = out_h;
    f.scale_x = 1.0 / ((double)out_w / w);
    f.scale_y = 1.0 / ((double)out_h / h);
    const size_t n = (size_t)out_h * out_w * 3;
    FD_TRY(ctx->scratch[4].reserve(n));
    FD_TRY(resize_launch(ctx, f, ctx->scratch[4].as<uint8_t>(), out_h, out_w));
    FD_CUDA(cudaMemcpyAsync(out, ctx->scratch[4].p, n, cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaStreamSynchronize(ctx->stream));
    return FD_OK;
}

FD_EXPORT int fd_detect(fd_ctx *ctx, const float *const *heads, int n_heads, float det_scale, float conf_thr, float iou_thr,
                        float *det, float *landmarks, int cap, int *num_det) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(heads && num_det && n_heads == 3 * ctx->dcfg.n_strides, "fd_detect: bad arguments");
    const DecodeCfg &d = ctx->dcfg;
    const float *dev_heads[3 * FD_MAX_STRIDES];
    for (int s = 0; s < d.n_strides; ++s) {
        const int hw = d.fh[s] * d.fw[s];
        const int ch[3] = {2 * d.A, 4 * d.A, 10 * d.A};
        for (int k = 0; k < 3; ++k) {
            FD_REQUIRE(heads[3 * s + k], "fd_detect: null head tensor");
            const size_t bytes = sizeof(float) * (size_t)ch[k] * hw;
            FD_TRY(ctx->pipe_heads[3 * s + k].reserve(bytes));
            FD_CUDA(cudaMemcpyAsync(ctx->pipe_heads[3 * s + k].p, heads[3 * s + k], bytes, cudaMemcpyHostToDevice, ctx->stream));
            dev_heads[3 * s + k] = ctx->pipe_heads[3 * s + k].as<float>();
        }
    }
    FD_TRY(detect_enqueue(ctx, dev_heads, 1, &det_scale, conf_thr, iou_thr));
    int32_t cnt = 0;
    int tot = 0;
    FD_TRY(fd_detect_fetch(ctx, &cnt, det, landmarks, cap, &tot));
    *num_det = tot;
    return FD_OK;
}

FD_EXPORT int fd_estimate_affine_partial_2d(fd_ctx *ctx, const float *from, const float *to, int n_sets, double *M, uint8_t *ok) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(n_sets >= 0 && (n_sets == 0 || (from && M && ok)), "fd_estimate_affine_partial_2d: bad arguments");
    if (n_sets == 0) return FD_OK;
    const size_t nb = sizeof(float) * 10 * (size_t)n_sets;
    FD_TRY(ctx->scratch[0].reserve(nb));
    FD_CUDA(cudaMemcpyAsync(ctx->scratch[0].p, from, nb, cudaMemcpyHostToDevice, ctx->stream));
    const float *d_to = nullptr;
    if (to) {
        FD_TRY(ctx->scratch[1].reserve(nb));
        FD_CUDA(cudaMemcpyAsync(ctx->scratch[1].p, to, nb, cudaMemcpyHostToDevice, ctx->stream));
        d_to = ctx->scratch[1].as<float>();
    }
    ctx->est_valid = false;   // align_M / align_ok are reused as scratch here
    FD_TRY(ctx->align_M.reserve(sizeof(double) * 12 * (size_t)n_sets));
    FD_TRY(ctx->align_ok.reserve((size_t)n_sets));
    FD_TRY(ctx->scratch[2].reserve(sizeof(double) * 6 * (size_t)n_sets));
    FD_TRY(estimate_launch(ctx, ctx->scratch[0].as<float>(), d_to, nullptr, n_sets, ctx->align_M.as<double>(),
                           ctx->scratch[2].as<double>(), ctx->align_ok.as<uint8_t>(), nullptr));
    FD_CUDA(cudaMemcpyAsync(M, ctx->scratch[2].p, sizeof(double) * 6 * (size_t)n_sets, cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaMemcpyAsync(ok, ctx->align_ok.p, (size_t)n_sets, cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaStreamSynchronize(ctx->stream));
    return FD_OK;
}

// M given (fd_warp_affine) or estimated from lmk (fd_align; bbox = the fallback's box, face_alignment.rs:64-116)
static int warp_host(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, const double *M, const float *lmk, const float *bbox,
                     uint8_t *out, int out_h, int out_w, double *M_out, int *mode_out) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(out && out_h > 0 && out_w > 0 && out_w <= 4096, "warp: bad output size");
    const uint8_t *d_img;
    int dp;
    FD_TRY(upload_image(ctx, 3, img, h, w, pitch, &d_img, &dp));
    FD_TRY(ctx->pinned[2].reserve(sizeof(FrameDev)));
    FD_CUDA(cudaEventSynchronize(ctx->ev[2]));
    FrameDev *f = ctx->pinned[2].as<FrameDev>();
    memset(f, 0, sizeof(*f));
    f->data = d_img; f->h = h; f->w = w; f->pitch = dp;
    FD_TRY(ctx->scratch[5].reserve(sizeof(FrameDev)));
    FD_CUDA(cudaMemcpyAsync(ctx->scratch[5].p, f, sizeof(FrameDev), cudaMemcpyHostToDevice, ctx->stream));
    FD_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    ctx->est_valid = false;
    FD_TRY(ctx->align_M.reserve(sizeof(double) * 12));
    FD_TRY(ctx->align_ok.reserve(16));
    FD_TRY(ctx->scratch[0].reserve(64 + sizeof(float) * 10 + sizeof(float) * 4 + 16));   // M or landmarks | bbox | mode
    unsigned char *sc0 = ctx->scratch[0].as<unsigned char>();
    if (M) {
        FD_CUDA(cudaMemcpyAsync(sc0, M, sizeof(double) * 6, cudaMemcpyHostToDevice, ctx->stream));
        FD_TRY(invert_launch(ctx, reinterpret_cast<double *>(sc0), 1, ctx->align_M.as<double>(), ctx->align_ok.as<uint8_t>()));
    } else {
        FD_CUDA(cudaMemcpyAsync(sc0, lmk, sizeof(float) * 10, cudaMemcpyHostToDevice, ctx->stream));
        FD_TRY(estimate_launch(ctx, reinterpret_cast<float *>(sc0), nullptr, nullptr, 1, ctx->align_M.as<double>(), nullptr,
                               ctx->align_ok.as<uint8_t>(), nullptr));
    }
    WarpFallback fb;
    if (bbox) {
        FD_CUDA(cudaMemcpyAsync(sc0 + 64, bbox, sizeof(float) * 4, cudaMemcpyHostToDevice, ctx->stream));
        fb.bbox = reinterpret_cast<float *>(sc0 + 64);
    }
    fb.mode_out = sc0 + 64 + 16;
    const size_t n = (size_t)out_h * out_w * 3;
    FD_TRY(ctx->scratch[4].reserve(n));
    FD_TRY(warp_launch(ctx, ctx->scratch[5].as<FrameDev>(), nullptr, ctx->align_M.as<double>(), ctx->align_ok.as<uint8_t>(), nullptr, 1,
                       ctx->scratch[4].as<uint8_t>(), out_w, out_h, fb, SRC_BGR));
    uint8_t mode = 0;
    double M12[12];
    FD_CUDA(cudaMemcpyAsync(out, ctx->scratch[4].p, n, cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaMemcpyAsync(&mode, fb.mode_out, 1, cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaMemcpyAsync(M12, ctx->align_M.p, sizeof(M12), cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaStreamSynchronize(ctx->stream));
    if (M_out && mode == 1) memcpy(M_out, M12, sizeof(double) * 6);
    if (mode_out) *mode_out = mode;
    if (!mode)
        return fail(FD_ERR_ESTIMATE, "fd_align: empty transform and the fallback crop (x0,y0)..(max(x2+22,W), max(y1+22,H)) is not inside "
                                     "the image (the reference returns Err from Mat::roi, face_alignment.rs:92-95)");
    return FD_OK;
}

FD_EXPORT int fd_warp_affine(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, const double *M, uint8_t *out, int out_h,
                             int out_w) {
    FD_REQUIRE(M, "fd_warp_affine: null M");
    return warp_host(ctx, img, h, w, pitch, M, nullptr, nullptr, out, out_h, out_w, nullptr, nullptr);
}
FD_EXPORT int fd_align(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, const float *bbox, const float *landmarks, uint8_t *crop,
                       double *M_out, int *mode_out) {
    // landmarks == None: array2_to_mat is skipped, cv::estimateAffinePartial2D asserts on the empty Mat and call() returns Err
    FD_REQUIRE(ctx && landmarks, "fd_align: landmarks == None (the reference returns Err: estimateAffinePartial2D on an empty Mat)");
    return warp_host(ctx, img, h, w, pitch, nullptr, landmarks, bbox, crop, ctx->cfg.crop_h, ctx->cfg.crop_w, M_out, mode_out);
}

// ---- N1: post-align model preprocessors ------------------------------------------------------------------------------
FD_EXPORT int fd_crops_to_tensor(fd_ctx *ctx, const uint8_t *crops_dev, int F, int in_h, int in_w, int out_h, int out_w,
                                 const float *mean_rgb, const float *mul_rgb, float *out_nchw_dev, int use_detect_count) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(F >= 0 && in_h > 0 && in_w > 0 && out_h > 0 && out_w > 0 && mean_rgb && mul_rgb, "fd_crops_to_tensor: bad arguments");
    FD_REQUIRE(F == 0 || (crops_dev && out_nchw_dev), "fd_crops_to_tensor: null buffers");
    FD_REQUIRE(!use_detect_count || ctx->last_B > 0, "fd_crops_to_tensor: no fd_detect_batch results to take the face count from");
    return crops_to_tensor_launch(ctx, crops_dev, use_detect_count ? ctx->status() + 2 : nullptr, F, in_h, in_w, out_h, out_w,
                                  mean_rgb, mul_rgb, out_nchw_dev);
}

FD_EXPORT int fd_model_preprocess(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, int out_h, int out_w,
                                  const float *mean_rgb, const float *mul_rgb, float *out_nchw) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(img && out_nchw && h > 0 && w > 0 && pitch >= w * 3 && out_h > 0 && out_w > 0 && mean_rgb && mul_rgb,
               "fd_model_preprocess: bad arguments");
    FD_TRY(ctx->scratch[3].reserve((size_t)h * w * 3));
    FD_CUDA(cudaMemcpy2DAsync(ctx->scratch[3].p, (size_t)w * 3, img, pitch, (size_t)w * 3, h, cudaMemcpyHostToDevice, ctx->stream));
    const size_t n = (size_t)3 * out_h * out_w;
    FD_TRY(ctx->scratch[4].reserve(sizeof(float) * n));
    FD_TRY(crops_to_tensor_launch(ctx, ctx->scratch[3].as<uint8_t>(), nullptr, 1, h, w, out_h, out_w, mean_rgb, mul_rgb,
                                  ctx->scratch[4].as<float>()));
    FD_CUDA(cudaMemcpyAsync(out_nchw, ctx->scratch[4].p, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaStreamSynchronize(ctx->stream));
    return FD_OK;
}

// ---- N2: raw_output_contents -> decode --------------------------------------------------------------------------------
FD_EXPORT int fd_detect_batch_raw(fd_ctx *ctx, const uint8_t *const *raw, const size_t *nbytes, const int64_t (*shape)[4], int n_heads,
                                  const float *det_scale_host, float conf_thr, float iou_thr) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(raw && nbytes && shape && det_scale_host, "fd_detect_batch_raw: bad arguments");
    const DecodeCfg &d = ctx->dcfg;
    FD_REQUIRE(n_heads == 3 * d.n_strides, "fd_detect_batch_raw: n_heads must be 3 * n_strides");
    const int64_t B = shape[0][0];
    FD_REQUIRE(B > 0 && B <= (1 << 20), "fd_detect_batch_raw: bad batch dimension");
    const float *dev_heads[3 * FD_MAX_STRIDES];
    for (int s = 0; s < d.n_strides; ++s) {
        const int ch[3] = {2 * d.A, 4 * d.A, 10 * d.A};
        for (int k = 0; k < 3; ++k) {
            const int i = 3 * s + k;
            FD_REQUIRE(raw[i], "fd_detect_batch_raw: null output");
            const int64_t *sh = shape[i];
            const int64_t n = sh[0] * sh[1] * sh[2] * sh[3];
            // Array4::from_shape_vec(dims, u8_to_f32_vec(bytes)): chunks_exact(4) drops a trailing partial element
            FD_REQUIRE(sh[0] > 0 && sh[1] > 0 && sh[2] > 0 && sh[3] > 0 && (int64_t)(nbytes[i] / 4) == n,
                       "fd_detect_batch_raw: shape does not match the byte length (ShapeError in the reference)");
            FD_REQUIRE(sh[0] == B && sh[1] == ch[k] && sh[2] == d.fh[s] && sh[3] == d.fw[s],
                       "fd_detect_batch_raw: output shape does not match the detector geometry");
            const size_t bytes = sizeof(float) * (size_t)n;
            FD_TRY(ctx->pipe_heads[i].reserve(bytes));
            FD_CUDA(cudaMemcpyAsync(ctx->pipe_heads[i].p, raw[i], bytes, cudaMemcpyHostToDevice, ctx->stream));
            dev_heads[i] = ctx->pipe_heads[i].as<float>();
        }
    }
    return detect_enqueue(ctx, dev_heads, (int)B, det_scale_host, conf_thr, iou_thr);
}

// ---- N3: FaceSelection -----------------------------------------------------------------------------------------------
FD_EXPORT int fd_select_params_default(fd_select_params *p) {
    FD_REQUIRE(p, "fd_select_params_default: null");
    p->margin_center_left_ratio = 0.3f;    // face_pipeline/config.rs:110-113
    p->margin_center_right_ratio = 0.3f;
    p->margin_edge_ratio = 0.1f;
    p->minimum_face_ratio = 0.0075f;
    return FD_OK;
}

FD_EXPORT int fd_face_selection(fd_ctx *ctx, int img_h, int img_w, const float *face_boxes, const float *key_points, int M, int is_enroll,
                                const fd_select_params *params, int *box_index, int *kp_index) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(img_h > 0 && img_w > 0 && M >= 0 && (M == 0 || face_boxes) && box_index && kp_index, "fd_face_selection: bad arguments");
    fd_select_params p;
    if (params) p = *params;
    else FD_TRY(fd_select_params_default(&p));
    const size_t nb = sizeof(float) * 5 * (size_t)std::max(M, 1), nl = sizeof(float) * 10 * (size_t)std::max(M, 1);
    FD_TRY(ctx->scratch[0].reserve(nb));
    FD_TRY(ctx->scratch[1].reserve(nl));
    FD_TRY(ctx->scratch[2].reserve(sizeof(FrameDev) + 4 * sizeof(int)));
    if (M) FD_CUDA(cudaMemcpyAsync(ctx->scratch[0].p, face_boxes, sizeof(float) * 5 * (size_t)M, cudaMemcpyHostToDevice, ctx->stream));
    if (M && key_points) FD_CUDA(cudaMemcpyAsync(ctx->scratch[1].p, key_points, sizeof(float) * 10 * (size_t)M, cudaMemcpyHostToDevice, ctx->stream));
    struct { FrameDev f; int off[2]; int sel[2]; } h;
    memset(&h, 0, sizeof(h));
    h.f.h = img_h; h.f.w = img_w;
    h.off[0] = 0; h.off[1] = M;
    FD_CUDA(cudaMemcpyAsync(ctx->scratch[2].p, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    unsigned char *base = ctx->scratch[2].as<unsigned char>();
    FD_TRY(select_launch(ctx, reinterpret_cast<int *>(base + offsetof(decltype(h), off)), ctx->scratch[0].as<float>(),
                         key_points ? ctx->scratch[1].as<float>() : nullptr, reinterpret_cast<FrameDev *>(base), 1, &p, is_enroll,
                         reinterpret_cast<int *>(base + offsetof(decltype(h), sel)), nullptr, nullptr));
    int sel[2];
    FD_CUDA(cudaMemcpyAsync(sel, base + offsetof(decltype(h), sel), sizeof(sel), cudaMemcpyDeviceToHost, ctx->stream));
    FD_CUDA(cudaStreamSynchronize(ctx->stream));
    *box_index = sel[0];
    *kp_index = sel[1];
    return FD_OK;
}

static int select_detections(fd_ctx *ctx, FrameList frames, int B, int is_enroll, const fd_select_params *params, int32_t *sel_host) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(frames.any() && B > 0 && B == ctx->last_B, "fd_select_detections: needs the frames of the last fd_detect_batch");
    if (sel_host) FD_TRY(detect_resolve(ctx));
    fd_select_params p;
    if (params) p = *params;
    else FD_TRY(fd_select_params_default(&p));
    FD_TRY(upload_frame_table(ctx, frames, B, nullptr, nullptr));
    FD_TRY(ctx->select_sel.reserve(sizeof(int) * 2 * (size_t)B));
    FD_TRY(ctx->select_lmk.reserve(sizeof(float) * 10 * (size_t)B));
    FD_TRY(ctx->select_fidx.reserve(sizeof(int) * (size_t)B));
    FD_TRY(select_launch(ctx, ctx->out_offsets.as<int>(), ctx->out_det.as<float>(), ctx->out_lmk.as<float>(), ctx->frames_dev.as<FrameDev>(), B,
                         &p, is_enroll, ctx->select_sel.as<int>(), ctx->select_lmk.as<float>(), ctx->select_fidx.as<int>()));
    ctx->select_B = B;
    if (sel_host) {
        FD_CUDA(cudaMemcpyAsync(sel_host, ctx->select_sel.p, sizeof(int) * 2 * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
        FD_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return FD_OK;
}

FD_EXPORT int fd_select_detections(fd_ctx *ctx, const fd_frame *frames, int B, int is_enroll, const fd_select_params *params, int32_t *sel_host) {
    FrameList fl;
    fl.bgr = frames;
    return select_detections(ctx, fl, B, is_enroll, params, sel_host);
}
FD_EXPORT int fd_select_detections_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, int is_enroll, const fd_select_params *params,
                                        int32_t *sel_host) {
    FrameList fl;
    FD_TRY(yuv420_frames(frames, layout, &fl));
    return select_detections(ctx, fl, B, is_enroll, params, sel_host);
}
FD_EXPORT int fd_select_detections_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, int is_enroll, const fd_select_params *params,
                                        int32_t *sel_host) {
    return fd_select_detections_yuv420(ctx, frames, FD_YUV420_NV12, B, is_enroll, params, sel_host);
}
FD_EXPORT int fd_select_detections_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, int is_enroll, const fd_select_params *params,
                                          int32_t *sel_host) {
    FrameList fl;
    FD_TRY(yuv422_frames(frames, layout, &fl));
    return select_detections(ctx, fl, B, is_enroll, params, sel_host);
}
FD_EXPORT int fd_select_detections_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, int is_enroll, const fd_select_params *params,
                                       int32_t *sel_host) {
    FrameList fl;
    FD_TRY(rgb_frames(frames, layout, &fl));
    return select_detections(ctx, fl, B, is_enroll, params, sel_host);
}

static int align_selected(fd_ctx *ctx, FrameList frames, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(frames.any() && B > 0 && B == ctx->select_B && crops_dev,
               "fd_align_selected: needs the frames of the last fd_select_detections");
    FD_TRY(upload_frame_table(ctx, frames, B, nullptr, nullptr));
    // Images without a selection (or whose selection has no key points) carry NaN key points: the estimate fails there and,
    // as the reference's call(&image, box, None) errs on the empty landmark Mat, the crop is zero-filled with ok = 0; a
    // selection whose key points are degenerate takes the bbox-crop fallback on its selected box (ok = 2).
    WarpFallback fb = detect_fallback(ctx);
    fb.sel = ctx->select_sel.as<int>();
    return align_enqueue(ctx, ctx->select_lmk.as<float>(), ctx->select_fidx.as<int32_t>(), nullptr, B, crops_dev, M_dev, ok_dev, false, fb);
}

FD_EXPORT int fd_align_selected(fd_ctx *ctx, const fd_frame *frames, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FrameList fl;
    fl.bgr = frames;
    return align_selected(ctx, fl, B, crops_dev, M_dev, ok_dev);
}
FD_EXPORT int fd_align_selected_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(yuv420_frames(frames, layout, &fl));
    return align_selected(ctx, fl, B, crops_dev, M_dev, ok_dev);
}
FD_EXPORT int fd_align_selected_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    return fd_align_selected_yuv420(ctx, frames, FD_YUV420_NV12, B, crops_dev, M_dev, ok_dev);
}
FD_EXPORT int fd_align_selected_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(yuv422_frames(frames, layout, &fl));
    return align_selected(ctx, fl, B, crops_dev, M_dev, ok_dev);
}
FD_EXPORT int fd_align_selected_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev) {
    FrameList fl;
    FD_TRY(rgb_frames(frames, layout, &fl));
    return align_selected(ctx, fl, B, crops_dev, M_dev, ok_dev);
}

// ---- end-to-end with host buffers ------------------------------------------------------------------------------------
namespace fd {

// Host replica of y_taps (fd_resize.cuh): the one or two source rows destination row dy of cv::resize reads.
static void host_y_rows(int dy, double scale_y, int sh, int *y0, int *y1, bool *two) {
    volatile float fy = (float)(((double)dy + 0.5) * scale_y - 0.5);
    const int sy = (int)floorf(fy);
    volatile float fr = fy - (float)sy;
    volatile float w1 = fr * 2048.0f;
    const long b1 = lrintf(w1);   // cvRound: round-half-even in the default rounding mode
    *y0 = std::min(std::max(sy, 0), sh - 1);
    *y1 = std::min(std::max(sy + 1, 0), sh - 1);
    *two = b1 != 0;
}

static int sat_int_rn(double v) {   // __double2int_rn: round-half-even, saturating, NaN -> 0
    if (!(v == v)) return 0;
    const double r = nearbyint(v);
    if (r >= 2147483647.0) return 2147483647;
    if (r <= -2147483648.0) return (-2147483647 - 1);
    return (int)r;
}

// Source pixel rectangle [x0,x1] x [y0,y1] (inclusive, clipped to the frame) the fixed-point warp of one face reads:
// the tap coordinates of warp_fixed_kernel / warp_kernel are monotone in x and in y, so their extremes are at the crop's
// corners; +1 for the second tap of each axis.  Returns false when the crop reads nothing inside the frame.
static bool warp_source_rect(const double *iM, int cw, int ch, int fw, int fh, int *x0, int *y0, int *x1, int *y1) {
    long long lx = (1ll << 40), ly = (1ll << 40), hx = -(1ll << 40), hy = -(1ll << 40);
    const int xs[2] = {0, cw - 1}, ys[2] = {0, ch - 1};
    for (int cy = 0; cy < 2; ++cy)
        for (int cx = 0; cx < 2; ++cx) {
            const int X0 = sat_int_rn((iM[1] * ys[cy] + iM[2]) * 1024) + 16, Y0 = sat_int_rn((iM[4] * ys[cy] + iM[5]) * 1024) + 16;
            const int dx = sat_int_rn(iM[0] * xs[cx] * 1024), dy = sat_int_rn(iM[3] * xs[cx] * 1024);
            const int X = (int)((unsigned)X0 + (unsigned)dx) >> 5, Y = (int)((unsigned)Y0 + (unsigned)dy) >> 5;
            const long long sx = X >> 5, sy = Y >> 5;
            lx = std::min(lx, sx); hx = std::max(hx, sx + 1);
            ly = std::min(ly, sy); hy = std::max(hy, sy + 1);
        }
    lx = std::max<long long>(lx, 0); ly = std::max<long long>(ly, 0);
    hx = std::min<long long>(hx, fw - 1); hy = std::min<long long>(hy, fh - 1);
    if (lx > hx || ly > hy) return false;
    *x0 = (int)lx; *y0 = (int)ly; *x1 = (int)hx; *y1 = (int)hy;
    return true;
}

// rows first + step * j, j < count, of one plane
struct RowRun {
    int first, step, count;
};

// One plane of a host frame and its copy in the device arena.  Frame row y lies in plane row y >> ys; frame columns
// [x0, x1] lie in plane bytes [unit * (x0 >> xs), unit * ((x1 >> xs) + 1)).
struct HostPlane {
    const uint8_t *src;
    int spitch;
    size_t off;                 // offset in the device arena
    int dpitch;                 // 16-byte multiple
    int row_bytes, rows, xs, unit, ys;
    bool joined;                // the next plane follows this one, in host and in device memory: a whole-frame copy takes both
    std::vector<RowRun> have;   // rows on the device when the frame is not full (disjoint runs of one step)
};

struct HostFrame {
    int h, w;
    bool full;   // every plane is on the device
    int np;
    HostPlane pl[3];
};

static HostPlane host_plane(const uint8_t *src, int spitch, int row_bytes, int rows, int xs, int unit, int ys, size_t *arena) {
    HostPlane p;
    p.src = src;
    p.spitch = spitch;
    p.dpitch = (row_bytes + 15) & ~15;
    p.off = *arena;
    p.row_bytes = row_bytes;
    p.rows = rows;
    p.xs = xs;
    p.unit = unit;
    p.ys = ys;
    p.joined = false;
    *arena += ((size_t)p.dpitch * rows + 255) & ~(size_t)255;
    return p;
}

// the planes of host frame i (validated by fill_frame_of) and their places in the arena, each plane at a 256-byte aligned
// start with a 16-byte multiple pitch (bulk-copy preprocess, interior warp reads): BGR / RGB24 3w, RGBA / BGRA 4w, GRAY8 w,
// packed 4:2:2 2w (whole macropixels), NV12 / NV21 a Y plane of w and h/2 chroma rows of w (U,V pairs), I420 / YV12 a Y plane
// of w and the two chroma planes at round16(w/2), the second (h/2) pitches after the first as the descriptor wants it.
static void host_planes(const FrameList &frames, int i, HostFrame *hf, size_t *arena) {
    hf->full = false;
    if (frames.yuv) {
        const fd_frame_nv12 &f = frames.yuv[i];
        hf->h = f.height;
        hf->w = f.width;
        hf->np = 2;
        hf->pl[0] = host_plane(f.y, f.pitch_y, f.width, f.height, 0, 1, 0, arena);
        if (yuv420_format(frames.layout) != SRC_PLANAR) {
            hf->pl[1] = host_plane(f.uv, f.pitch_uv, f.width, f.height / 2, 1, 2, 1, arena);
            return;
        }
        HostPlane both = host_plane(f.uv, f.pitch_uv, f.width / 2, f.height, 1, 1, 1, arena);
        both.rows = f.height / 2;
        both.joined = true;
        hf->pl[1] = hf->pl[2] = both;
        hf->pl[2].src += (size_t)both.rows * f.pitch_uv;
        hf->pl[2].off += (size_t)both.rows * both.dpitch;
        hf->pl[2].joined = false;
        hf->np = 3;
        return;
    }
    const fd_frame &f = frames.packed ? frames.packed[i] : frames.rgb ? frames.rgb[i] : frames.bgr[i];
    hf->h = f.height;
    hf->w = f.width;
    hf->np = 1;
    if (frames.packed) hf->pl[0] = host_plane(f.data, f.pitch, 2 * f.width, f.height, 1, 4, 0, arena);
    else {
        const int bpp = frames.rgb ? rgb_bpp(frames.layout) : 3;
        hf->pl[0] = host_plane(f.data, f.pitch, bpp * f.width, f.height, 0, bpp, 0, arena);
    }
}

// rows first + step * j (j < count) of plane p, host to device: one copy
static int upload_rows(fd_ctx *ctx, const HostPlane &p, uint8_t *arena, int first, int step, int count, int64_t *h2d) {
    if (count <= 0) return FD_OK;
    uint8_t *dst = arena + p.off + (size_t)first * p.dpitch;
    const uint8_t *src = p.src + (size_t)first * p.spitch;
    if (step == 1 && p.spitch == p.dpitch)
        FD_CUDA(cudaMemcpyAsync(dst, src, (size_t)p.dpitch * (count - 1) + p.row_bytes, cudaMemcpyHostToDevice, ctx->stream));
    else
        FD_CUDA(cudaMemcpy2DAsync(dst, (size_t)step * p.dpitch, src, (size_t)step * p.spitch, p.row_bytes, count, cudaMemcpyHostToDevice,
                                  ctx->stream));
    *h2d += (int64_t)p.row_bytes * count;
    return FD_OK;
}

// whole frame: one copy a plane (the two chroma planes of I420 / YV12 as one)
static int upload_full(fd_ctx *ctx, HostFrame &hf, uint8_t *arena, int64_t *h2d) {
    for (int q = 0; q < hf.np; ++q) {
        HostPlane p = hf.pl[q];
        if (p.joined) p.rows += hf.pl[++q].rows;
        FD_TRY(upload_rows(ctx, p, arena, 0, 1, p.rows, h2d));
    }
    hf.full = true;
    return FD_OK;
}

// adds the run to p.have; false when it overlaps a run already there without being the same
static bool add_run(HostPlane &p, RowRun r) {
    if (r.count <= 0) return true;
    for (const RowRun &o : p.have) {
        if (o.first == r.first && o.count == r.count && o.step == r.step) return true;
        if (o.step != r.step) return false;
        const bool same_rows = (o.first - r.first) % r.step == 0;
        if (same_rows && r.first <= o.first + o.step * (o.count - 1) && o.first <= r.first + r.step * (r.count - 1)) return false;
    }
    p.have.push_back(r);
    return true;
}

// Only the source rows the letterbox resize reads (face_detection.rs:156): for an integer down-scale k they form at most two
// arithmetic progressions of stride k (1080p -> 640x360: rows 3y+1; 4K: rows 6y+2 and 6y+3), each ONE strided 2-D copy a
// plane.  A 4:2:0 chroma plane holds rows y >> 1 of them: two progressions of stride k for an odd k (1080p: chroma rows 3m and
// 3m+2), one of stride k/2 for an even k (4K: chroma rows 3y+1).  Returns *done = false when the pattern is not worth it (most
// rows needed, or no short description): the caller uploads the frame.
static int upload_preprocess_rows(fd_ctx *ctx, HostFrame &hf, int new_h, double scale_y, uint8_t *arena, int64_t *h2d, bool *done) {
    *done = false;
    const int h = hf.h;
    const long long k = llround(scale_y);
    if (k < 2 || fabs(scale_y - (double)k) > 1e-12 || new_h < 2) return FD_OK;
    // rows of dy = 0 and their stride-k continuation must reproduce every dy's rows
    int a0, a1, c0, c1;
    bool two0, two;
    host_y_rows(0, scale_y, h, &a0, &a1, &two0);
    for (int dy = 1; dy < new_h; ++dy) {
        host_y_rows(dy, scale_y, h, &c0, &c1, &two);
        if (two != two0 || c0 != a0 + (int)k * dy || (two && c1 != a1 + (int)k * dy)) return FD_OK;
    }
    if (two0 && k < 3) return FD_OK;
    const RowRun luma[2] = {{a0, (int)k, new_h}, {a1, (int)k, new_h}};
    for (int q = 0; q < hf.np; ++q) {
        HostPlane &p = hf.pl[q];
        p.have.clear();
        for (int t = 0; t < (two0 ? 2 : 1); ++t) {
            const RowRun &r = luma[t];
            bool ok;
            if (!p.ys) ok = add_run(p, r);
            else if (r.step % 2 == 0) ok = add_run(p, {r.first >> 1, r.step / 2, r.count});
            else ok = add_run(p, {r.first >> 1, r.step, (r.count + 1) / 2}) && add_run(p, {(r.first + r.step) >> 1, r.step, r.count / 2});
            if (!ok) return FD_OK;
        }
    }
    for (int q = 0; q < hf.np; ++q)
        for (const RowRun &r : hf.pl[q].have) FD_TRY(upload_rows(ctx, hf.pl[q], arena, r.first, r.step, r.count, h2d));
    *done = true;
    return FD_OK;
}

// bytes of the frame's rows already on the device (upload_preprocess_rows)
static int64_t have_bytes(const HostFrame &hf) {
    int64_t n = 0;
    for (int q = 0; q < hf.np; ++q)
        for (const RowRun &r : hf.pl[q].have) n += (int64_t)hf.pl[q].row_bytes * r.count;
    return n;
}

// the rows upload_preprocess_rows left out: per plane and residue of the runs' step, the gaps between the runs
static int upload_complement_rows(fd_ctx *ctx, HostFrame &hf, uint8_t *arena, int64_t *h2d) {
    for (int q = 0; q < hf.np; ++q) {
        const HostPlane &p = hf.pl[q];
        const int s = p.have[0].step;
        std::vector<RowRun> runs = p.have;
        std::sort(runs.begin(), runs.end(), [](const RowRun &a, const RowRun &b) { return a.first < b.first; });
        for (int res = 0; res < s && res < p.rows; ++res) {
            int next = res;   // the first row of this residue not yet accounted for
            for (const RowRun &r : runs) {
                if (r.first % s != res) continue;
                FD_TRY(upload_rows(ctx, p, arena, next, s, (r.first - next) / s, h2d));
                next = r.first + s * r.count;
            }
            FD_TRY(upload_rows(ctx, p, arena, next, s, (p.rows - next + s - 1) / s, h2d));
        }
    }
    hf.full = true;
    return FD_OK;
}

// Plane bytes the warp of pixel rectangle [x0,x1] x [y0,y1] reads; upload them when `arena` is given
static int upload_rect(fd_ctx *ctx, const HostFrame &hf, int x0, int y0, int x1, int y1, uint8_t *arena, int64_t *bytes) {
    for (int q = 0; q < hf.np; ++q) {
        const HostPlane &p = hf.pl[q];
        const int r0 = y0 >> p.ys, rows = (y1 >> p.ys) - r0 + 1;
        const size_t b0 = (size_t)p.unit * (x0 >> p.xs), wbytes = (size_t)p.unit * ((x1 >> p.xs) + 1) - b0;
        if (arena)
            FD_CUDA(cudaMemcpy2DAsync(arena + p.off + (size_t)r0 * p.dpitch + b0, p.dpitch, p.src + (size_t)r0 * p.spitch + b0, p.spitch,
                                      wbytes, rows, cudaMemcpyHostToDevice, ctx->stream));
        *bytes += (int64_t)wbytes * rows;
    }
    return FD_OK;
}

}  // namespace fd

FD_EXPORT int fd_pipeline_opts_default(fd_pipeline_opts *o) {
    FD_REQUIRE(o, "fd_pipeline_opts_default: null");
    memset(o, 0, sizeof(*o));
    return fd_select_params_default(&o->select_params);
}

// frames: HOST pixel frames in any layout, or (dev_frames != nullptr) BGR frames already resident on the device
// (fd_decode_jpeg_batch)
static int pipeline_host_impl(fd_ctx *ctx, FrameList frames, const fd_frame *dev_frames, int B, const float *const *heads_host, int n_heads,
                              float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out, int64_t h2d_so_far) {
    FD_REQUIRE(heads_host && out && B > 0, "fd_pipeline_host: bad arguments");
    FD_REQUIRE(n_heads == 3 * ctx->dcfg.n_strides, "fd_pipeline_host: n_heads must be 3 * n_strides");
    FD_REQUIRE(out->counts && out->det && out->landmarks && out->crops && out->cap_rows > 0, "fd_pipeline_host: bad outputs");
    fd_pipeline_opts o;
    if (opts) o = *opts;
    else FD_TRY(fd_pipeline_opts_default(&o));
    const bool select = o.select != 0, demand = o.upload == FD_UPLOAD_ON_DEMAND && !dev_frames;
    struct BlockingScope {   // sleep, do not spin, while this call waits on PCIe
        fd_ctx *c; bool prev;
        explicit BlockingScope(fd_ctx *c_) : c(c_), prev(c_->blocking_sync) { c->blocking_sync = true; }
        ~BlockingScope() { c->blocking_sync = prev; }
    } blocking_scope(ctx);
    FD_REQUIRE(!select || out->cap_rows >= B, "fd_pipeline_host: select mode writes one crop per image (cap_rows >= B)");
    const DecodeCfg &d = ctx->dcfg;
    const int cw = ctx->cfg.crop_w, ch = ctx->cfg.crop_h;
    int64_t h2d = h2d_so_far, d2h = 0;
    // 1. frames H2D into one device arena (host_planes).  FD_UPLOAD_ON_DEMAND: only the rows the letterbox resize reads now;
    //    the pixels the warps read follow after detection (step 4).  dfl describes the frames on the device, in their layout.
    std::vector<HostFrame> hf(dev_frames ? 0 : B);
    std::vector<fd_frame> dframes(B);
    std::vector<fd_frame_nv12> dyuv(frames.yuv ? B : 0);
    std::vector<float> ds(B);
    FrameList dfl = frames;
    if (dev_frames) {
        for (int i = 0; i < B; ++i) {
            dframes[i] = dev_frames[i];
            FrameDev geo;
            FD_TRY(fill_frame(ctx, dframes[i], dframes[i].data, &geo, &ds[i]));
        }
        dfl.bgr = dframes.data();
    } else {
        size_t arena = 0;
        std::vector<FrameDev> geo(B);
        for (int i = 0; i < B; ++i) {
            int rb;
            FD_TRY(fill_frame_of(ctx, frames, i, &geo[i], &ds[i], &rb));
            host_planes(frames, i, &hf[i], &arena);
        }
        FD_TRY(ctx->pipe_frames.reserve(arena + 256));
        uint8_t *base = ctx->pipe_frames.as<uint8_t>();
        for (int i = 0; i < B; ++i) {
            const HostPlane *p = hf[i].pl;
            if (frames.yuv) dyuv[i] = fd_frame_nv12{base + p[0].off, base + p[1].off, hf[i].h, hf[i].w, p[0].dpitch, p[1].dpitch};
            else dframes[i] = fd_frame{base + p[0].off, hf[i].h, hf[i].w, p[0].dpitch};
            bool sparse = false;
            if (demand) FD_TRY(upload_preprocess_rows(ctx, hf[i], geo[i].new_h, geo[i].scale_y, base, &h2d, &sparse));
            if (!sparse) FD_TRY(upload_full(ctx, hf[i], base, &h2d));
        }
        if (frames.yuv) dfl.yuv = dyuv.data();
        else if (frames.packed) dfl.packed = dframes.data();
        else if (frames.rgb) dfl.rgb = dframes.data();
        else dfl.bgr = dframes.data();
    }
    if (out->det_scale) std::copy(ds.begin(), ds.end(), out->det_scale);
    // 2. preprocess -> CNN input tensor (stays on the device unless out->tensor is given)
    const size_t tn = (size_t)B * 3 * ctx->cfg.image_h * ctx->cfg.image_w;
    FD_TRY(ctx->pipe_tensor.reserve(sizeof(float) * tn));
    FD_TRY(preprocess_batch(ctx, dfl, B, ctx->pipe_tensor.as<float>(), nullptr));
    // 3. heads (the CNN outputs), decode + NMS.  The score planes are dense reads: the A foreground channels of each image go
    //    to the device by DMA (face_detection.rs:322 never reads the background half).  The bbox / landmark tensors are read
    //    only at the anchors that pass the threshold (~450 of 16 800 per image): when the caller's buffers are pinned, the
    //    detect kernel reads those few sectors straight from host memory (zero-copy over PCIe) instead of copying 14 planes.
    const float *dev_heads[3 * FD_MAX_STRIDES];
    for (int s = 0; s < d.n_strides; ++s) {
        const int hw = d.fh[s] * d.fw[s];
        const int chn[3] = {2 * d.A, 4 * d.A, 10 * d.A};
        for (int k = 0; k < 3; ++k) {
            const size_t bytes = sizeof(float) * (size_t)B * chn[k] * hw;
            const float *mapped = nullptr;
            if (k != 0 && o.heads_zero_copy) {
                cudaPointerAttributes at;
                if (cudaPointerGetAttributes(&at, heads_host[3 * s + k]) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer)
                    mapped = static_cast<const float *>(at.devicePointer);
                else
                    cudaGetLastError();   // pageable memory: not an error, take the copy
            }
            if (mapped) {
                dev_heads[3 * s + k] = mapped;
                continue;
            }
            FD_TRY(ctx->pipe_heads[3 * s + k].reserve(bytes));
            if (k == 0) {
                const size_t img = sizeof(float) * (size_t)chn[0] * hw, fg = img / 2;
                FD_CUDA(cudaMemcpy2DAsync(ctx->pipe_heads[3 * s].as<unsigned char>() + fg, img,
                                          reinterpret_cast<const unsigned char *>(heads_host[3 * s]) + fg, img, fg, (size_t)B,
                                          cudaMemcpyHostToDevice, ctx->stream));
                h2d += (int64_t)(fg * (size_t)B);
            } else {
                FD_CUDA(cudaMemcpyAsync(ctx->pipe_heads[3 * s + k].p, heads_host[3 * s + k], bytes, cudaMemcpyHostToDevice, ctx->stream));
                h2d += (int64_t)bytes;
            }
            dev_heads[3 * s + k] = ctx->pipe_heads[3 * s + k].as<float>();
        }
    }
    FD_TRY(detect_enqueue(ctx, dev_heads, B, ds.data(), conf_thr, iou_thr));
    const size_t crop_bytes = (size_t)cw * ch * 3;
    FD_TRY(ctx->pipe_crops.reserve(crop_bytes * (size_t)out->cap_rows));
    FD_TRY(ctx->pipe_mode.reserve((size_t)out->cap_rows));
    uint8_t *crops_dev = ctx->pipe_crops.as<uint8_t>(), *mode_dev = ctx->pipe_mode.as<uint8_t>();
    int total = 0, n_crops = 0;
    if (!demand && !select) {
        // 4a. whole frames are on the device: align every detection without a host round trip, then fetch
        FD_TRY(align_detections(ctx, dfl, B, crops_dev, out->cap_rows, nullptr, mode_dev));
        FD_TRY(fd_detect_fetch(ctx, out->counts, out->det, out->landmarks, out->cap_rows, &total));
        n_crops = total;
    } else {
        // 4b. fetch the detections first (the reference has a host round trip here too: gRPC response, face_detection.rs:279,
        //     then FaceSelection / FaceAlignment on the host, face_pipeline/pipeline.rs:208-216)
        FD_TRY(fd_detect_fetch(ctx, out->counts, out->det, out->landmarks, out->cap_rows, &total));
        const int F = select ? B : total;
        n_crops = F;
        WarpFallback fb = detect_fallback(ctx);
        const int32_t *fidx_dev = ctx->out_frame_idx.as<int32_t>();
        if (select) {   // FaceSelection::call per image on the device, then the estimate of the B selected faces
            FD_TRY(select_detections(ctx, dfl, B, o.is_enroll, &o.select_params, nullptr));
            fb.sel = ctx->select_sel.as<int>();
            fidx_dev = ctx->select_fidx.as<int32_t>();
            ctx->est_valid = false;
        }
        if (F > 0) {
            if (select || !ctx->est_valid || F > ctx->est_cap) {
                ctx->est_valid = false;
                FD_TRY(ctx->align_M.reserve(sizeof(double) * 12 * (size_t)F));
                FD_TRY(ctx->align_ok.reserve((size_t)F));
                FD_TRY(estimate_launch(ctx, select ? ctx->select_lmk.as<float>() : ctx->out_lmk.as<float>(), nullptr, nullptr, F,
                                       ctx->align_M.as<double>(), nullptr, ctx->align_ok.as<uint8_t>(), nullptr));
            }
            if (demand) {
                // the transforms come back (96 B per face); the host turns them into the pixel rectangles the warps read
                std::vector<double> M12((size_t)F * 12);
                std::vector<uint8_t> okh(F);
                std::vector<int> selh(select ? 2 * (size_t)B : 0);
                FD_CUDA(cudaMemcpyAsync(M12.data(), ctx->align_M.p, sizeof(double) * 12 * (size_t)F, cudaMemcpyDeviceToHost, ctx->stream));
                FD_CUDA(cudaMemcpyAsync(okh.data(), ctx->align_ok.p, (size_t)F, cudaMemcpyDeviceToHost, ctx->stream));
                if (select) FD_CUDA(cudaMemcpyAsync(selh.data(), ctx->select_sel.p, sizeof(int) * 2 * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
                FD_TRY(wait_stream(ctx));
                d2h += (int64_t)F * 97 + (int64_t)selh.size() * 4;
                struct Rect { int x0, y0, x1, y1; };
                std::vector<std::vector<Rect>> rects(B);
                std::vector<int64_t> rect_bytes(B, 0);
                int f = 0;
                for (int b = 0; b < B; ++b) {
                    const int nf = select ? 1 : out->counts[b];
                    for (int j = 0; j < nf; ++j, ++f) {
                        if (hf[b].full) continue;
                        if (select && (selh[2 * b] < 0 || selh[2 * b + 1] < 0)) continue;   // nothing to align: zero crop
                        Rect r;
                        if (!okh[f]) {   // bbox-crop fallback reads (x0,y0)..(W,H): rare, take the whole frame
                            rect_bytes[b] = INT64_MAX / 4;
                            continue;
                        }
                        if (!warp_source_rect(&M12[(size_t)f * 12 + 6], cw, ch, hf[b].w, hf[b].h, &r.x0, &r.y0, &r.x1, &r.y1))
                            continue;
                        rects[b].push_back(r);
                        FD_TRY(upload_rect(ctx, hf[b], r.x0, r.y0, r.x1, r.y1, nullptr, &rect_bytes[b]));
                    }
                }
                uint8_t *base = ctx->pipe_frames.as<uint8_t>();
                for (int b = 0; b < B; ++b) {
                    if (hf[b].full || rect_bytes[b] == 0) continue;
                    int64_t frame_bytes = 0;
                    for (int q = 0; q < hf[b].np; ++q) frame_bytes += (int64_t)hf[b].pl[q].row_bytes * hf[b].pl[q].rows;
                    if (rect_bytes[b] >= frame_bytes - have_bytes(hf[b])) {   // many overlapping faces: the rest of the frame is cheaper
                        FD_TRY(upload_complement_rows(ctx, hf[b], base, &h2d));
                        continue;
                    }
                    for (const Rect &r : rects[b]) FD_TRY(upload_rect(ctx, hf[b], r.x0, r.y0, r.x1, r.y1, base, &h2d));
                }
            }
            FD_TRY(upload_frame_table(ctx, dfl, B, nullptr, nullptr));
            fb.mode_out = mode_dev;
            FD_TRY(warp_launch(ctx, ctx->frames_dev.as<FrameDev>(), fidx_dev, ctx->align_M.as<double>(), ctx->align_ok.as<uint8_t>(), nullptr,
                               std::min(F, (int)out->cap_rows), crops_dev, cw, ch, fb, ctx->frames_fmt));
            ctx->align_replay = false;
        }
        if (select && out->sel) {
            FD_CUDA(cudaMemcpyAsync(out->sel, ctx->select_sel.p, sizeof(int) * 2 * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
            d2h += (int64_t)sizeof(int) * 2 * B;
        }
    }
    if (o.heads_zero_copy) {   // sectors the detect kernel pulled from pinned host memory: 4 deltas per candidate, 10 per kept face
        int32_t st[8];
        if (fd_detect_last_stats(ctx, st) == FD_OK) {
            bool any = false;
            for (int i = 0; i < n_heads; ++i) any = any || (i % 3 != 0 && dev_heads[i] != ctx->pipe_heads[i].as<float>());
            if (any) h2d += 32ll * (4ll * st[2] + 10ll * total);
        }
    }
    // 5. results D2H
    out->total = total;
    out->n_crops = n_crops;
    d2h += (int64_t)sizeof(int) * (B + 1) + (int64_t)total * 15 * sizeof(float);
    if (n_crops) FD_CUDA(cudaMemcpyAsync(out->crops, crops_dev, crop_bytes * (size_t)n_crops, cudaMemcpyDeviceToHost, ctx->stream));
    d2h += (int64_t)crop_bytes * n_crops;
    if (out->align_mode && n_crops) {
        FD_CUDA(cudaMemcpyAsync(out->align_mode, mode_dev, (size_t)n_crops, cudaMemcpyDeviceToHost, ctx->stream));
        d2h += n_crops;
    }
    if (out->tensor) {
        FD_CUDA(cudaMemcpyAsync(out->tensor, ctx->pipe_tensor.p, sizeof(float) * tn, cudaMemcpyDeviceToHost, ctx->stream));
        d2h += (int64_t)sizeof(float) * tn;
    }
    FD_TRY(wait_stream(ctx));
    out->h2d_bytes = h2d;
    out->d2h_bytes = d2h;
    return FD_OK;
}

FD_EXPORT int fd_pipeline_host(fd_ctx *ctx, const fd_frame *frames, int B, const float *const *heads_host, int n_heads,
                               float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(frames, "fd_pipeline_host: null frames");
    FrameList fl;
    fl.bgr = frames;
    return pipeline_host_impl(ctx, fl, nullptr, B, heads_host, n_heads, conf_thr, iou_thr, opts, out, 0);
}
FD_EXPORT int fd_pipeline_host_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, const float *const *heads_host,
                                      int n_heads, float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out) {
    FD_TRY(check_ctx(ctx));
    FrameList fl;
    FD_TRY(yuv420_frames(frames, layout, &fl));
    FD_REQUIRE(frames, "fd_pipeline_host_yuv420: null frames");
    return pipeline_host_impl(ctx, fl, nullptr, B, heads_host, n_heads, conf_thr, iou_thr, opts, out, 0);
}
FD_EXPORT int fd_pipeline_host_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, const float *const *heads_host,
                                      int n_heads, float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out) {
    FD_TRY(check_ctx(ctx));
    FrameList fl;
    FD_TRY(yuv422_frames(frames, layout, &fl));
    FD_REQUIRE(frames, "fd_pipeline_host_yuv422: null frames");
    return pipeline_host_impl(ctx, fl, nullptr, B, heads_host, n_heads, conf_thr, iou_thr, opts, out, 0);
}
FD_EXPORT int fd_pipeline_host_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, const float *const *heads_host,
                                   int n_heads, float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out) {
    FD_TRY(check_ctx(ctx));
    FrameList fl;
    FD_TRY(rgb_frames(frames, layout, &fl));
    FD_REQUIRE(frames, "fd_pipeline_host_rgb: null frames");
    return pipeline_host_impl(ctx, fl, nullptr, B, heads_host, n_heads, conf_thr, iou_thr, opts, out, 0);
}

// FacePipeline::extract's real input (face_pipeline/pipeline.rs:188-196): encoded image bytes.  byte_data_to_opencv (N4) on the
// way in, then the same path with the frames already on the device — the compressed stream is all that crosses PCIe for them.
FD_EXPORT int fd_pipeline_host_jpeg(fd_ctx *ctx, const uint8_t *const *jpegs, const size_t *nbytes, int B, int n_threads,
                                    const float *const *heads_host, int n_heads, float conf_thr, float iou_thr, const fd_pipeline_opts *opts,
                                    fd_host_batch_out *out) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(jpegs && nbytes && B > 0, "fd_pipeline_host_jpeg: bad arguments");
    std::vector<fd_frame> dev((size_t)B);
    FD_TRY(fd_decode_jpeg_batch(ctx, jpegs, nbytes, B, n_threads, dev.data()));
    return pipeline_host_impl(ctx, FrameList(), dev.data(), B, heads_host, n_heads, conf_thr, iou_thr, opts, out, ctx->jpeg_last_h2d);
}

FD_EXPORT int fd_pipeline_tensor_dev(fd_ctx *ctx, const float **out_nchw_dev) {
    FD_REQUIRE(ctx && out_nchw_dev, "fd_pipeline_tensor_dev: null");
    *out_nchw_dev = ctx->pipe_tensor.as<float>();
    return FD_OK;
}
