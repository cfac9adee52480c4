/*
 * fd_b200.h — C ABI of the B200-native detection hot path for okieraised/rs-face-detection.
 *
 * One shared library (libfd_b200.so, hand-written CUDA for sm_100a).  Plain pointers and sizes only.
 * Every function returns an fd_status (0 = ok); fd_last_error() gives the thread-local message.
 * Reference citations are relative to the reference repo root.
 *
 * Threading: one fd_ctx per GPU per host thread; a ctx is not internally locked.  All work of a ctx is
 * issued on the ctx's own CUDA stream.  "host" pointers are ordinary (or pinned) host memory owned by the
 * caller; "dev" pointers are device memory on the ctx's GPU (fd_dev_alloc or any CUDA allocation).
 */
#ifndef FD_B200_H
#define FD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FD_MAX_STRIDES 8
#define FD_MAX_ANCHORS 4
#define FD_ABI_VERSION 2

typedef enum fd_status {
    FD_OK = 0,
    FD_ERR_INVALID = 1,    /* bad argument */
    FD_ERR_CUDA = 2,       /* CUDA runtime error (message in fd_last_error) */
    FD_ERR_NAN_SCORE = 3,  /* NaN key in fd_argsort_descending / fd_nms*: utils.rs:92 unwraps partial_cmp (panic); nms.rs:6
                              sorts with an inconsistent comparator (unspecified order).  The detect path never raises it:
                              `score >= thr` (face_detection.rs:375) drops a NaN score before any sort. */
    FD_ERR_CAPACITY = 4,   /* caller-provided output buffer too small */
    FD_ERR_NO_DEVICE = 5,  /* no usable CUDA device: there is NO CPU fallback */
    FD_ERR_ESTIMATE = 6    /* FaceAlignment: empty transform AND the bbox-crop fallback's ROI is outside the image (the reference
                              returns Err from Mat::roi, face_alignment.rs:92-95) */
} fd_status;

/* Constants of RetinaFaceDetection (face_detection.rs:19-38, 41-129), FaceDetectionConfig and
 * FaceAlignmentConfig (face_pipeline/config.rs:13-55) as one plain struct. */
typedef struct fd_config {
    int32_t image_w, image_h;                              /* detector input, config.rs:27 (640,640) */
    float conf_thr, iou_thr;                               /* config.rs:29-30 (0.7, 0.45) */
    int32_t n_strides;
    int32_t strides[FD_MAX_STRIDES];                       /* _feat_stride_fpn, face_detection.rs:52 */
    int32_t num_anchors;                                   /* A per stride, face_detection.rs:100-103 */
    float base_anchors[FD_MAX_STRIDES][FD_MAX_ANCHORS][4]; /* _anchors_fpn, face_detection.rs:94-98 */
    float pixel_means[3], pixel_stds[3], pixel_scale;      /* face_detection.rs:105-107 (BGR order) */
    float bbox_stds[4], landmark_std;                      /* face_detection.rs:91-92 */
    int32_t crop_w, crop_h;                                /* config.rs:45 (112,112) */
    float template_landmarks[5][2];                        /* config.rs:46-52 */
} fd_config;

typedef struct fd_ctx fd_ctx;

/* Frame descriptor: BGR u8 HWC (an OpenCV CV_8UC3 Mat: face_detection.rs:131, face_alignment.rs:27), pitch >= 3 * width.
 * The *_yuv422 calls describe a packed 4:2:2 frame with it too: `data` is the packed plane, height rows of width / 2
 * macropixels (4 bytes, 2 pixels each), pitch >= 2 * width; width even, any height >= 1.  The *_rgb calls describe an
 * interleaved RGB24, RGBA, BGRA or GRAY8 frame with it (FD_RGB_* below). */
typedef struct fd_frame {
    const uint8_t *data; /* dev pointer for *_batch functions */
    int32_t height, width, pitch;
} fd_frame;

/* Frame descriptor: NV12 video frame (a hardware decoder's output): a height x width Y plane and a height/2 x width plane of
 * interleaved U,V pairs, each row `pitch_*` bytes apart.  Device pointers; the planes may be separate allocations.  Width and
 * height must be even (cv::cvtColor rejects odd sizes).  The *_nv12 calls give the results of their BGR counterparts on the
 * frame cv::cvtColor(COLOR_YUV2BGR_NV12) makes (BT.601 limited range), without building it. */
struct fd_frame_nv12 {
    const uint8_t *y, *uv;
    int32_t height, width, pitch_y, pitch_uv;
};
typedef struct fd_frame_nv12 fd_frame_nv12;

/* Layouts of a 4:2:0 frame for the *_yuv420 calls, which describe every layout with fd_frame_nv12.  `y` is always the
 * height x width luma plane.  What `uv` points to (H = height, W = width, all rows `pitch_uv` bytes apart):
 *   FD_YUV420_NV12  interleaved U,V: H/2 rows of W bytes; pitch_uv >= W (NVDEC output)
 *   FD_YUV420_NV21  interleaved V,U: H/2 rows of W bytes; pitch_uv >= W (Android camera preview)
 *   FD_YUV420_I420  the U plane, H/2 rows of W/2 bytes; the V plane starts at uv + (H/2) * pitch_uv; pitch_uv >= W/2
 *                   (FFmpeg yuv420p, WebRTC I420Buffer)
 *   FD_YUV420_YV12  the V plane, H/2 rows of W/2 bytes; the U plane starts at uv + (H/2) * pitch_uv; pitch_uv >= W/2
 * I420 and YV12 are thus the single buffer cv::cvtColor reads, with pitches added; (H/2) * pitch_uv must stay below 2 GB.  The calls give the results of their
 * BGR counterparts on the frame cv::cvtColor(COLOR_YUV2BGR_NV12 / _NV21 / _I420 / _YV12) makes (BT.601 limited range),
 * without building it. */
enum { FD_YUV420_NV12 = 0, FD_YUV420_NV21 = 1, FD_YUV420_I420 = 2, FD_YUV420_YV12 = 3 };

/* Layouts of a packed 4:2:2 frame (an fd_frame) for the *_yuv422 calls: the byte order of one 2-pixel macropixel.  Pixel x
 * takes its own Y and the U, V of its pair x & ~1; there is no vertical subsampling.
 *   FD_YUV422_YUY2  Y0 U Y1 V (YUYV: V4L2_PIX_FMT_YUYV, GStreamer YUY2, FFmpeg yuyv422)
 *   FD_YUV422_UYVY  U Y0 V Y1 (GStreamer UYVY, FFmpeg uyvy422, DeckLink bmdFormat8BitYUV)
 *   FD_YUV422_YVYU  Y0 V Y1 U (GStreamer YVYU, FFmpeg yvyu422)
 * The calls give the results of their BGR counterparts on the frame cv::cvtColor(COLOR_YUV2BGR_YUY2 / _UYVY / _YVYU) makes
 * (BT.601 limited range), without building it. */
enum { FD_YUV422_YUY2 = 0, FD_YUV422_UYVY = 1, FD_YUV422_YVYU = 2 };

/* Layouts of an interleaved RGB-family frame (an fd_frame) for the *_rgb calls; pitch >= bytes per pixel * width, any
 * width and height >= 1.
 *   FD_RGB_RGB24  R G B      3 B/pixel
 *   FD_RGB_RGBA   R G B A    4 B/pixel, the fourth byte is ignored (also RGBX)
 *   FD_RGB_BGRA   B G R A    4 B/pixel, the fourth byte is ignored (also BGRX)
 *   FD_RGB_GRAY8  Y          1 B/pixel (B = G = R = Y)
 * The calls give the results of their BGR counterparts on the frame cv::cvtColor(COLOR_RGB2BGR / COLOR_RGBA2BGR /
 * COLOR_BGRA2BGR / COLOR_GRAY2BGR) makes, without building it. */
enum { FD_RGB_RGB24 = 0, FD_RGB_RGBA = 1, FD_RGB_BGRA = 2, FD_RGB_GRAY8 = 3 };

/* ---- library / context ---------------------------------------------------------------------------- */
int fd_abi_version(void);
const char *fd_last_error(void);
/* Fills the reference defaults; base anchors come from fd_generate_anchors_fpn2 (face_detection.rs:55-98). */
int fd_config_default(fd_config *cfg);
int fd_device_count(int *count);
int fd_ctx_create(int device_id, const fd_config *cfg, fd_ctx **out);
void fd_ctx_destroy(fd_ctx *ctx);
int fd_ctx_get_config(const fd_ctx *ctx, fd_config *out);
int fd_ctx_total_anchors(const fd_ctx *ctx, int32_t *out);   /* sum over strides of H*W*A (16800) */
void *fd_ctx_stream(fd_ctx *ctx);                             /* cudaStream_t */
int fd_ctx_synchronize(fd_ctx *ctx);
/* Tuning knob: tell the ctx how many contexts keep batches in flight on this GPU at the same time (default 1).  With
 * more than one, the per-image detect kernel is launched in its 32-register build so that it shares its SMs with the
 * other batch's bandwidth-bound kernels (slower alone, faster in aggregate).  Results are identical. */
int fd_ctx_set_sharing(fd_ctx *ctx, int contexts_in_flight);
/* number of kernels this ctx has launched since creation (bench.py's gpu_launches) */
int fd_ctx_launch_count(const fd_ctx *ctx, int64_t *out);

/* Per-kernel device timing for the bench harness: while enabled, every kernel launch of this ctx is followed by a CUDA
 * event on the ctx stream; fd_ctx_profile_fetch synchronises and writes one line per kernel, "name launches total_us",
 * where a launch's time is the gap since the previous launch's event (kernel + launch gap).  Not for production use. */
int fd_ctx_profile(fd_ctx *ctx, int enable);
int fd_ctx_profile_fetch(fd_ctx *ctx, char *buf, size_t cap);

/* ---- memory helpers (so a host language needs no CUDA binding of its own) --------------------------- */
int fd_dev_alloc(fd_ctx *ctx, size_t bytes, void **out);
int fd_dev_free(fd_ctx *ctx, void *ptr);
int fd_host_alloc_pinned(size_t bytes, void **out);
int fd_host_free_pinned(void *ptr);
int fd_memcpy_h2d(fd_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);     /* blocking */
int fd_memcpy_d2h(fd_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);     /* blocking */
int fd_memcpy_h2d_async(fd_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
int fd_memcpy_d2h_async(fd_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);
int fd_memset_dev(fd_ctx *ctx, void *dst_dev, int value, size_t bytes);

/* ---- init-time anchor tables: HOST code, no GPU (generate_anchors.rs) ------------------------------- */
/* generate_anchors.rs:41-59 ; out (n_ratios*n_scales, 4) */
int fd_generate_anchors(int base_size, const float *ratios, int n_ratios, const float *scales, int n_scales,
                        float *out, int *n_out);
/* generate_anchors.rs:61-93 ; out ((dense?2:1)*n_ratios*n_scales, 4) */
int fd_generate_anchors2(int base_size, const float *ratios, int n_ratios, const float *scales, int n_scales,
                         int stride, int dense_anchor, float *out, int *n_out);
/* generate_anchors.rs:95-114 ; level i uses ratios[i], scales[i]; out (n_levels, 4) */
int fd_generate_anchors_fpn(const int *base_size, const float *ratios, const float *scales, int n_levels, float *out);
/* generate_anchors.rs:116-138 ; cfg = per stride {base_size, ratios, scales}; strides processed in
 * descending order; out receives, per stride in that order, its (n_ratios*n_scales*(dense?2:1), 4) block. */
typedef struct fd_anchor_cfg {
    int32_t stride, base_size;
    int32_t n_ratios, n_scales;
    float ratios[8], scales[8];
    int32_t allowed_border;
} fd_anchor_cfg;
int fd_generate_anchors_fpn2(int dense_anchor, const fd_anchor_cfg *cfg, int n_cfg, float *out, int *rows_per_stride,
                             int *strides_sorted);

/* ---- drop-in single ops: HOST pointers in/out, blocking, computed on the GPU ------------------------ */
/* processing::nms::nms(&Array2<f32>, f32) -> Vec<usize>  (nms.rs:3-65).  dets (K,5) any order; keep (cap>=K)
 * receives indices into dets in pick order (stable descending-score sort done on the device). */
int fd_nms(fd_ctx *ctx, const float *dets, int K, float thresh, int32_t *keep, int *num_keep);
/* Diagnostics of the last NMS with K > 4096 on this ctx (blocks): out[8] = {spatial path used, kept, decision
 * epochs, grid width, grid height, cell size (f32 bits), 0, 0}. */
int fd_nms_last_stats(fd_ctx *ctx, int32_t *out);
/* rcnn::cpu_nms::cpu_nms variant (cpu_nms.rs:10-55): suppresses on ovr >= thresh. */
int fd_cpu_nms(fd_ctx *ctx, const float *dets, int K, float thresh, int32_t *keep, int *num_keep);
/* Contract of the reference's C symbol `_nms` (gpu_nms.hpp:6-8, nms_kernel.cu:91-144): boxes (n, boxes_dim>=4)
 * ALREADY sorted by score descending; keep = indices into the sorted array. */
int fd_nms_sorted(fd_ctx *ctx, const float *boxes, int n, int boxes_dim, float thresh, int32_t *keep, int *num_out);
/* The literal reference symbols, so src/rcnn/gpu_nms.rs links unchanged (uses a lazily created per-device ctx). */
void _nms(int32_t *keep, int *num_out, const float *boxes_host, int boxes_num, int boxes_dim, float thresh, int device_id);
void _set_device(int device_id);
/* utils::argsort_descending (utils.rs:87-95): stable; NaN -> FD_ERR_NAN_SCORE. */
int fd_argsort_descending(fd_ctx *ctx, const float *scores, int n, int32_t *order);
/* rcnn::anchors::anchors (anchors.rs:3-21): out (H,W,A,4). */
int fd_anchors_plane(fd_ctx *ctx, int height, int width, int stride, const float *base_anchors, int A, float *out);
/* RetinaFaceDetection::bbox_pred (face_detection.rs:516-549): boxes (n,4), deltas (n,ncols>=4); columns >=4 copied. */
int fd_bbox_pred(fd_ctx *ctx, const float *boxes, const float *deltas, int n, int ncols, float *out);
/* bbox_transform::nonlinear_pred (bbox_transform.rs:90-120): every group of 4 columns regressed. */
int fd_nonlinear_pred(fd_ctx *ctx, const float *boxes, const float *deltas, int n, int ncols, float *out);
/* landmark_pred (face_detection.rs:551-570 (n,5,2) == bbox_transform.rs:123-160 (n,10)). */
int fd_landmark_pred(fd_ctx *ctx, const float *boxes, const float *deltas, int n, float *out);
/* bbox_transform::clip_boxes / clip_points (bbox_transform.rs:27-65), in place. */
int fd_clip_boxes(fd_ctx *ctx, float *boxes, int rows, int cols, int im_h, int im_w);
int fd_clip_points(fd_ctx *ctx, float *points, int rows, int cols, int im_h, int im_w);
/* bbox_transform::iou_pred (:162-186), nonlinear_transform (:67-88). */
int fd_iou_pred(fd_ctx *ctx, const float *boxes, const float *deltas, int n, int ncols, int num_classes, float *out);
int fd_nonlinear_transform(fd_ctx *ctx, const float *ex_rois, const float *gt_rois, int n, float *out);
/* rcnn::bbox::bbox_overlaps == bbox_transform::bbox_overlaps_py (bbox.rs:4-30): out (n,k). */
int fd_bbox_overlaps(fd_ctx *ctx, const float *boxes, int n, const float *query, int k, float *out);
/* RetinaFaceDetection::_preprocess geometry (face_detection.rs:140-153), host arithmetic. */
int fd_letterbox_geometry(const fd_ctx *ctx, int img_h, int img_w, int *new_w, int *new_h, float *det_scale);
/* _preprocess + tensor loop (face_detection.rs:131-230) for ONE host image -> (1,3,image_h,image_w) f32 host. */
int fd_preprocess(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, float *out_nchw, float *det_scale);
/* cv::resize(INTER_LINEAR) 8UC3 as called at face_detection.rs:156 (host in/out). */
int fd_resize_linear(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, uint8_t *out, int out_h, int out_w);
/* _forward post-CNN half + _postprocess (face_detection.rs:319-493) for ONE image, host tensors.
 * heads[3*s+0..2] = scores (2A,H,W), bbox (4A,H,W), landmarks (10A,H,W) of stride s.
 * det (cap,5), landmarks (cap,10). */
int fd_detect(fd_ctx *ctx, const float *const *heads, int n_heads, float det_scale, float conf_thr, float iou_thr,
              float *det, float *landmarks, int cap, int *num_det);
/* cv::estimateAffinePartial2D(from, to, LMEDS, 3.0, 2000, 0.99, 10) for n_sets sets of 5 points
 * (face_alignment.rs:50-59).  from (n_sets,5,2); to = NULL -> ctx template.  M (n_sets,2,3) f64; ok (n_sets). */
int fd_estimate_affine_partial_2d(fd_ctx *ctx, const float *from, const float *to, int n_sets, double *M, uint8_t *ok);
/* cv::warpAffine(img, M, (crop_w,crop_h), INTER_LINEAR, BORDER_CONSTANT, 0) (face_alignment.rs:119-126), host in/out. */
int fd_warp_affine(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, const double *M, uint8_t *out,
                   int out_h, int out_w);
/* FaceAlignment::call (face_alignment.rs:27-141) for ONE host image and ONE face: the similarity warp, or — when
 * estimateAffinePartial2D returns an empty matrix (degenerate / non-finite landmarks) — the bbox-crop fallback (:64-116):
 * det = bbox (NULL = None: the image inset by 1/16), ROI (max(x1-22,0), max(y1-22,0)) .. (max(x2+22,W), max(y1+22,H)) exactly
 * as written there (`max`, det[1]), cv::resize to the crop size.  mode_out (optional): 1 = warp, 2 = fallback crop.
 * Errors like the reference: landmarks NULL (None: OpenCV asserts on the empty Mat) -> FD_ERR_INVALID; fallback ROI not
 * inside the image (Mat::roi) -> FD_ERR_ESTIMATE.  M_out is written only in mode 1. */
int fd_align(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, const float *bbox /*4 or NULL*/,
             const float *landmarks /*5x2*/, uint8_t *crop /*crop_h x crop_w x 3*/, double *M_out /*2x3 or NULL*/, int *mode_out);

/* ---- batched device-resident pipeline (the benchmarked path); asynchronous on the ctx stream --------- */
/* fd_nms with DEVICE buffers (asynchronous): dets_dev (K,5); keep_dev (K) int32; num_keep_dev (2) int32 =
 * {count, NaN flag}.  The sort and the whole suppression sweep stay on the device. */
int fd_nms_device(fd_ctx *ctx, const float *dets_dev, int K, float thresh, int32_t *keep_dev, int32_t *num_keep_dev);
/* frames: HOST array of B descriptors whose .data are DEV pointers.  out_nchw_dev (B,3,image_h,image_w) f32.
 * det_scale_host (B) is written before return (pure host arithmetic). */
int fd_preprocess_batch(fd_ctx *ctx, const fd_frame *frames, int B, float *out_nchw_dev, float *det_scale_host);
/* fd_preprocess_batch on NV12 frames: the tensor and det_scale of cv::cvtColor(COLOR_YUV2BGR_NV12) followed by
 * fd_preprocess_batch, reading only the Y and UV rows the resize taps.  FD_ERR_INVALID for an odd width or height, a pitch
 * below the width or a null plane. */
int fd_preprocess_batch_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, float *out_nchw_dev, float *det_scale_host);
/* fd_preprocess_batch_nv12 for any FD_YUV420_* layout (layout FD_YUV420_NV12 is fd_preprocess_batch_nv12).  FD_ERR_INVALID
 * for an odd width or height, a null plane, pitch_y below the width, pitch_uv below the layout's minimum or an unknown
 * layout.  The same for the other *_yuv420 calls. */
int fd_preprocess_batch_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, float *out_nchw_dev,
                               float *det_scale_host);
/* fd_preprocess_batch on packed 4:2:2 frames in an FD_YUV422_* layout, reading only the packed rows the resize taps.
 * FD_ERR_INVALID for a null data pointer, a width that is not positive and even, a height below 1, a pitch below 2 * width or
 * an unknown layout (also when B == 0).  The same for the other *_yuv422 calls. */
int fd_preprocess_batch_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, float *out_nchw_dev, float *det_scale_host);
/* fd_preprocess_batch on interleaved RGB-family frames in an FD_RGB_* layout.  FD_ERR_INVALID for a null data pointer, a
 * height or width below 1, a pitch below bytes per pixel * width or an unknown layout (also when B == 0).  The same for the
 * other *_rgb calls. */
int fd_preprocess_batch_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, float *out_nchw_dev, float *det_scale_host);
/* heads_dev[3*s+0..2]: (B,2A,H,W), (B,4A,H,W), (B,10A,H,W) dev tensors of stride s.  Results stay on the device
 * inside the ctx until fd_detect_fetch / fd_align_detections.  Asynchronous.  Images with more than 4096 candidates
 * (and, the first time a ctx meets one, images with more than 1024) are completed by fd_detect_fetch / fd_detect_view;
 * an fd_align_detections enqueued before that is re-run there (call fd_detect_fetch first when other consumers, e.g.
 * fd_select_detections without sel_host, must see such images). */
int fd_detect_batch(fd_ctx *ctx, const float *const *heads_dev, int n_heads, int B, const float *det_scale_host,
                    float conf_thr, float iou_thr);
/* Blocks; copies the compact results of the last fd_detect_batch: counts (B), det (total,5), landmarks (total,10),
 * rows in frame order then pick order.  cap_rows = capacity of det/landmarks in rows. */
int fd_detect_fetch(fd_ctx *ctx, int32_t *counts, float *det, float *landmarks, int cap_rows, int *total);
/* Device views of the last fd_detect_batch results (valid until the next call). */
typedef struct fd_det_view {
    const int32_t *counts_dev;    /* (B) */
    const int32_t *offsets_dev;   /* (B+1) exclusive prefix */
    const float *det_dev;         /* (total,5) */
    const float *landmarks_dev;   /* (total,10) */
    const int32_t *frame_idx_dev; /* (total) */
    const int32_t *candidates_dev; /* (B) pre-NMS candidate counts K */
} fd_det_view;
int fd_detect_view(fd_ctx *ctx, fd_det_view *out);
/* Diagnostics of the last fd_detect_batch, read without completing anything (blocks on the ctx stream): out[8] =
 * {images the detect kernel deferred to fd_detect_fetch's host-driven NMS path, largest per-image candidate count K,
 *  total candidates, faces the kernel finished itself, 1 if the single fused kernel ran (0: three-kernel path),
 *  1 if the launch kept 1024 < K <= 4096 images on the device, 0, 0}.  bench.py reports the first two. */
int fd_detect_last_stats(fd_ctx *ctx, int32_t *out);
/* Aligns F faces: landmarks_dev (F,10) in original-frame coordinates, frame_idx_dev (F) into frames, bbox_dev (F,4) or
 * NULL (bbox == None) for the fallback.  crops_dev (F,crop_h,crop_w,3) u8; M_dev (F,6) f64 or NULL; ok_dev (F) u8 or NULL:
 * 1 = similarity warp, 2 = bbox-crop fallback (face_alignment.rs:64-116), 0 = the reference returns Err (crop zero-filled). */
int fd_align_batch(fd_ctx *ctx, const fd_frame *frames, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                   const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);
/* fd_align_batch on NV12 frames: crops, M and modes of cv::cvtColor(COLOR_YUV2BGR_NV12) followed by fd_align_batch
 * (BORDER_CONSTANT is black in BGR). */
int fd_align_batch_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                        const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);
/* fd_align_batch_nv12 for any FD_YUV420_* layout. */
int fd_align_batch_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, const float *landmarks_dev,
                          const int32_t *frame_idx_dev, const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);
/* fd_align_batch on packed 4:2:2 frames in an FD_YUV422_* layout (BORDER_CONSTANT is black in BGR). */
int fd_align_batch_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                          const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);
/* fd_align_batch on interleaved RGB-family frames in an FD_RGB_* layout (BORDER_CONSTANT is black in BGR). */
int fd_align_batch_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, const float *landmarks_dev, const int32_t *frame_idx_dev,
                       const float *bbox_dev, int F, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);
/* Aligns every detection of the last fd_detect_batch without a host round trip (fallback box = the detection's own box).
 * crops_dev has room for cap_faces crops; detections beyond cap_faces are not aligned (fd_detect_fetch still reports them). */
int fd_align_detections(fd_ctx *ctx, const fd_frame *frames, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                        uint8_t *ok_dev);
/* fd_align_detections on NV12 frames: the results of cv::cvtColor(COLOR_YUV2BGR_NV12) followed by fd_align_detections,
 * re-run on the NV12 frames by fd_detect_fetch / fd_detect_view when deferred images change the detections. */
int fd_align_detections_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                             uint8_t *ok_dev);
/* fd_align_detections_nv12 for any FD_YUV420_* layout; a replay at fd_detect_fetch / fd_detect_view reads the frames in
 * the layout given here. */
int fd_align_detections_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, uint8_t *crops_dev, int cap_faces,
                               double *M_dev, uint8_t *ok_dev);
/* fd_align_detections on packed 4:2:2 frames in an FD_YUV422_* layout; a replay at fd_detect_fetch / fd_detect_view reads the
 * frames in the layout given here. */
int fd_align_detections_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                               uint8_t *ok_dev);
/* fd_align_detections on interleaved RGB-family frames in an FD_RGB_* layout; a replay at fd_detect_fetch / fd_detect_view
 * reads the frames in the layout given here. */
int fd_align_detections_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, uint8_t *crops_dev, int cap_faces, double *M_dev,
                            uint8_t *ok_dev);

/* ---- SURVEY 8(f) N1: post-align model preprocessors, fused onto the aligned crops ----------------------- */
/* FaceExtraction::_preprocess (face_extraction.rs:38-77: mean 127.5, mul 0.0078125), FaceQuality::call
 * (face_quality.rs:43-101: mean {123.675,116.28,103.53}, mul {0.01712475,0.017507,0.01742919}),
 * FaceQualityAssessment::call (face_quality_assessment.rs:48-88: mean 127.5, mul 0.00784313725):
 * cv::resize INTER_LINEAR to (out_w,out_h) -> BGR2RGB -> (p - mean[i]) * mul[i] (i in RGB order) -> NCHW f32.
 * crops_dev (F,in_h,in_w,3) u8 (e.g. the fd_align_* output) -> out_nchw_dev (F,3,out_h,out_w).  Asynchronous.
 * use_detect_count != 0: process min(F, faces of the last fd_detect_batch), counted on the device. */
int fd_crops_to_tensor(fd_ctx *ctx, const uint8_t *crops_dev, int F, int in_h, int in_w, int out_h, int out_w,
                       const float *mean_rgb, const float *mul_rgb, float *out_nchw_dev, int use_detect_count);
/* the same for ONE host image (the reference processes `&[Mat]` one Mat at a time), blocking */
int fd_model_preprocess(fd_ctx *ctx, const uint8_t *img, int h, int w, int pitch, int out_h, int out_w,
                        const float *mean_rgb, const float *mul_rgb, float *out_nchw);

/* ---- SURVEY 8(f) N2: the CNN's wire format ---------------------------------------------------------------------- */
/* Triton ModelInferResponse.raw_output_contents -> decode + NMS without a host-side f32 conversion (face_detection.rs:286-312,
 * utils.rs:126-132 u8_to_f32_vec): raw[i] = the little-endian f32 bytes of output i (any host alignment), nbytes[i] its
 * length, shape[i] = its 4 dims (N,C,H,W), outputs ordered like fd_detect_batch (scores, bbox, landmarks per stride).
 * Like the reference, trailing bytes that do not fill an f32 are ignored and a shape whose product differs from the f32
 * count is an error (Array4::from_shape_vec).  The bytes are copied once, host -> device, and read in place by the decode
 * kernel (the GPU is little-endian).  Tensors the server already left in device memory (Triton CUDA shared memory,
 * client.rs:169-188) go to fd_detect_batch directly.  Results as fd_detect_batch; B = shape[0][0]. */
int fd_detect_batch_raw(fd_ctx *ctx, const uint8_t *const *raw, const size_t *nbytes, const int64_t (*shape)[4], int n_heads,
                        const float *det_scale_host, float conf_thr, float iou_thr);

/* ---- SURVEY 8(f) N3: FaceSelection (pipeline/module/face_selection.rs), one face per image ------------------- */
typedef struct fd_select_params {   /* FaceSelectionConfig::new, face_pipeline/config.rs:107-116 */
    float margin_center_left_ratio, margin_center_right_ratio, margin_edge_ratio, minimum_face_ratio;
} fd_select_params;
int fd_select_params_default(fd_select_params *p);   /* 0.3, 0.3, 0.1, 0.0075 */
/* FaceSelection::call (face_selection.rs:72-189) for ONE image, host in/out, computed on the GPU.  face_boxes (M,5);
 * key_points (M,5,2) or NULL (None).  box_index / kp_index: row of the selected box and of the row whose key points the
 * reference returns (the FIRST row within 2 px of the selected box), -1 = None. */
int fd_face_selection(fd_ctx *ctx, int img_h, int img_w, const float *face_boxes, const float *key_points, int M, int is_enroll,
                      const fd_select_params *params, int *box_index, int *kp_index);
/* The same over the detections of the last fd_detect_batch, one warp per image, asynchronous.  sel_host (B,2) or NULL:
 * {row of the selected detection, row of its key points} as rows of the fd_detect_fetch arrays (-1 = None).  With sel_host
 * the call blocks (and first completes images the detect kernel deferred); without it nothing leaves the device. */
int fd_select_detections(fd_ctx *ctx, const fd_frame *frames, int B, int is_enroll, const fd_select_params *params, int32_t *sel_host);
/* fd_select_detections on NV12 frames (the selection reads only their sizes): the selections of
 * cv::cvtColor(COLOR_YUV2BGR_NV12) followed by fd_select_detections. */
int fd_select_detections_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, int is_enroll, const fd_select_params *params,
                              int32_t *sel_host);
/* fd_select_detections_nv12 for any FD_YUV420_* layout. */
int fd_select_detections_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, int is_enroll,
                                const fd_select_params *params, int32_t *sel_host);
/* fd_select_detections on packed 4:2:2 frames in an FD_YUV422_* layout (the selection reads only their sizes). */
int fd_select_detections_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, int is_enroll, const fd_select_params *params,
                                int32_t *sel_host);
/* fd_select_detections on interleaved RGB-family frames in an FD_RGB_* layout (the selection reads only their sizes). */
int fd_select_detections_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, int is_enroll, const fd_select_params *params,
                             int32_t *sel_host);
/* FaceAlignment::call on the selection of the last fd_select_detections (face_pipeline/pipeline.rs:216-232): one crop per
 * image, crops_dev (B,crop_h,crop_w,3); images without a selection or without key points (the reference's call(.., None)
 * returns Err) get ok = 0 and a zero crop; ok = 2 marks the bbox-crop fallback on the selected box.  M_dev (B,6) / ok_dev (B) optional. */
int fd_align_selected(fd_ctx *ctx, const fd_frame *frames, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);
/* fd_align_selected on NV12 frames: the results of cv::cvtColor(COLOR_YUV2BGR_NV12) followed by fd_align_selected. */
int fd_align_selected_nv12(fd_ctx *ctx, const fd_frame_nv12 *frames, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);
/* fd_align_selected_nv12 for any FD_YUV420_* layout. */
int fd_align_selected_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, uint8_t *crops_dev, double *M_dev,
                             uint8_t *ok_dev);
/* fd_align_selected on packed 4:2:2 frames in an FD_YUV422_* layout. */
int fd_align_selected_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);
/* fd_align_selected on interleaved RGB-family frames in an FD_RGB_* layout. */
int fd_align_selected_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, uint8_t *crops_dev, double *M_dev, uint8_t *ok_dev);

/* ---- SURVEY 8(f) N4: utils::byte_data_to_opencv (utils.rs:8-52 = cv::imdecode(bytes, IMREAD_UNCHANGED)), baseline JPEG ------- */
/* Host-only header parse: image size and luma sampling (11 = 4:4:4, 21 = 4:2:2, 22 = 4:2:0).  FD_ERR_INVALID for streams the
 * decoder does not cover (progressive, arithmetic, grayscale, CMYK, non-interleaved scans): the reference hands those to OpenCV. */
int fd_jpeg_info(const uint8_t *jpeg, size_t nbytes, int *height, int *width, int *subsampling);
/* Decodes B JPEG streams (host memory) into DEVICE-resident BGR frames, bit-identical to cv2.imdecode (libjpeg-turbo islow IDCT,
 * fancy upsampling, 16-bit colour tables).  The streams are copied to the device as they are and entropy-decoded there: one
 * restart interval per thread when a stream carries restart markers less than 32 MCUs apart (DRI / RSTn; the device locates
 * them); otherwise — no markers, or long intervals — unstuffed on the device and decoded by self-synchronising sub-sequences,
 * restart markers serving as known-state
 * boundaries (exact: the rounds run to their fixed point; the call synchronises the ctx stream once per group of rounds, so
 * the count fd_jpeg_last_stats reports is a multiple of the group size).  Only a stream with more than
 * two DC / AC tables is Huffman-decoded on the host.  The host parses headers and tables only (up to n_threads threads, 0 =
 * hardware concurrency, one image per thread).  Dequantisation + IDCT and
 * upsampling + colour conversion are CUDA kernels on the ctx stream.  frames_out[i] = {device pointer owned by the ctx and valid
 * until the next call, h, w, pitch = align16(3w)}: feed it to fd_preprocess_batch / fd_align_detections directly. */
int fd_decode_jpeg_batch(fd_ctx *ctx, const uint8_t *const *jpegs, const size_t *nbytes, int B, int n_threads, fd_frame *frames_out);
/* Of the last fd_decode_jpeg_batch: out[4] = {bytes copied host -> device, images whose Huffman stage ran on the device, images
 * entropy-decoded on the host, (synchronisation rounds << 32) | images decoded by the self-synchronising path}. */
int fd_jpeg_last_stats(const fd_ctx *ctx, int64_t *out);
/* One stream to a HOST buffer (the reference's call shape: one Mat out), blocking.  out_bgr: height rows of `pitch` bytes. */
int fd_imdecode(fd_ctx *ctx, const uint8_t *jpeg, size_t nbytes, uint8_t *out_bgr, int pitch);

/* ---- end-to-end with HOST buffers (bench.py "e2e"): H2D frames + heads, full path, D2H results -------- */
typedef struct fd_host_batch_out {
    int32_t *counts;      /* (B) detections per image */
    float *det;           /* (cap_rows,5) */
    float *landmarks;     /* (cap_rows,10) */
    uint8_t *crops;       /* (cap_rows,crop_h,crop_w,3): one per detection, or (select) one per image */
    float *det_scale;     /* (B) */
    float *tensor;        /* (B,3,image_h,image_w) or NULL: CNN input stays on the device (Triton CUDA-shm) */
    uint8_t *align_mode;  /* (cap_rows) or NULL: per crop 1 = similarity warp, 2 = bbox-crop fallback, 0 = the reference errs (zero crop) */
    int32_t *sel;         /* (B,2) or NULL, select mode: {row of the selected detection, row of its key points}, -1 = None */
    int32_t cap_rows;
    int32_t total;        /* out: detections */
    int32_t n_crops;      /* out: crops written (total, or B in select mode) */
    int64_t h2d_bytes, d2h_bytes; /* out: bytes moved */
} fd_host_batch_out;
enum { FD_UPLOAD_FULL = 0, FD_UPLOAD_ON_DEMAND = 1 };
typedef struct fd_pipeline_opts {
    int32_t select;     /* 0: align every detection (BASELINE config 4).  1: FacePipeline::extract's flow (face_pipeline/pipeline.rs:
                           196-232): FaceSelection::call picks one face per image and only that face is aligned (crop b = image b) */
    int32_t is_enroll;  /* FaceSelection::call is_enroll */
    int32_t upload;     /* FD_UPLOAD_FULL: every frame crosses PCIe whole.  FD_UPLOAD_ON_DEMAND: first only the source rows the
                           letterbox resize reads (1080p -> 640x360: one row in three), then, once the detections are known, only the
                           pixel rectangles the warps read (or the rest of the frame when that is cheaper).  Same results. */
    int32_t heads_zero_copy; /* 1: bbox / landmark head tensors in PINNED host memory are not copied; the detect kernel reads the few
                           sectors it needs (anchors above the threshold) straight from host memory.  Pageable buffers are copied. */
    fd_select_params select_params;
} fd_pipeline_opts;
int fd_pipeline_opts_default(fd_pipeline_opts *opts);   /* select 0, FD_UPLOAD_FULL, heads_zero_copy 0, fd_select_params_default */
/* frames[].data are HOST pointers here (pinned for full PCIe rate); heads_host as in fd_detect_batch but host memory.
 * opts NULL = defaults.  Blocks until the outputs are in host memory. */
int fd_pipeline_host(fd_ctx *ctx, const fd_frame *frames, int B, const float *const *heads_host, int n_heads,
                     float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out);
/* fd_pipeline_host on HOST frames in another layout: the descriptors of fd_preprocess_batch_yuv420 / _yuv422 / _rgb, with
 * host pointers, and the same FD_ERR_INVALID rules (an I420 / YV12 frame's second chroma plane starts (H/2) * pitch_uv after
 * uv, as av_image_alloc and av_frame_get_buffer lay it out).  Every output equals fd_pipeline_host's on cv::cvtColor(
 * COLOR_YUV2BGR_<layout> / RGB2BGR / RGBA2BGR / BGRA2BGR / GRAY2BGR) of the frames, for both upload modes and both flows; only
 * the layout's own bytes cross PCIe (1080p: NV12 / I420 half of BGR's, YUY2 two thirds, GRAY8 one third), and
 * FD_UPLOAD_ON_DEMAND sends per plane only the rows the resize reads and the rectangles the warps read. */
int fd_pipeline_host_yuv420(fd_ctx *ctx, const fd_frame_nv12 *frames, int32_t layout, int B, const float *const *heads_host,
                            int n_heads, float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out);
int fd_pipeline_host_yuv422(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, const float *const *heads_host,
                            int n_heads, float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out);
int fd_pipeline_host_rgb(fd_ctx *ctx, const fd_frame *frames, int32_t layout, int B, const float *const *heads_host,
                         int n_heads, float conf_thr, float iou_thr, const fd_pipeline_opts *opts, fd_host_batch_out *out);
/* The same with the frames given as JPEG streams — FacePipeline::extract's real input (face_pipeline/pipeline.rs:188-196,
 * byte_data_to_opencv): fd_decode_jpeg_batch (host Huffman on n_threads threads, CUDA IDCT / upsampling / colour) on the way in,
 * then the path above with the frames already on the device.  h2d_bytes counts the coefficient upload.  opts->upload is ignored. */
int fd_pipeline_host_jpeg(fd_ctx *ctx, const uint8_t *const *jpegs, const size_t *nbytes, int B, int n_threads,
                          const float *const *heads_host, int n_heads, float conf_thr, float iou_thr, const fd_pipeline_opts *opts,
                          fd_host_batch_out *out);
/* Device tensor written by the last fd_pipeline_host / usable as the CNN input. */
int fd_pipeline_tensor_dev(fd_ctx *ctx, const float **out_nchw_dev);

#ifdef __cplusplus
}
#endif
#endif /* FD_B200_H */
