// fd_internal.cuh — shared internals of libfd_b200.so (context, error plumbing, device helpers).
// Product code: hand-written CUDA for sm_100a.  No CPU fallback anywhere: every entry point needs a GPU.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <utility>
#include <vector>
#include "../../include/fd_b200.h"

#define FD_EXPORT extern "C" __attribute__((visibility("default")))

namespace fd {

void set_error(const std::string &msg);
int fail(int code, const std::string &msg);

#define FD_CUDA(call)                                                                                   \
    do {                                                                                                \
        cudaError_t _e = (call);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            return ::fd::fail(FD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));        \
    } while (0)
#define FD_TRY(call)                 \
    do {                             \
        int _s = (call);             \
        if (_s != FD_OK) return _s;  \
    } while (0)
#define FD_REQUIRE(cond, msg)                                           \
    do {                                                                \
        if (!(cond)) return ::fd::fail(FD_ERR_INVALID, (msg));          \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);  // grows (never shrinks); contents are NOT preserved on growth
    void release();
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};
struct PinnedBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);
    void release();
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// Source pixel format of a frame table; the preprocess and warp kernels are instantiated once per format.
enum SrcFmt : int {
    SRC_BGR = 0,
    SRC_NV12 = 1,     // FrameDev::uv: interleaved U,V
    SRC_NV21 = 2,     // FrameDev::uv: interleaved V,U
    SRC_PLANAR = 3,   // I420 and YV12: FrameDev::uv is the U plane, FrameDev::v_plane() the V plane
};

// Per-frame descriptor as the kernels see it.
struct FrameDev {
    const uint8_t *data;     // BGR pixels, or the Y plane of a 4:2:0 frame
    int h, w, pitch;
    int new_w, new_h;        // letterbox content size
    double scale_x, scale_y; // cv::resize inverse scales
    const uint8_t *uv;       // NV12/NV21: the interleaved chroma plane (h/2 rows of w bytes); planar: the U plane (h/2 rows
                             // of w/2 bytes); nullptr for a BGR frame
    int pitch_uv;            // of the chroma plane(s)
    int v_off;               // planar: start of the V plane minus start of the U plane, in bytes; 0 otherwise (fills the
                             // padding, so the table keeps its size)
    __host__ __device__ const uint8_t *v_plane() const { return uv + v_off; }   // planar only
};
static_assert(sizeof(FrameDev) == 64, "FrameDev: one 64-byte entry per frame");

// Decode geometry passed by value to kernels.
struct DecodeCfg {
    int n_strides, A;
    int stride[FD_MAX_STRIDES];
    int fh[FD_MAX_STRIDES], fw[FD_MAX_STRIDES];
    int pos_off[FD_MAX_STRIDES + 1];    // prefix of H*W over strides
    int anchor_off[FD_MAX_STRIDES + 1]; // prefix of H*W*A
    float base[FD_MAX_STRIDES][FD_MAX_ANCHORS][4];
    float bbox_stds[4], landmark_std;
    float clip_w, clip_h; // image_w-1, image_h-1 as f32 (bbox_transform.rs:30-31)
    int total_pos, total_anchors;
};

}  // namespace fd

struct fd_ctx {
    int device = 0;
    fd_config cfg{};
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;  // copy stream for the host pipeline
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_j[2] = {nullptr, nullptr};   // fd_decode_jpeg_batch: joins of the two copy queues
    cudaEvent_t ev_block = nullptr;  // cudaEventBlockingSync: host waits that sleep instead of spinning (fd_pipeline_host)
    bool blocking_sync = false;
    int num_sms = 0;
    int max_smem_optin = 0;
    int64_t launches = 0;
    bool trace_on = false;       // FD_TRACE=1: an event after every launch, dumped by fd_ctx_synchronize
    bool profile_on = false;     // fd_ctx_profile: same marks, aggregated by fd_ctx_profile_fetch
    std::vector<std::pair<std::string, cudaEvent_t>> trace;
    fd::DecodeCfg dcfg{};

    // generic scratch for the host-pointer drop-in ops
    fd::DevBuf scratch[6];
    fd::PinnedBuf pinned[3];

    // batched pipeline state
    fd::DevBuf frames_dev;       // FrameDev[B]
    int frames_fmt = fd::SRC_BGR;   // source format of the frames in frames_dev (the kernels reading it take that variant)
    fd::DevBuf det_scale_dev;    // float[B]
    fd::DevBuf cand_count;       // int[B] (+ error flags)
    fd::DevBuf cand_keys;        // u64[B][total_anchors]
    fd::DevBuf cand_box;         // float4[B][total_anchors] (indexed by anchor id)
    fd::DevBuf cand_lmk;         // float[B][total_anchors][10]
    fd::DevBuf keep_src;         // int[B][total_anchors] kept anchor ids in pick order
    fd::DevBuf keep_count;       // int[B]
    fd::DevBuf status_dev;       // int[2][8], ping-pong per detect call: [0]=nan flag, [1]=n_big, [2]=total faces, [4..7] scratch
    int status_cur = 0;          // half (0 or 8) the last fd_detect_batch used
    int *status() const { return reinterpret_cast<int *>(status_dev.p) + status_cur; }
    fd::DevBuf big_list;         // int[B] images that need the big path
    fd::DevBuf out_offsets;      // int[B+1]
    fd::DevBuf out_det;          // float[total][5]
    fd::DevBuf out_lmk;          // float[total][10]
    fd::DevBuf out_frame_idx;    // int[total]
    fd::DevBuf align_M;          // double[F][12] (M, inverse)
    fd::DevBuf align_ok;         // u8[F]
    fd::DevBuf tickets;          // int[16] work tickets of the persistent kernels (zero between launches)
    fd::DevBuf select_sel, select_lmk, select_fidx;   // fd_select_detections results: int[B][2], float[B][10], int[B]
    int select_B = 0;
    fd::DevBuf scan_agg;         // u64[B] epoch-tagged kept counts of the fused detect kernel
    unsigned scan_epoch = 0;
    int est_cap = 0;             // faces align_M / align_ok have room for at detect time
    int align_cap_hint = 0;      // largest crop capacity an align call has asked for
    bool crowded = false;        // a detect call met an image with more than 1024 candidates: keep room for the general NMS
    bool share_sms = false;      // fd_ctx_set_sharing: prefer kernels that leave room for another batch's kernels on the SMs
    bool est_valid = false;      // align_M / align_ok hold the estimates of the last fd_detect_batch (fused kernel)
    fd::DevBuf nms_ws[8];        // big-path workspaces
    fd::DevBuf nms_ws_sp[4];     // spatial big-path workspaces
    fd::DevBuf pipe_frames;      // host pipeline: device copies of frames
    fd::DevBuf pipe_heads[3 * FD_MAX_STRIDES];
    fd::DevBuf pipe_tensor;
    fd::DevBuf pipe_crops;
    fd::DevBuf jpeg_coef, jpeg_planes, jpeg_frames, jpeg_desc;   // fd_decode_jpeg_batch: coefficients, component planes, BGR frames
    fd::DevBuf jpeg_raw;                   // self-synchronising decode: segments as received (jpeg_stream holds them unstuffed)
    fd::DevBuf jpeg_stream, jpeg_aux;      // compressed streams, Huffman + restart-interval tables (device entropy decoding)
    fd::DevBuf jpeg_sync, jpeg_flags;      // self-synchronising decode: exit states / block counts per sub-sequence, change flags
    fd::PinnedBuf jpeg_coef_host, jpeg_desc_host, jpeg_aux_host, jpeg_flags_host;
    int jpeg_last_selfsync = 0, jpeg_last_rounds = 0;
    int64_t jpeg_last_h2d = 0;
    int jpeg_last_B = 0;
    int jpeg_last_gpu_entropy = 0;          // images of the last batch whose Huffman stage ran on the device
    fd::DevBuf pipe_mode;        // u8[cap_rows] per-crop align mode of the host pipeline
    int last_B = 0;
    int last_out_cap = 0;
    bool last_fused = false;     // the last fd_detect_batch ran the single fused kernel
    bool detect_pending = false; // results enqueued, NaN check / big-path fix-up not yet done (lazy, at fetch)
    float last_iou = 0.f;
    std::vector<unsigned char> frames_shadow;    // host copy of the descriptor table currently on the device
    std::vector<float> det_scale_shadow;
    // last fd_align_detections call, replayed by the lazy fix-up if the detections it consumed were incomplete
    bool align_replay = false;
    uint8_t *align_crops = nullptr;
    int align_cap = 0;
    double *align_M_out = nullptr;
    uint8_t *align_ok_out = nullptr;
};

namespace fd {

int check_ctx(const fd_ctx *ctx);

void trace_mark(fd_ctx *ctx, const char *file, int line, const char *name);
// Per-launch timing (FD_TRACE=1 or fd_ctx_profile): an event before and after the launch on the ctx stream.
#define FD_LAUNCH_CHECK_NAMED(ctx, name)                                          \
    do {                                                                          \
        (ctx)->launches++;                                                        \
        FD_CUDA(cudaGetLastError());                                              \
        if ((ctx)->trace_on) ::fd::trace_mark((ctx), __FILE__, __LINE__, (name)); \
    } while (0)
#define FD_LAUNCH_CHECK(ctx) FD_LAUNCH_CHECK_NAMED(ctx, nullptr)

// Programmatic dependent launch of a step kernel (preprocess, detect, warp) on the ctx stream: the kernel may be scheduled
// while the kernel before it on the stream is still running, once that one has run griddepcontrol.launch_dependents (or
// exited).  Every kernel launched this way executes pdl_wait() before its first global memory access, which returns when
// the previous grid has completed and its writes are visible — so a caller's kernel that writes frames or heads just
// before the call is still complete and visible, as with a plain launch.  Not with fd_ctx_set_sharing: there another
// batch's kernels fill the SMs this step leaves idle, and CTAs waiting resident for their predecessor would take their place
// (two batches in flight measured 318 k instead of 421 k frames/s); the launch is then a plain one and the wait a no-op.
template <typename... KArgs, typename... Args>
int launch_pdl(fd_ctx *ctx, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = ctx->share_sms ? 0 : 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FD_CUDA(cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...));
    return FD_OK;
}

// ---- device helpers ---------------------------------------------------------------------------------
#ifdef __CUDACC__

// launch_pdl kernels: wait for the previous grid on the stream (complete, writes visible) / let the next one be scheduled
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Maps an f32 to a u32 whose ASCENDING order is the DESCENDING float order (for finite / inf values).
__device__ __forceinline__ uint32_t desc_key(float f) {
    uint32_t u = (f == 0.0f) ? 0u : __float_as_uint(f);  // -0.0 == +0.0 under partial_cmp: one key, stable tie
    uint32_t asc = (u & 0x80000000u) ? ~u : (u | 0x80000000u);  // ascending-orderable
    return ~asc;
}

__device__ __forceinline__ float box_area(float4 b) {
    // (x2 - x1 + 1) * (y2 - y1 + 1), each op rounded separately (nms.rs:46,50)
    return __fmul_rn(__fadd_rn(__fsub_rn(b.z, b.x), 1.0f), __fadd_rn(__fsub_rn(b.w, b.y), 1.0f));
}

// MODE 0: processing::nms::nms — a box survives iff ovr <= thr (nms.rs:58), so suppress = !(ovr <= thr)
// MODE 1: rcnn::cpu_nms — suppress iff ovr >= thr (cpu_nms.rs:48)
//
// Full IEEE expression (used when any box is degenerate / non-finite or thr is negative, NaN or huge):
template <int MODE>
__device__ __forceinline__ bool iou_suppresses_full(const float4 a, const float4 b, const float thr) {
    float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
    float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
    float w = fmaxf(0.0f, __fadd_rn(__fsub_rn(xx2, xx1), 1.0f));
    float h = fmaxf(0.0f, __fadd_rn(__fsub_rn(yy2, yy1), 1.0f));
    float inter = __fmul_rn(w, h);
    float uni = __fsub_rn(__fadd_rn(box_area(a), box_area(b)), inter);
    float ovr = __fdiv_rn(inter, uni);
    return MODE == 0 ? !(ovr <= thr) : (ovr >= thr);
}

// Exact test WITHOUT the division, valid when every box has a finite positive area and thr is an ordinary
// non-negative threshold (the kernels check both):  the float quotient fl(inter/uni) exceeds thr exactly when the real
// quotient lies beyond the midpoint m between thr and its neighbouring float (ties resolved by round-to-even, `incl`).
// inter and uni are the same separately-rounded f32 values the reference computes; m has <= 25 significant bits and
// uni 24, so m*uni is exact in fp64 and the comparison is exact.  Non-intersecting pairs (ovr == +0) exit early.
struct IouParams {
    float thr;
    double m;   // decision boundary
    int incl;   // boundary itself suppresses
    int fast;   // thr admits this test (host side); the kernels AND it with the per-problem box check
};
__device__ __forceinline__ bool iou_suppresses_exact(const float4 a, const float area_a, const float4 b, const float area_b,
                                                     const IouParams &p) {
    float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
    float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
    float w = __fadd_rn(__fsub_rn(xx2, xx1), 1.0f);
    float h = __fadd_rn(__fsub_rn(yy2, yy1), 1.0f);
    if (!(w > 0.0f && h > 0.0f)) return false;
    float inter = __fmul_rn(w, h);
    float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
    double lhs = (double)inter, rhs = p.m * (double)uni;
    return p.incl ? (lhs >= rhs) : (lhs > rhs);
}

__device__ __forceinline__ bool box_is_fast_ok(float4 b) {
    float a = box_area(b);
    return isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w) && isfinite(a) && a > 0.0f;
}

#endif  // __CUDACC__

// stage entry points implemented across the .cu files
int preprocess_launch(fd_ctx *ctx, const FrameDev *frames_dev, int B, float *out_nchw_dev, int max_row_bytes, bool rows_aligned16,
                      int fmt);
int resize_launch(fd_ctx *ctx, const FrameDev &frame, uint8_t *out_dev, int out_h, int out_w);
int crops_to_tensor_launch(fd_ctx *ctx, const uint8_t *crops_dev, const int *count_dev, int F, int in_h, int in_w, int out_h,
                           int out_w, const float *mean_rgb, const float *mul_rgb, float *out_dev);
struct IouParams make_iou_params(float thr, int mode);
int detect_fused_launch(fd_ctx *ctx, const float *const *heads_dev, int B, float conf_thr, float iou_thr, int est_cap, bool *launched);
int nms_batch_small_image(fd_ctx *ctx, int b, int K, float iou_thr);
int decode_launch(fd_ctx *ctx, const float *const *heads_dev, int B, float conf_thr);
int nms_batch_launch(fd_ctx *ctx, int B, float iou_thr);
int nms_batch_big_image(fd_ctx *ctx, int b, int K, float iou_thr);
int finalize_launch(fd_ctx *ctx, int B);
int nms_device(fd_ctx *ctx, const float *dets_dev, int K, int stride_floats, float thr, int mode, bool presorted,
               int32_t *keep_dev, int32_t *num_keep_dev);
int nms_last_stats(fd_ctx *ctx, int32_t out[8]);
int argsort_device(fd_ctx *ctx, const float *scores_as_dets, int n, int stride, int32_t *order_dev, int32_t *flag_dev);
int estimate_launch(fd_ctx *ctx, const float *from_dev, const float *to_dev, const int *count_dev, int F_cap,
                    double *M12_dev, double *M_out_dev, uint8_t *ok_dev, uint8_t *ok_out_dev);
int ticket_buffer(fd_ctx *ctx);
int select_launch(fd_ctx *ctx, const int *offsets_dev, const float *det_dev, const float *lmk_dev, const FrameDev *frames_dev, int B,
                  const fd_select_params *p, int is_enroll, int *sel_dev, float *sel_lmk_dev, int *sel_frame_idx_dev);
int invert_launch(fd_ctx *ctx, const double *M_dev, int F, double *M12_dev, uint8_t *ok_dev);
// inputs of FaceAlignment::call's bbox-crop fallback (face_alignment.rs:64-116), taken by faces whose estimate is empty
struct WarpFallback {
    const float *bbox = nullptr;   // device rows x1,y1,x2,y2,... bbox_stride floats apart; nullptr: bbox == None
    int bbox_stride = 4;
    const int *sel = nullptr;      // optional device (F,2) {bbox row, key-point row}; key-point row < 0: landmarks == None -> Err
    uint8_t *mode_out = nullptr;   // optional device (F): 1 warp, 2 fallback crop, 0 the reference returns Err (zero crop)
};
int warp_launch(fd_ctx *ctx, const FrameDev *frames_dev, const int32_t *frame_idx_dev, const double *M12_dev,
                const uint8_t *ok_dev, const int *count_dev, int F_cap, uint8_t *crops_dev, int cw, int ch, const WarpFallback &fb,
                int fmt);

}  // namespace fd
