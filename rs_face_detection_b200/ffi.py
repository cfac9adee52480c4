"""ctypes binding of libfd_b200.so — the same C ABI (include/fd_b200.h) a Rust `build.rs` links.

There is NO CPU fallback: importing works without a GPU (so the symbol table can be checked), but creating a
Context raises FdError unless a CUDA device is present, and a missing library raises at load time.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FD_B200_LIB") or os.path.join(_HERE, "libfd_b200.so")   # FD_B200_LIB: A/B a differently built library

FD_MAX_STRIDES = 8
FD_MAX_ANCHORS = 4
FD_OK, FD_ERR_INVALID, FD_ERR_CUDA, FD_ERR_NAN_SCORE, FD_ERR_CAPACITY, FD_ERR_NO_DEVICE, FD_ERR_ESTIMATE = range(7)

c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)
c_i32p = C.POINTER(C.c_int32)
c_u8p = C.POINTER(C.c_uint8)


class FdError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("fd_b200 error %d: %s" % (code, msg))
        self.code = code


class FdConfig(C.Structure):
    _fields_ = [
        ("image_w", C.c_int32), ("image_h", C.c_int32),
        ("conf_thr", C.c_float), ("iou_thr", C.c_float),
        ("n_strides", C.c_int32), ("strides", C.c_int32 * FD_MAX_STRIDES),
        ("num_anchors", C.c_int32),
        ("base_anchors", C.c_float * (FD_MAX_STRIDES * FD_MAX_ANCHORS * 4)),
        ("pixel_means", C.c_float * 3), ("pixel_stds", C.c_float * 3), ("pixel_scale", C.c_float),
        ("bbox_stds", C.c_float * 4), ("landmark_std", C.c_float),
        ("crop_w", C.c_int32), ("crop_h", C.c_int32),
        ("template_landmarks", C.c_float * 10),
    ]


class FdFrame(C.Structure):
    _fields_ = [("data", C.c_void_p), ("height", C.c_int32), ("width", C.c_int32), ("pitch", C.c_int32)]


class FdFrameNV12(C.Structure):
    _fields_ = [("y", C.c_void_p), ("uv", C.c_void_p), ("height", C.c_int32), ("width", C.c_int32), ("pitch_y", C.c_int32),
                ("pitch_uv", C.c_int32)]


class FdAnchorCfg(C.Structure):
    _fields_ = [("stride", C.c_int32), ("base_size", C.c_int32), ("n_ratios", C.c_int32), ("n_scales", C.c_int32),
                ("ratios", C.c_float * 8), ("scales", C.c_float * 8), ("allowed_border", C.c_int32)]


class FdDetView(C.Structure):
    _fields_ = [("counts_dev", C.c_void_p), ("offsets_dev", C.c_void_p), ("det_dev", C.c_void_p),
                ("landmarks_dev", C.c_void_p), ("frame_idx_dev", C.c_void_p), ("candidates_dev", C.c_void_p)]


class FdSelectParams(C.Structure):
    _fields_ = [("margin_center_left_ratio", C.c_float), ("margin_center_right_ratio", C.c_float),
                ("margin_edge_ratio", C.c_float), ("minimum_face_ratio", C.c_float)]


class FdHostBatchOut(C.Structure):
    _fields_ = [("counts", c_i32p), ("det", c_f32p), ("landmarks", c_f32p), ("crops", c_u8p), ("det_scale", c_f32p),
                ("tensor", c_f32p), ("align_mode", c_u8p), ("sel", c_i32p), ("cap_rows", C.c_int32), ("total", C.c_int32),
                ("n_crops", C.c_int32), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64)]


FD_UPLOAD_FULL, FD_UPLOAD_ON_DEMAND = 0, 1
# layouts of a 4:2:0 frame for the *_yuv420 calls (include/fd_b200.h): what an fd_frame_nv12's `uv` points to
FD_YUV420_NV12, FD_YUV420_NV21, FD_YUV420_I420, FD_YUV420_YV12 = 0, 1, 2, 3


class FdPipelineOpts(C.Structure):
    _fields_ = [("select", C.c_int32), ("is_enroll", C.c_int32), ("upload", C.c_int32), ("heads_zero_copy", C.c_int32),
                ("select_params", FdSelectParams)]


# every symbol include/fd_b200.h declares (tests/test_abi.py checks the header against this list and the .so)
SYMBOLS = [
    "fd_abi_version", "fd_last_error", "fd_config_default", "fd_device_count", "fd_ctx_create", "fd_ctx_destroy",
    "fd_ctx_get_config", "fd_ctx_total_anchors", "fd_ctx_stream", "fd_ctx_synchronize", "fd_ctx_launch_count",
    "fd_ctx_profile", "fd_ctx_profile_fetch", "fd_ctx_set_sharing",
    "fd_dev_alloc", "fd_dev_free", "fd_host_alloc_pinned", "fd_host_free_pinned", "fd_memcpy_h2d", "fd_memcpy_d2h",
    "fd_memcpy_h2d_async", "fd_memcpy_d2h_async", "fd_memset_dev",
    "fd_generate_anchors", "fd_generate_anchors2", "fd_generate_anchors_fpn", "fd_generate_anchors_fpn2",
    "fd_nms", "fd_nms_last_stats", "fd_cpu_nms", "fd_nms_sorted", "_nms", "_set_device", "fd_argsort_descending", "fd_anchors_plane",
    "fd_bbox_pred", "fd_nonlinear_pred", "fd_landmark_pred", "fd_clip_boxes", "fd_clip_points", "fd_iou_pred",
    "fd_nonlinear_transform", "fd_bbox_overlaps", "fd_letterbox_geometry", "fd_preprocess", "fd_resize_linear",
    "fd_detect", "fd_estimate_affine_partial_2d", "fd_warp_affine", "fd_align",
    "fd_nms_device", "fd_preprocess_batch", "fd_detect_batch", "fd_detect_fetch", "fd_detect_view", "fd_detect_last_stats", "fd_align_batch",
    "fd_align_detections", "fd_crops_to_tensor", "fd_model_preprocess", "fd_detect_batch_raw", "fd_select_params_default", "fd_face_selection",
    "fd_select_detections", "fd_align_selected", "fd_jpeg_info", "fd_decode_jpeg_batch", "fd_jpeg_last_stats", "fd_imdecode", "fd_pipeline_opts_default", "fd_pipeline_host", "fd_pipeline_host_jpeg", "fd_pipeline_tensor_dev",
    "fd_preprocess_batch_nv12", "fd_align_batch_nv12", "fd_align_detections_nv12", "fd_select_detections_nv12", "fd_align_selected_nv12",
    "fd_preprocess_batch_yuv420", "fd_align_batch_yuv420", "fd_align_detections_yuv420", "fd_select_detections_yuv420",
    "fd_align_selected_yuv420",
]

_lib = None


def load():
    """Loads the CUDA library.  Raises if it has not been built: the product path never degrades to a CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FdError(FD_ERR_NO_DEVICE, "libfd_b200.so is not built (run `python -m rs_face_detection_b200.build`); "
                                            "there is no CPU fallback")
        _lib = C.CDLL(LIB_PATH)
        _lib.fd_last_error.restype = C.c_char_p
        _lib.fd_ctx_stream.restype = C.c_void_p
        for name in SYMBOLS:
            getattr(_lib, name)  # AttributeError here == ABI drift
    return _lib


def _chk(rc):
    if rc != FD_OK:
        raise FdError(rc, load().fd_last_error().decode("utf-8", "replace"))


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a, t):
    return a.ctypes.data_as(t)


def _devptr(x):
    """int | torch.Tensor | DeviceBuffer -> raw device address"""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    if hasattr(x, "ptr"):
        return x.ptr
    raise TypeError("not a device pointer: %r" % (x,))


class PinnedArray:
    """numpy view over page-locked host memory (fd_host_alloc_pinned): full-rate DMA source and, for the head tensors,
    directly readable by the kernels (fd_pipeline_opts.heads_zero_copy).  Keep the object alive while the array is in use."""

    def __init__(self, shape, dtype):
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _chk(load().fd_host_alloc_pinned(C.c_size_t(max(self.nbytes, 1)), C.byref(p)))
        self.ptr = p.value
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self.ptr:
            self.array = None
            load().fd_host_free_pinned(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def pinned_like(arr):
    """-> PinnedArray holding a copy of arr"""
    pa = PinnedArray(arr.shape, arr.dtype)
    pa.array[...] = arr
    return pa


def default_config():
    cfg = FdConfig()
    _chk(load().fd_config_default(C.byref(cfg)))
    return cfg


def device_count():
    n = C.c_int(0)
    rc = load().fd_device_count(C.byref(n))
    return n.value if rc == FD_OK else 0


# ---- init-time anchor tables (host arithmetic inside the library; generate_anchors.rs) ----------------------------
def generate_anchors2(base_size, ratios, scales, stride=0, dense_anchor=False):
    ratios, scales = _f32(ratios), _f32(scales)
    out = np.empty((len(ratios) * len(scales) * 2, 4), np.float32)
    n = C.c_int()
    _chk(load().fd_generate_anchors2(int(base_size), _ptr(ratios, c_f32p), len(ratios), _ptr(scales, c_f32p), len(scales),
                                     int(stride), int(dense_anchor), _ptr(out, c_f32p), C.byref(n)))
    return out[:n.value].copy()


def generate_anchors(base_size, ratios, scales):
    return generate_anchors2(base_size, ratios, scales, 0, False)


def generate_anchors_fpn(base_size, ratios, scales):
    bs = np.ascontiguousarray(base_size, np.int32)
    ratios, scales = _f32(ratios), _f32(scales)
    out = np.empty((len(bs), 4), np.float32)
    _chk(load().fd_generate_anchors_fpn(_ptr(bs, c_i32p), _ptr(ratios, c_f32p), _ptr(scales, c_f32p), len(bs), _ptr(out, c_f32p)))
    return [out[i:i + 1].copy() for i in range(len(bs))]


def generate_anchors_fpn2(dense_anchor, cfg):
    """cfg: {"32": {"base_size":16,"ratios":[1.0],"scales":[32,16],"allowed_border":9999}, ...} (generate_anchors.rs:116)."""
    arr = (FdAnchorCfg * len(cfg))()
    for i, (k, v) in enumerate(cfg.items()):
        arr[i].stride = int(k)
        arr[i].base_size = int(v["base_size"])
        arr[i].n_ratios, arr[i].n_scales = len(v["ratios"]), len(v["scales"])
        for j, r in enumerate(v["ratios"]):
            arr[i].ratios[j] = r
        for j, s in enumerate(v["scales"]):
            arr[i].scales[j] = s
        arr[i].allowed_border = int(v.get("allowed_border", 9999))
    out = np.empty((len(cfg) * 128, 4), np.float32)
    rows = (C.c_int * len(cfg))()
    strides = (C.c_int * len(cfg))()
    _chk(load().fd_generate_anchors_fpn2(int(dense_anchor), arr, len(cfg), _ptr(out, c_f32p), rows, strides))
    res, r0 = [], 0
    for i in range(len(cfg)):
        res.append(out[r0:r0 + rows[i]].copy())
        r0 += rows[i]
    return res


class DeviceBuffer:
    """Device allocation owned through the C ABI (no torch needed)."""

    def __init__(self, ctx, nbytes):
        self.ctx, self.nbytes = ctx, int(nbytes)
        p = C.c_void_p()
        _chk(load().fd_dev_alloc(ctx.handle, C.c_size_t(max(self.nbytes, 1)), C.byref(p)))
        self.ptr = p.value

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        _chk(load().fd_memcpy_h2d(self.ctx.handle, C.c_void_p(self.ptr), arr.ctypes.data_as(C.c_void_p), C.c_size_t(arr.nbytes)))
        return self

    def download(self, shape, dtype):
        out = np.empty(shape, dtype)
        assert out.nbytes <= self.nbytes
        _chk(load().fd_memcpy_d2h(self.ctx.handle, out.ctypes.data_as(C.c_void_p), C.c_void_p(self.ptr), C.c_size_t(out.nbytes)))
        return out

    def free(self):
        if self.ptr:
            load().fd_dev_free(self.ctx.handle, C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One fd_ctx: one GPU, one stream.  Every method is a thin call into the C ABI."""

    def __init__(self, device=0, cfg=None):
        self.lib = load()
        self.handle = C.c_void_p()
        self.cfg = cfg if cfg is not None else default_config()
        _chk(self.lib.fd_ctx_create(int(device), C.byref(self.cfg), C.byref(self.handle)))
        n = C.c_int32()
        _chk(self.lib.fd_ctx_total_anchors(self.handle, C.byref(n)))
        self.total_anchors = n.value
        self.device = device

    def close(self):
        if self.handle:
            self.lib.fd_ctx_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- plumbing
    def synchronize(self):
        _chk(self.lib.fd_ctx_synchronize(self.handle))

    def stream(self):
        return self.lib.fd_ctx_stream(self.handle)

    def launch_count(self):
        n = C.c_int64()
        _chk(self.lib.fd_ctx_launch_count(self.handle, C.byref(n)))
        return n.value

    def set_sharing(self, contexts_in_flight):
        _chk(self.lib.fd_ctx_set_sharing(self.handle, int(contexts_in_flight)))

    def profile(self, enable=True):
        """per-kernel CUDA-event marks on the ctx stream (bench.py's per-kernel lines)"""
        _chk(self.lib.fd_ctx_profile(self.handle, 1 if enable else 0))

    def profile_fetch(self):
        """{kernel name: (launches, total_us)} since the last fetch"""
        buf = C.create_string_buffer(1 << 16)
        _chk(self.lib.fd_ctx_profile_fetch(self.handle, buf, C.c_size_t(len(buf))))
        out = {}
        for line in buf.value.decode().splitlines():
            name, n, us = line.rsplit(" ", 2)
            out[name] = (int(n), float(us))
        return out

    def alloc(self, nbytes):
        return DeviceBuffer(self, nbytes)

    def to_device(self, arr):
        arr = np.ascontiguousarray(arr)
        return DeviceBuffer(self, arr.nbytes).upload(arr)

    def feat_shapes(self):
        c = self.cfg
        return [((c.image_h + c.strides[s] - 1) // c.strides[s], (c.image_w + c.strides[s] - 1) // c.strides[s])
                for s in range(c.n_strides)]

    # ---- drop-in single ops (host arrays)
    def _nms(self, fn, dets, thresh):
        dets = _f32(dets).reshape(-1, 5)
        keep = np.empty(max(dets.shape[0], 1), np.int32)
        n = C.c_int()
        _chk(fn(self.handle, _ptr(dets, c_f32p), dets.shape[0], C.c_float(thresh), _ptr(keep, c_i32p), C.byref(n)))
        return keep[:n.value].copy()

    def nms(self, dets, thresh):
        return self._nms(self.lib.fd_nms, dets, thresh)

    def nms_last_stats(self):
        out = np.zeros(8, np.int32)
        _chk(self.lib.fd_nms_last_stats(self.handle, _ptr(out, c_i32p)))
        return dict(spatial=int(out[0]), kept=int(out[1]), epochs=int(out[2]), grid=(int(out[3]), int(out[4])),
                    cell=float(out[5:6].view(np.float32)[0]))

    def cpu_nms(self, dets, thresh):
        return self._nms(self.lib.fd_cpu_nms, dets, thresh)

    def nms_sorted(self, boxes, thresh):
        boxes = _f32(boxes)
        keep = np.empty(max(boxes.shape[0], 1), np.int32)
        n = C.c_int()
        _chk(self.lib.fd_nms_sorted(self.handle, _ptr(boxes, c_f32p), boxes.shape[0], boxes.shape[1] if boxes.ndim == 2 else 5,
                                    C.c_float(thresh), _ptr(keep, c_i32p), C.byref(n)))
        return keep[:n.value].copy()

    def argsort_descending(self, scores):
        scores = _f32(scores).ravel()
        order = np.empty(len(scores), np.int32)
        _chk(self.lib.fd_argsort_descending(self.handle, _ptr(scores, c_f32p), len(scores), _ptr(order, c_i32p)))
        return order

    def anchors_plane(self, height, width, stride, base):
        base = _f32(base)
        out = np.empty((height, width, base.shape[0], 4), np.float32)
        _chk(self.lib.fd_anchors_plane(self.handle, height, width, stride, _ptr(base, c_f32p), base.shape[0], _ptr(out, c_f32p)))
        return out

    def _pred(self, fn, boxes, deltas):
        boxes, deltas = _f32(boxes), _f32(deltas)
        if boxes.shape[0] == 0:
            return np.zeros((0, deltas.shape[1]), np.float32)
        out = np.empty_like(deltas)
        _chk(fn(self.handle, _ptr(boxes, c_f32p), _ptr(deltas, c_f32p), boxes.shape[0], deltas.shape[1], _ptr(out, c_f32p)))
        return out

    def bbox_pred(self, boxes, deltas):
        return self._pred(self.lib.fd_bbox_pred, boxes, deltas)

    def nonlinear_pred(self, boxes, deltas):
        return self._pred(self.lib.fd_nonlinear_pred, boxes, deltas)

    def landmark_pred(self, boxes, deltas):
        boxes, deltas = _f32(boxes), _f32(deltas)
        shape = deltas.shape
        if boxes.shape[0] == 0:
            return np.zeros((0,) + tuple(shape[1:]), np.float32)
        out = np.empty_like(deltas)
        _chk(self.lib.fd_landmark_pred(self.handle, _ptr(boxes, c_f32p), _ptr(deltas, c_f32p), boxes.shape[0], _ptr(out, c_f32p)))
        return out.reshape(shape)

    def clip_boxes(self, boxes, im_shape):
        boxes = _f32(boxes).copy()
        _chk(self.lib.fd_clip_boxes(self.handle, _ptr(boxes, c_f32p), boxes.shape[0], boxes.shape[1], int(im_shape[0]), int(im_shape[1])))
        return boxes

    def clip_points(self, points, im_shape):
        points = _f32(points).copy()
        _chk(self.lib.fd_clip_points(self.handle, _ptr(points, c_f32p), points.shape[0], points.shape[1], int(im_shape[0]), int(im_shape[1])))
        return points

    def iou_pred(self, boxes, deltas, num_classes):
        boxes, deltas = _f32(boxes), _f32(deltas)
        out = np.empty_like(deltas)
        _chk(self.lib.fd_iou_pred(self.handle, _ptr(boxes, c_f32p), _ptr(deltas, c_f32p), boxes.shape[0], deltas.shape[1],
                                  int(num_classes), _ptr(out, c_f32p)))
        return out

    def nonlinear_transform(self, ex, gt):
        ex, gt = _f32(ex), _f32(gt)
        out = np.empty((ex.shape[0], 4), np.float32)
        _chk(self.lib.fd_nonlinear_transform(self.handle, _ptr(ex, c_f32p), _ptr(gt, c_f32p), ex.shape[0], _ptr(out, c_f32p)))
        return out

    def bbox_overlaps(self, boxes, query):
        boxes, query = _f32(boxes), _f32(query)
        out = np.empty((boxes.shape[0], query.shape[0]), np.float32)
        _chk(self.lib.fd_bbox_overlaps(self.handle, _ptr(boxes, c_f32p), boxes.shape[0], _ptr(query, c_f32p), query.shape[0], _ptr(out, c_f32p)))
        return out

    def letterbox_geometry(self, h, w):
        nw, nh, sc = C.c_int(), C.c_int(), C.c_float()
        _chk(self.lib.fd_letterbox_geometry(self.handle, h, w, C.byref(nw), C.byref(nh), C.byref(sc)))
        return nw.value, nh.value, np.float32(sc.value)

    def preprocess(self, img):
        img = np.ascontiguousarray(img, np.uint8)
        out = np.empty((1, 3, self.cfg.image_h, self.cfg.image_w), np.float32)
        sc = C.c_float()
        _chk(self.lib.fd_preprocess(self.handle, _ptr(img, c_u8p), img.shape[0], img.shape[1], img.strides[0], _ptr(out, c_f32p), C.byref(sc)))
        return out, np.float32(sc.value)

    def resize_linear(self, img, dsize):
        img = np.ascontiguousarray(img, np.uint8)
        dw, dh = dsize
        out = np.empty((dh, dw, 3), np.uint8)
        _chk(self.lib.fd_resize_linear(self.handle, _ptr(img, c_u8p), img.shape[0], img.shape[1], img.strides[0], _ptr(out, c_u8p), dh, dw))
        return out

    def detect(self, heads, det_scale, conf_thr=None, iou_thr=None):
        """heads: 9 host arrays of ONE image -> det (M,5), landmarks (M,5,2)."""
        heads = [_f32(h) for h in heads]
        arr = (c_f32p * len(heads))(*[_ptr(h, c_f32p) for h in heads])
        cap = self.total_anchors
        det = np.empty((cap, 5), np.float32)
        lmk = np.empty((cap, 10), np.float32)
        n = C.c_int()
        _chk(self.lib.fd_detect(self.handle, arr, len(heads), C.c_float(det_scale),
                                C.c_float(self.cfg.conf_thr if conf_thr is None else conf_thr),
                                C.c_float(self.cfg.iou_thr if iou_thr is None else iou_thr),
                                _ptr(det, c_f32p), _ptr(lmk, c_f32p), cap, C.byref(n)))
        return det[:n.value].copy(), lmk[:n.value].reshape(-1, 5, 2).copy()

    def estimate_affine_partial_2d(self, src, dst=None):
        src = _f32(src).reshape(-1, 10)
        n = src.shape[0]
        M = np.empty((n, 2, 3), np.float64)
        ok = np.zeros(n, np.uint8)
        d = None
        if dst is not None:
            d = _f32(np.broadcast_to(_f32(dst).reshape(-1, 10), (n, 10)))
        _chk(self.lib.fd_estimate_affine_partial_2d(self.handle, _ptr(src, c_f32p), _ptr(d, c_f32p) if d is not None else None,
                                                    n, _ptr(M, c_f64p), _ptr(ok, c_u8p)))
        return M, ok

    def warp_affine(self, img, M, dsize=(112, 112)):
        img = np.ascontiguousarray(img, np.uint8)
        M = np.ascontiguousarray(M, np.float64).reshape(6)
        dw, dh = dsize
        out = np.empty((dh, dw, 3), np.uint8)
        _chk(self.lib.fd_warp_affine(self.handle, _ptr(img, c_u8p), img.shape[0], img.shape[1], img.strides[0], _ptr(M, c_f64p),
                                     _ptr(out, c_u8p), dh, dw))
        return out

    def align(self, img, landmarks, bbox=None, with_mode=False):
        """FaceAlignment::call: -> (crop, M) or, with_mode, (crop, M, mode): mode 1 = similarity warp, 2 = bbox-crop
        fallback (face_alignment.rs:64-116; M is None then).  Raises FdError where the reference returns Err."""
        img = np.ascontiguousarray(img, np.uint8)
        lmk = _f32(landmarks).reshape(10) if landmarks is not None else None
        bb = _f32(bbox).reshape(-1)[:4].copy() if bbox is not None else None
        out = np.empty((self.cfg.crop_h, self.cfg.crop_w, 3), np.uint8)
        M = np.empty((2, 3), np.float64)
        mode = C.c_int(0)
        _chk(self.lib.fd_align(self.handle, _ptr(img, c_u8p), img.shape[0], img.shape[1], img.strides[0],
                               _ptr(bb, c_f32p) if bb is not None else None, _ptr(lmk, c_f32p) if lmk is not None else None,
                               _ptr(out, c_u8p), _ptr(M, c_f64p), C.byref(mode)))
        if mode.value != 1:
            M = None
        return (out, M, mode.value) if with_mode else (out, M)

    # ---- batched, device-resident
    @staticmethod
    def _frames(frames):
        """frames: list of (dev_ptr, h, w, pitch), or the fd_frame array a previous frame_table() call built"""
        if isinstance(frames, C.Array):
            return frames
        arr = (FdFrame * len(frames))()
        for i, (p, h, w, pitch) in enumerate(frames):
            arr[i].data, arr[i].height, arr[i].width, arr[i].pitch = _devptr(p), h, w, pitch
        return arr

    @staticmethod
    def _frames_nv12(frames):
        """frames: list of (y_dev_ptr, uv_dev_ptr, h, w, pitch_y, pitch_uv), or an fd_frame_nv12 array from frame_table_nv12()"""
        if isinstance(frames, C.Array):
            return frames
        arr = (FdFrameNV12 * len(frames))()
        for i, (y, uv, h, w, py, puv) in enumerate(frames):
            arr[i].y, arr[i].uv, arr[i].height, arr[i].width, arr[i].pitch_y, arr[i].pitch_uv = _devptr(y), _devptr(uv), h, w, py, puv
        return arr

    def frame_table_nv12(self, frames):
        return self._frames_nv12(frames)

    def frame_table(self, frames):
        """Builds the fd_frame array once (a streaming caller reuses it: filling 64 ctypes structs per call costs more
        host time than the kernels they describe)."""
        return self._frames(frames)

    @staticmethod
    def head_table(heads_dev):
        return (C.c_void_p * len(heads_dev))(*[_devptr(h) for h in heads_dev])

    def nms_device(self, dets_dev, K, thresh, keep_dev, num_keep_dev):
        _chk(self.lib.fd_nms_device(self.handle, C.c_void_p(_devptr(dets_dev)), int(K), C.c_float(thresh),
                                    C.c_void_p(_devptr(keep_dev)), C.c_void_p(_devptr(num_keep_dev))))

    def preprocess_batch(self, frames, out_dev):
        arr = self._frames(frames)
        ds = np.empty(len(frames), np.float32)
        _chk(self.lib.fd_preprocess_batch(self.handle, arr, len(frames), C.c_void_p(_devptr(out_dev)), _ptr(ds, c_f32p)))
        return ds

    def detect_batch(self, heads_dev, B, det_scale, conf_thr=None, iou_thr=None):
        ptrs = heads_dev if isinstance(heads_dev, C.Array) else self.head_table(heads_dev)
        ds = _f32(det_scale)
        _chk(self.lib.fd_detect_batch(self.handle, ptrs, len(heads_dev), B, _ptr(ds, c_f32p),
                                      C.c_float(self.cfg.conf_thr if conf_thr is None else conf_thr),
                                      C.c_float(self.cfg.iou_thr if iou_thr is None else iou_thr)))

    def detect_fetch(self, B, cap_rows=None):
        cap = self.total_anchors * B if cap_rows is None else cap_rows
        tot = C.c_int()
        counts = np.empty(B, np.int32)
        # first query the total so the host buffers can be sized
        _chk(self.lib.fd_detect_fetch(self.handle, _ptr(counts, c_i32p), None, None, 0, C.byref(tot)))
        n = min(tot.value, cap)
        det = np.empty((max(n, 1), 5), np.float32)
        lmk = np.empty((max(n, 1), 10), np.float32)
        _chk(self.lib.fd_detect_fetch(self.handle, _ptr(counts, c_i32p), _ptr(det, c_f32p), _ptr(lmk, c_f32p), max(n, 1), C.byref(tot)))
        return counts, det[:tot.value], lmk[:tot.value].reshape(-1, 5, 2)

    def detect_view(self):
        v = FdDetView()
        _chk(self.lib.fd_detect_view(self.handle, C.byref(v)))
        return v

    def detect_last_stats(self):
        """{deferred_images, max_candidates, total_candidates, faces_on_device, fused, crowded} of the last detect_batch"""
        out = np.zeros(8, np.int32)
        _chk(self.lib.fd_detect_last_stats(self.handle, _ptr(out, c_i32p)))
        return dict(deferred_images=int(out[0]), max_candidates=int(out[1]), total_candidates=int(out[2]), faces_on_device=int(out[3]),
                    fused=bool(out[4]), crowded=bool(out[5]))

    def align_batch(self, frames, landmarks_dev, frame_idx_dev, F, crops_dev, M_dev=None, ok_dev=None, bbox_dev=None):
        arr = self._frames(frames)
        _chk(self.lib.fd_align_batch(self.handle, arr, len(frames), C.c_void_p(_devptr(landmarks_dev)),
                                     C.c_void_p(_devptr(frame_idx_dev)), C.c_void_p(_devptr(bbox_dev)), F,
                                     C.c_void_p(_devptr(crops_dev)), C.c_void_p(_devptr(M_dev)), C.c_void_p(_devptr(ok_dev))))

    def align_detections(self, frames, crops_dev, cap_faces, M_dev=None, ok_dev=None):
        arr = self._frames(frames)
        _chk(self.lib.fd_align_detections(self.handle, arr, len(frames), C.c_void_p(_devptr(crops_dev)), cap_faces,
                                          C.c_void_p(_devptr(M_dev)), C.c_void_p(_devptr(ok_dev))))

    # ---- NV12 video frames: the results of cv2.cvtColor(COLOR_YUV2BGR_NV12) followed by the BGR call
    def preprocess_batch_nv12(self, frames, out_dev):
        arr = self._frames_nv12(frames)
        ds = np.empty(len(frames), np.float32)
        _chk(self.lib.fd_preprocess_batch_nv12(self.handle, arr, len(frames), C.c_void_p(_devptr(out_dev)), _ptr(ds, c_f32p)))
        return ds

    def align_batch_nv12(self, frames, landmarks_dev, frame_idx_dev, F, crops_dev, M_dev=None, ok_dev=None, bbox_dev=None):
        arr = self._frames_nv12(frames)
        _chk(self.lib.fd_align_batch_nv12(self.handle, arr, len(frames), C.c_void_p(_devptr(landmarks_dev)),
                                          C.c_void_p(_devptr(frame_idx_dev)), C.c_void_p(_devptr(bbox_dev)), F,
                                          C.c_void_p(_devptr(crops_dev)), C.c_void_p(_devptr(M_dev)), C.c_void_p(_devptr(ok_dev))))

    def align_detections_nv12(self, frames, crops_dev, cap_faces, M_dev=None, ok_dev=None):
        arr = self._frames_nv12(frames)
        _chk(self.lib.fd_align_detections_nv12(self.handle, arr, len(frames), C.c_void_p(_devptr(crops_dev)), cap_faces,
                                               C.c_void_p(_devptr(M_dev)), C.c_void_p(_devptr(ok_dev))))

    def select_detections_nv12(self, frames, is_enroll=False, params=None, fetch=True):
        arr = self._frames_nv12(frames)
        prm = None if params is None else (C.c_float * 4)(*params)
        sel = np.empty((len(frames), 2), np.int32) if fetch else None
        _chk(self.lib.fd_select_detections_nv12(self.handle, arr, len(frames), int(bool(is_enroll)), prm,
                                                None if sel is None else _ptr(sel, c_i32p)))
        return sel

    def align_selected_nv12(self, frames, crops_dev, M_dev=None, ok_dev=None):
        arr = self._frames_nv12(frames)
        _chk(self.lib.fd_align_selected_nv12(self.handle, arr, len(frames), C.c_void_p(_devptr(crops_dev)), C.c_void_p(_devptr(M_dev)),
                                             C.c_void_p(_devptr(ok_dev))))

    # ---- 4:2:0 frames in any FD_YUV420_* layout (descriptors from frame_table_nv12): the results of cv2.cvtColor(
    # COLOR_YUV2BGR_NV12 / _NV21 / _I420 / _YV12) followed by the BGR call
    def preprocess_batch_yuv420(self, frames, layout, out_dev):
        arr = self._frames_nv12(frames)
        ds = np.empty(len(frames), np.float32)
        _chk(self.lib.fd_preprocess_batch_yuv420(self.handle, arr, int(layout), len(frames), C.c_void_p(_devptr(out_dev)),
                                                 _ptr(ds, c_f32p)))
        return ds

    def align_batch_yuv420(self, frames, layout, landmarks_dev, frame_idx_dev, F, crops_dev, M_dev=None, ok_dev=None, bbox_dev=None):
        arr = self._frames_nv12(frames)
        _chk(self.lib.fd_align_batch_yuv420(self.handle, arr, int(layout), len(frames), C.c_void_p(_devptr(landmarks_dev)),
                                            C.c_void_p(_devptr(frame_idx_dev)), C.c_void_p(_devptr(bbox_dev)), F,
                                            C.c_void_p(_devptr(crops_dev)), C.c_void_p(_devptr(M_dev)), C.c_void_p(_devptr(ok_dev))))

    def align_detections_yuv420(self, frames, layout, crops_dev, cap_faces, M_dev=None, ok_dev=None):
        arr = self._frames_nv12(frames)
        _chk(self.lib.fd_align_detections_yuv420(self.handle, arr, int(layout), len(frames), C.c_void_p(_devptr(crops_dev)), cap_faces,
                                                 C.c_void_p(_devptr(M_dev)), C.c_void_p(_devptr(ok_dev))))

    def select_detections_yuv420(self, frames, layout, is_enroll=False, params=None, fetch=True):
        arr = self._frames_nv12(frames)
        prm = None if params is None else (C.c_float * 4)(*params)
        sel = np.empty((len(frames), 2), np.int32) if fetch else None
        _chk(self.lib.fd_select_detections_yuv420(self.handle, arr, int(layout), len(frames), int(bool(is_enroll)), prm,
                                                  None if sel is None else _ptr(sel, c_i32p)))
        return sel

    def align_selected_yuv420(self, frames, layout, crops_dev, M_dev=None, ok_dev=None):
        arr = self._frames_nv12(frames)
        _chk(self.lib.fd_align_selected_yuv420(self.handle, arr, int(layout), len(frames), C.c_void_p(_devptr(crops_dev)),
                                               C.c_void_p(_devptr(M_dev)), C.c_void_p(_devptr(ok_dev))))

    # ---- N2: Triton raw_output_contents
    def detect_batch_raw(self, raw, shapes, det_scale, conf_thr, iou_thr):
        """raw: list of bytes-like objects (little-endian f32), shapes: list of 4-tuples (N,C,H,W)"""
        n = len(raw)
        keep = [np.frombuffer(r, np.uint8) if not isinstance(r, np.ndarray) else r for r in raw]
        ptrs = (C.c_void_p * n)(*[k.ctypes.data for k in keep])
        nb = (C.c_size_t * n)(*[k.nbytes for k in keep])
        sh = ((C.c_int64 * 4) * n)(*[(C.c_int64 * 4)(*s_) for s_ in shapes])
        ds = _f32(det_scale)
        _chk(self.lib.fd_detect_batch_raw(self.handle, ptrs, nb, sh, n, _ptr(ds, c_f32p), C.c_float(conf_thr), C.c_float(iou_thr)))

    # ---- N3: FaceSelection
    def face_selection(self, img_hw, face_boxes, key_points=None, is_enroll=False, params=None):
        fb = _f32(face_boxes).reshape(-1, 5)
        kp = None if key_points is None else _f32(key_points).reshape(-1, 10)
        prm = None if params is None else (C.c_float * 4)(*params)
        bi, ki = C.c_int(-1), C.c_int(-1)
        _chk(self.lib.fd_face_selection(self.handle, int(img_hw[0]), int(img_hw[1]), _ptr(fb, c_f32p), None if kp is None else _ptr(kp, c_f32p),
                                        len(fb), int(bool(is_enroll)), prm, C.byref(bi), C.byref(ki)))
        return bi.value, ki.value

    def select_detections(self, frames, is_enroll=False, params=None, fetch=True):
        arr = self._frames(frames)
        prm = None if params is None else (C.c_float * 4)(*params)
        sel = np.empty((len(frames), 2), np.int32) if fetch else None
        _chk(self.lib.fd_select_detections(self.handle, arr, len(frames), int(bool(is_enroll)), prm, None if sel is None else _ptr(sel, c_i32p)))
        return sel

    def align_selected(self, frames, crops_dev, M_dev=None, ok_dev=None):
        arr = self._frames(frames)
        _chk(self.lib.fd_align_selected(self.handle, arr, len(frames), C.c_void_p(_devptr(crops_dev)), C.c_void_p(_devptr(M_dev)),
                                        C.c_void_p(_devptr(ok_dev))))

    def crops_to_tensor(self, crops_dev, F, in_hw, out_hw, mean_rgb, mul_rgb, out_dev, use_detect_count=False):
        mean, mul = _f32(mean_rgb), _f32(mul_rgb)
        _chk(self.lib.fd_crops_to_tensor(self.handle, C.c_void_p(_devptr(crops_dev)), int(F), in_hw[0], in_hw[1], out_hw[0], out_hw[1],
                                         _ptr(mean, c_f32p), _ptr(mul, c_f32p), C.c_void_p(_devptr(out_dev)), int(use_detect_count)))

    def model_preprocess(self, img, out_size, mean_rgb, mul_rgb):
        img = np.ascontiguousarray(img, np.uint8)
        mean, mul = _f32(mean_rgb), _f32(mul_rgb)
        ow, oh = out_size
        out = np.empty((3, oh, ow), np.float32)
        _chk(self.lib.fd_model_preprocess(self.handle, _ptr(img, c_u8p), img.shape[0], img.shape[1], img.strides[0], oh, ow,
                                          _ptr(mean, c_f32p), _ptr(mul, c_f32p), _ptr(out, c_f32p)))
        return out

    # ---- N4: JPEG decode (utils.rs:8-52)
    def imdecode(self, data):
        """byte_data_to_opencv / cv::imdecode(bytes, IMREAD_UNCHANGED) for a baseline 3-component JPEG -> (h, w, 3) BGR u8 (host)"""
        buf = np.frombuffer(bytes(data), np.uint8)
        h, w = C.c_int(0), C.c_int(0)
        _chk(self.lib.fd_jpeg_info(_ptr(buf, c_u8p), C.c_size_t(len(buf)), C.byref(h), C.byref(w), None))
        out = np.empty((h.value, w.value, 3), np.uint8)
        _chk(self.lib.fd_imdecode(self.handle, _ptr(buf, c_u8p), C.c_size_t(len(buf)), _ptr(out, c_u8p), w.value * 3))
        return out

    def jpeg_last_stats(self):
        out = (C.c_int64 * 4)()
        _chk(self.lib.fd_jpeg_last_stats(self.handle, out))
        return dict(h2d_bytes=int(out[0]), device_entropy_images=int(out[1]), host_entropy_images=int(out[2]),
                    selfsync_images=int(out[3] & 0xFFFFFFFF), selfsync_rounds=int(out[3] >> 32))

    def decode_jpeg_batch(self, jpegs, n_threads=0):
        """jpegs: list of bytes-like JPEG streams -> fd_frame array of device-resident BGR frames (valid until the next call)"""
        bufs = [np.frombuffer(bytes(j), np.uint8) if not isinstance(j, np.ndarray) else j for j in jpegs]
        B = len(bufs)
        ptrs = (C.c_void_p * B)(*[b.ctypes.data for b in bufs])
        lens = (C.c_size_t * B)(*[b.size for b in bufs])
        frames = (FdFrame * B)()
        _chk(self.lib.fd_decode_jpeg_batch(self.handle, ptrs, lens, B, int(n_threads), frames))
        self._jpeg_keepalive = bufs
        return frames

    def pipeline_host(self, frames_host, heads_host, cap_rows, conf_thr=None, iou_thr=None, want_tensor=False, bufs=None,
                      select=False, is_enroll=False, upload=FD_UPLOAD_FULL, select_params=None, heads_zero_copy=False, jpeg=False,
                      jpeg_threads=0):
        """frames_host: list of HxWx3 u8 arrays (host, ideally pinned); heads_host: 9 host arrays (B,C,H,W).
        select: FacePipeline::extract's flow (one selected face per image is aligned; crop b belongs to image b).
        upload: FD_UPLOAD_FULL | FD_UPLOAD_ON_DEMAND.  -> (bufs, total detections, h2d bytes, d2h bytes); bufs also
        holds "n_crops"."""
        B = len(frames_host)
        if jpeg:     # frames_host: list of 1-D u8 arrays holding JPEG streams (fd_pipeline_host_jpeg)
            jp = (C.c_void_p * B)(*[f.ctypes.data for f in frames_host])
            jl = (C.c_size_t * B)(*[f.size for f in frames_host])
        else:
            arr = (FdFrame * B)()
            for i, f in enumerate(frames_host):
                arr[i].data, arr[i].height, arr[i].width, arr[i].pitch = f.ctypes.data, f.shape[0], f.shape[1], f.strides[0]
        hp = (C.c_void_p * len(heads_host))(*[h.ctypes.data for h in heads_host])
        if bufs is None:
            bufs = dict(counts=np.empty(B, np.int32), det=np.empty((cap_rows, 5), np.float32),
                        lmk=np.empty((cap_rows, 10), np.float32),
                        crops=np.empty((cap_rows, self.cfg.crop_h, self.cfg.crop_w, 3), np.uint8),
                        det_scale=np.empty(B, np.float32), align_mode=np.zeros(cap_rows, np.uint8),
                        sel=np.full((B, 2), -1, np.int32),
                        tensor=np.empty((B, 3, self.cfg.image_h, self.cfg.image_w), np.float32) if want_tensor else None)
        out = FdHostBatchOut()
        out.counts, out.det, out.landmarks = _ptr(bufs["counts"], c_i32p), _ptr(bufs["det"], c_f32p), _ptr(bufs["lmk"], c_f32p)
        out.crops, out.det_scale = _ptr(bufs["crops"], c_u8p), _ptr(bufs["det_scale"], c_f32p)
        out.tensor = _ptr(bufs["tensor"], c_f32p) if bufs.get("tensor") is not None else None
        out.align_mode = _ptr(bufs["align_mode"], c_u8p) if bufs.get("align_mode") is not None else None
        out.sel = _ptr(bufs["sel"], c_i32p) if bufs.get("sel") is not None else None
        out.cap_rows = cap_rows
        opts = FdPipelineOpts()
        _chk(self.lib.fd_pipeline_opts_default(C.byref(opts)))
        opts.select, opts.is_enroll, opts.upload = int(bool(select)), int(bool(is_enroll)), int(upload)
        opts.heads_zero_copy = int(bool(heads_zero_copy))
        if select_params is not None:
            opts.select_params = FdSelectParams(*select_params)
        ct = C.c_float(self.cfg.conf_thr if conf_thr is None else conf_thr)
        it = C.c_float(self.cfg.iou_thr if iou_thr is None else iou_thr)
        if jpeg:
            _chk(self.lib.fd_pipeline_host_jpeg(self.handle, jp, jl, B, int(jpeg_threads), hp, len(heads_host), ct, it, C.byref(opts), C.byref(out)))
        else:
            _chk(self.lib.fd_pipeline_host(self.handle, arr, B, hp, len(heads_host), ct, it, C.byref(opts), C.byref(out)))
        bufs["n_crops"] = out.n_crops
        return bufs, out.total, out.h2d_bytes, out.d2h_bytes
