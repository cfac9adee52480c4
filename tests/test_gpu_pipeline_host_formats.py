"""fd_pipeline_host_yuv420 / _yuv422 / _rgb: the end-to-end host-memory call on 4:2:0, packed 4:2:2 and RGB-family frames.

Every output must equal, byte for byte, what fd_pipeline_host gives on cv2.cvtColor(COLOR_YUV2BGR_<layout> / RGB2BGR /
RGBA2BGR / BGRA2BGR / GRAY2BGR) of the frames with the same options (tests/yuv420_ref.py, yuv422_ref.py and rgb_ref.py restate
the conversions and are pinned against cv2), for both upload modes and both flows; the BGR results are checked against the
oracle.  The host frames live in pitched buffers whose padding, leading bytes and RGBA / BGRA alpha bytes are noise; the first
frame of a batch has tight rows (one contiguous copy a plane), the others padded ones (2-D copies).  h2d_bytes must follow the
layout's bytes: whole planes under FD_UPLOAD_FULL, only the rows the resize reads under FD_UPLOAD_ON_DEMAND."""
import numpy as np
import pytest

from rgb_ref import BGRA, BPP, GRAY8, RGB24, RGBA, bgr_to_rgb, rgb_to_bgr
from rs_face_detection_b200.utils import synth
from yuv420_ref import I420, NV12, NV21, PLANAR, YV12, bgr_to_yuv420, yuv420_to_bgr
from yuv422_ref import UYVY, YUY2, YVYU, bgr_to_yuv422, yuv422_to_bgr

pytestmark = pytest.mark.gpu
CONF, IOU = 0.7, 0.4
LAYOUTS = ([("yuv420", l) for l in (NV12, NV21, I420, YV12)] + [("yuv422", l) for l in (YUY2, UYVY, YVYU)]
           + [("rgb", l) for l in (RGB24, RGBA, BGRA, GRAY8)])
IDS = ["%s-%d" % k for k in LAYOUTS]
# 1080p and 4K (exact 3x / 6x decimation: strided row copies), 720p (2x with two taps: whole frame), a small upscaled frame
SIZES = [(1080, 1920), (2160, 3840), (720, 1280), (62, 86)]


def _frame_bytes(kind, layout, H, W):
    if kind == "yuv420":
        return H * W * 3 // 2
    return H * W * (2 if kind == "yuv422" else BPP[layout])


class HostFrames:
    """B host frames in (kind, layout), in noisy pitched numpy buffers, and the BGR frames cvtColor makes of them"""

    def __init__(self, kind, layout, sizes, seed):
        rng = np.random.default_rng(seed)
        self.kind, self.layout, self.sizes = kind, layout, sizes
        self.bufs, self.desc, self.bgr = [], [], []
        for i, (H, W) in enumerate(sizes):
            src = synth.make_frame(H, W, seed + i)
            pad = 0 if i == 0 else 16 + 3 * i
            if kind == "yuv420":
                y, chroma = bgr_to_yuv420(src, layout)
                yb, y_off, py = self._place(rng, y, pad)
                cb, c_off, pc = self._place(rng, chroma, pad)
                self.desc.append((yb.ctypes.data + y_off, cb.ctypes.data + c_off, H, W, py, pc))
                self.bgr.append(yuv420_to_bgr(yb[y_off:y_off + H * py].reshape(H, py), cb[c_off:], layout, H, W, pc))
                self.bufs += [yb, cb]
                continue
            rows = bgr_to_yuv422(src, layout) if kind == "yuv422" else bgr_to_rgb(src, layout, alpha=rng.integers(0, 256, (H, W), np.uint8))
            b, off, p = self._place(rng, rows, pad)
            self.desc.append((b.ctypes.data + off, H, W, p))
            self.bgr.append((yuv422_to_bgr if kind == "yuv422" else rgb_to_bgr)(b[off:], layout, H, W, p))
            self.bufs.append(b)

    @staticmethod
    def _place(rng, rows, pad):
        """rows (R, n) -> (noise buffer, offset of the first row, pitch)"""
        R, n = rows.shape
        off = 0 if pad == 0 else 1 + pad % 5
        pitch = n + pad
        buf = rng.integers(0, 256, off + R * pitch + 64, np.uint8)
        buf[off:off + R * pitch].reshape(R, pitch)[:, :n] = rows
        return buf, off, pitch

    def bytes(self):
        return sum(_frame_bytes(self.kind, self.layout, H, W) for H, W in self.sizes)

    def run(self, ctx, heads, cap_rows, **kw):
        call = getattr(ctx, "pipeline_host_" + self.kind)
        return call(self.desc, self.layout, heads, cap_rows, conf_thr=CONF, iou_thr=IOU, **kw)


def _assert_same(got, ref, what):
    bufs, total, _, _ = got
    rbufs, rtotal, _, _ = ref
    assert total == rtotal and bufs["n_crops"] == rbufs["n_crops"], what
    n = bufs["n_crops"]
    for k in ("counts", "det_scale", "sel"):
        np.testing.assert_array_equal(bufs[k], rbufs[k], err_msg="%s %s" % (what, k))
    if rbufs.get("tensor") is not None:
        np.testing.assert_array_equal(bufs["tensor"], rbufs["tensor"], err_msg="%s tensor" % what)
    for k in ("det", "lmk"):
        np.testing.assert_array_equal(bufs[k][:total], rbufs[k][:total], err_msg="%s %s" % (what, k))
    for k in ("crops", "align_mode"):
        np.testing.assert_array_equal(bufs[k][:n], rbufs[k][:n], err_msg="%s %s" % (what, k))


def _heads(B, seed, n_faces=8):
    return synth.make_heads(B, seed=seed, n_faces=n_faces, content_hw=(360, 640))[0]


@pytest.mark.parametrize("kind,layout", LAYOUTS, ids=IDS)
def test_outputs_equal_bgr_on_converted_frames(ctx, oracle, kind, layout):
    """every layout x {FULL, ON_DEMAND} x {all faces, select, select + is_enroll} == fd_pipeline_host on the cvtColor frames.
    Each ON_DEMAND call follows a call on different frames of the same geometry, so a byte the upload misses holds wrong data.
    Under FULL, h2d_bytes differs from BGR's by exactly the difference of the frame bytes."""
    from test_gpu_pipeline import _check_all_faces
    B = len(SIZES)
    fr = HostFrames(kind, layout, SIZES, 500 + 10 * layout)
    decoy = HostFrames(kind, layout, SIZES, 900 + 10 * layout)
    heads = _heads(B, 5000 + layout)
    cap = B * 64
    for upload in (0, 1):
        for select, is_enroll in ((False, False), (True, False), (True, True)):
            kw = dict(upload=upload, select=select, is_enroll=is_enroll, want_tensor=True)
            what = "%s layout %d upload %d select %d enroll %d" % (kind, layout, upload, select, is_enroll)
            if upload:
                decoy.run(ctx, heads, cap, **kw)
            got = fr.run(ctx, heads, cap, **kw)
            ref = ctx.pipeline_host(fr.bgr, heads, cap, conf_thr=CONF, iou_thr=IOU, **kw)
            assert ref[1] > B * 2, what
            _assert_same(got, ref, what)
            if not upload:
                assert got[2] - ref[2] == fr.bytes() - sum(3 * H * W for H, W in SIZES), what
            if not upload and not select:
                _check_all_faces(oracle, fr.bgr, heads, ref[0], ref[1], CONF, IOU)


# preprocess row bytes per frame under FD_UPLOAD_ON_DEMAND (1080p: rows 3y+1, 4:2:0 chroma rows 3m and 3m+2; 4K: rows 6y+2
# and 6y+3, chroma rows 3y+1)
ROW_BYTES = {
    (1080, 1920): {"bgr": 2073600, "yuv420": 1382400, "yuv422": 1382400, 3: 2073600, 4: 2764800, 1: 691200},
    (2160, 3840): {"bgr": 8294400, "yuv420": 4147200, "yuv422": 5529600, 3: 8294400, 4: 11059200, 1: 2764800},
}


@pytest.mark.parametrize("kind,layout", LAYOUTS, ids=IDS)
def test_on_demand_sends_the_rows_the_resize_reads(ctx, kind, layout):
    """no face (every score below the threshold): ON_DEMAND sends per plane only the rows the preprocess reads at 1080p and
    4K, and whole frames at the other scales; the outputs still equal BGR's"""
    B = len(SIZES)
    fr = HostFrames(kind, layout, SIZES, 700 + layout)
    heads = _heads(B, 5100)
    for h in heads[0::3]:
        h[:, 2:] = 0.0
    got = fr.run(ctx, heads, 64, upload=1, want_tensor=True)
    ref = ctx.pipeline_host(fr.bgr, heads, 64, conf_thr=CONF, iou_thr=IOU, upload=1, want_tensor=True)
    assert ref[1] == 0
    _assert_same(got, ref, "no faces")
    want = 0
    for H, W in SIZES:
        if (H, W) in ROW_BYTES:
            rb = ROW_BYTES[(H, W)]
            want += rb[kind if kind != "rgb" else BPP[layout]] - rb["bgr"]
        else:
            want += _frame_bytes(kind, layout, H, W) - 3 * H * W
    assert got[2] - ref[2] == want


@pytest.mark.parametrize("kind,layout", [("yuv420", NV12), ("yuv420", I420), ("yuv422", YUY2), ("rgb", RGBA), ("rgb", GRAY8)])
def test_select_flow_on_demand_sends_less(ctx, kind, layout):
    """FacePipeline::extract's flow at 1080p: the preprocess rows and one face rectangle per image, under 0.75 of FULL.  The
    bbox / landmark heads are read in place from pinned memory (heads_zero_copy), so the frames make most of the bytes."""
    from rs_face_detection_b200.ffi import pinned_like
    B = 5
    fr = HostFrames(kind, layout, [(1080, 1920)] * B, 800 + layout)
    pinned = [pinned_like(h) for h in _heads(B, 5200, n_faces=5)]
    heads = [p.array for p in pinned]
    full = fr.run(ctx, heads, B * 64, select=True, heads_zero_copy=True)
    dem = fr.run(ctx, heads, B * 64, select=True, upload=1, heads_zero_copy=True)
    _assert_same(dem, full, "select")
    assert dem[2] < 0.75 * full[2]
    for p in pinned:
        p.free()


def test_deferred_image_gives_the_bgr_crops(ctx):
    """an image with K > 4096 candidates is completed at the fetch; the align enqueued before it replays in the layout"""
    from test_gpu_detect_limits import _blank, _groups, _plant
    rng = np.random.default_rng(90)
    heads = _blank(2, 0.1)
    grp = _groups(rng, 1025, 4)
    grp[-1] = grp[-1][:4097 - 4 * 1024]
    assert _plant(heads, 0, rng, grp, "distinct") == 4097
    _plant(heads, 1, rng, _groups(rng, 20, 1, rows=44), "distinct")
    for kind, layout in [("yuv420", I420), ("yuv422", UYVY), ("rgb", BGRA), ("rgb", GRAY8)]:
        fr = HostFrames(kind, layout, [(1080, 1920)] * 2, 95 + layout)
        for upload in (0, 1):
            got = fr.run(ctx, heads, 2048, upload=upload)
            ref = ctx.pipeline_host(fr.bgr, heads, 2048, conf_thr=CONF, iou_thr=IOU, upload=upload)
            assert ref[0]["counts"][0] == 1025
            _assert_same(got, ref, "%s %d deferred" % (kind, layout))


def test_bad_descriptors_are_rejected(ctx):
    """odd 4:2:0 size, pitch below the minimum, null plane, unknown layout: FD_ERR_INVALID, and the ctx works afterwards"""
    from rs_face_detection_b200.ffi import FD_ERR_INVALID, FdError
    heads = _heads(1, 5300)
    y = np.zeros(1082 * 1920, np.uint8)
    c = np.zeros(541 * 1920, np.uint8)
    px = np.zeros(1080 * 1920 * 4, np.uint8)
    Y, C_ = y.ctypes.data, c.ctypes.data
    bad = [
        ("yuv420", NV12, (Y, C_, 1081, 1920, 1920, 1920)),      # odd height
        ("yuv420", NV12, (Y, C_, 1080, 1919, 1920, 1920)),      # odd width
        ("yuv420", NV12, (Y, C_, 1080, 1920, 1918, 1920)),      # pitch_y < W
        ("yuv420", I420, (Y, C_, 1080, 1920, 1920, 958)),       # pitch_uv < W/2
        ("yuv420", NV21, (Y, 0, 1080, 1920, 1920, 1920)),       # null chroma
        ("yuv420", 4, (Y, C_, 1080, 1920, 1920, 1920)),         # unknown layout
        ("yuv422", YUY2, (px.ctypes.data, 1080, 1920, 3838)),  # pitch < 2W
        ("yuv422", YVYU, (0, 1080, 1920, 3840)),               # null data
        ("yuv422", 3, (px.ctypes.data, 1080, 1920, 3840)),
        ("rgb", RGBA, (px.ctypes.data, 1080, 1920, 7679)),     # pitch < 4W
        ("rgb", GRAY8, (0, 1080, 1920, 1920)),
        ("rgb", 4, (px.ctypes.data, 1080, 1920, 7680)),
    ]
    for kind, layout, d in bad:
        with pytest.raises(FdError) as e:
            getattr(ctx, "pipeline_host_" + kind)([d], layout, heads, 64, conf_thr=CONF, iou_thr=IOU)
        assert e.value.code == FD_ERR_INVALID, (kind, layout, d)
    fr = HostFrames("yuv420", NV12, [(1080, 1920)], 5301)
    _assert_same(fr.run(ctx, heads, 64), ctx.pipeline_host(fr.bgr, heads, 64, conf_thr=CONF, iou_thr=IOU), "after errors")


def test_bgr_and_jpeg_calls_unchanged_after_a_layout_call():
    """a layout call, then fd_pipeline_host and fd_pipeline_host_jpeg on one ctx: the same results as before it"""
    cv2 = pytest.importorskip("cv2")
    from rs_face_detection_b200 import Context
    B = 3
    frames = [synth.make_frame(1080, 1920, 5400 + i) for i in range(B)]
    streams = [np.asarray(cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, 90])[1], np.uint8).ravel() for f in frames]
    heads = _heads(B, 5401)
    c = Context(0)
    try:
        def both():
            return [c.pipeline_host(frames, heads, B * 64, conf_thr=CONF, iou_thr=IOU, want_tensor=True, upload=u) for u in (0, 1)] + \
                   [c.pipeline_host(streams, heads, B * 64, conf_thr=CONF, iou_thr=IOU, want_tensor=True, jpeg=True)]
        before = both()
        for kind, layout in [("yuv420", YV12), ("yuv422", YUY2), ("rgb", RGB24)]:
            HostFrames(kind, layout, [(1080, 1920)] * B, 5402).run(c, heads, B * 64, upload=1)
            after = both()
            for a, b in zip(after, before):
                _assert_same(a, b, "after %s %d" % (kind, layout))
                assert a[2] == b[2] and a[3] == b[3]
    finally:
        c.close()
