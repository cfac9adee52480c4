"""End-to-end: preprocess -> decode -> NMS -> align, device-resident and through the host-buffer call, vs the oracle's
whole-frame CPU path (BASELINE config 2 geometry at a reduced batch)."""
import numpy as np
import pytest

from detect_ref import assert_rows_exact, decode_rows
from rs_face_detection_b200.utils import synth

pytestmark = pytest.mark.gpu


def _check_rows(cfg, heads_b, det_scale, det, lmk, edet, elmk, what=""):
    """rows bit for bit (tests/detect_ref.py): landmarks and scores equal the oracle's, boxes a correctly rounded exp's"""
    assert_rows_exact(det, lmk, (edet, elmk), decode_rows(heads_b, cfg, det_scale, cfg.conf_thr, cfg.iou_thr), what)


def _oracle_frame(oracle, cfg, frame, heads_b):
    return oracle.pipeline_frame(cfg, frame, heads_b)


def test_pipeline_host_matches_oracle(ctx, oracle):
    B = 4
    frames = [synth.make_frame(1080, 1920, 2000 + i) for i in range(B - 1)] + [synth.make_frame(2160, 3840, 2099)]
    heads, _ = synth.make_heads(B, seed=3000, n_faces=20, content_hw=(360, 640))
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.4)
    bufs, total, h2d, d2h = ctx.pipeline_host(frames, heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4, want_tensor=True)
    assert total == bufs["counts"].sum() and total > B * 10
    assert h2d >= sum(f.nbytes for f in frames) and d2h > total * 112 * 112 * 3
    off = 0
    for b in range(B):
        tensor, det, lmk, crops = _oracle_frame(oracle, cfg, frames[b], [h[b] for h in heads])
        n = bufs["counts"][b]
        assert n == len(det)
        np.testing.assert_array_equal(bufs["tensor"][b], tensor[0])
        _check_rows(cfg, [h[b] for h in heads], bufs["det_scale"][b], bufs["det"][off:off + n], bufs["lmk"][off:off + n], det, lmk, "image %d" % b)
        # crops: the landmarks are the oracle's, bit for bit, so every crop is the oracle's own end-to-end crop.  Only a
        # bbox-fallback crop (mode 2) reads the box, which may differ from the oracle's where its libm expf misrounds.
        for i in range(n):
            same_box = bufs["det"][off + i].tobytes() == det[i].tobytes()
            if same_box or bufs["align_mode"][off + i] != 2:
                np.testing.assert_array_equal(bufs["crops"][off + i], crops[i], err_msg="image %d face %d" % (b, i))
            crop, _ = oracle.align_face(frames[b], bufs["lmk"][off + i])     # and the oracle aligned with the GPU's own rows
            np.testing.assert_array_equal(bufs["crops"][off + i], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
        off += n


def _check_all_faces(oracle, frames, heads, bufs, total, conf, iou):
    cfg = oracle.make_det_cfg(conf_thr=conf, iou_thr=iou)
    off = 0
    for b in range(len(frames)):
        tensor, det, lmk, _ = _oracle_frame(oracle, cfg, frames[b], [h[b] for h in heads])
        n = bufs["counts"][b]
        assert n == len(det)
        _check_rows(cfg, [h[b] for h in heads], bufs["det_scale"][b], bufs["det"][off:off + n], bufs["lmk"][off:off + n], det, lmk, "image %d" % b)
        for i in range(n):
            crop, _, mode = oracle.align_face(frames[b], bufs["lmk"][off + i], bbox=bufs["det"][off + i], with_mode=True)
            assert bufs["align_mode"][off + i] == mode
            np.testing.assert_array_equal(bufs["crops"][off + i], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
        off += n
    assert off == total == bufs["n_crops"]


@pytest.mark.parametrize("shapes", [[(1080, 1920)] * 3 + [(2160, 3840)], [(720, 1280), (1080, 1920), (600, 800), (1081, 1923)]])
def test_pipeline_host_on_demand_upload(ctx, oracle, shapes):
    """FD_UPLOAD_ON_DEMAND (preprocess rows first, then only the pixels the warps read) gives the same bytes out as whole-frame
    upload — over exact 3x / 6x decimations (strided row copies), a non-integer scale and an odd pitch (whole-frame path)."""
    from rs_face_detection_b200.ffi import FD_UPLOAD_ON_DEMAND
    B = len(shapes)
    frames = [synth.make_frame(h, w, 2300 + i) for i, (h, w) in enumerate(shapes)]
    heads, _ = synth.make_heads(B, seed=3100, n_faces=6, content_hw=(360, 640))
    full, total_f, h2d_f, _ = ctx.pipeline_host(frames, heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4, want_tensor=True)
    dem, total_d, h2d_d, _ = ctx.pipeline_host(frames, heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4, want_tensor=True,
                                               upload=FD_UPLOAD_ON_DEMAND)
    assert total_f == total_d > 0
    for k in ("counts", "tensor", "det_scale"):
        np.testing.assert_array_equal(full[k], dem[k])
    for k in ("det", "lmk"):
        np.testing.assert_array_equal(full[k][:total_f], dem[k][:total_d])
    np.testing.assert_array_equal(full["crops"][:total_f], dem["crops"][:total_d])
    np.testing.assert_array_equal(full["align_mode"][:total_f], dem["align_mode"][:total_d])
    _check_all_faces(oracle, frames, heads, dem, total_d, 0.7, 0.4)
    assert h2d_d <= h2d_f * 1.02      # never (noticeably) more than whole frames


@pytest.mark.parametrize("upload", [0, 1])
@pytest.mark.parametrize("is_enroll", [False, True])
def test_pipeline_host_select_flow(ctx, oracle, upload, is_enroll):
    """FacePipeline::extract's flow (face_pipeline/pipeline.rs:196-232): detect -> FaceSelection::call -> align the ONE selected
    face.  Crop b belongs to image b; an image without a selection gets a zero crop with mode 0 (the reference returns Err)."""
    B = 5
    frames = [synth.make_frame(1080, 1920, 2400 + i) for i in range(B)]
    heads, _ = synth.make_heads(B, seed=3200, n_faces=5, content_hw=(360, 640))
    for h in heads[0::3]:
        h[B - 1, 2:] = 0.0            # last image: no foreground score passes -> no detection -> nothing selected
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.4)
    bufs, total, h2d, d2h = ctx.pipeline_host(frames, heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4, select=True, is_enroll=is_enroll,
                                              upload=upload)
    assert bufs["n_crops"] == B and bufs["counts"][B - 1] == 0
    off = 0
    picked = 0
    for b in range(B):
        n = bufs["counts"][b]
        det, lmk = bufs["det"][off:off + n], bufs["lmk"][off:off + n].reshape(-1, 5, 2)
        bi, ki = oracle.face_selection((1080, 1920), det, lmk, is_enroll) if n else (-1, -1)
        want = (off + bi if bi >= 0 else -1, off + ki if ki >= 0 else -1)
        assert tuple(bufs["sel"][b]) == want
        if bi >= 0 and ki >= 0:
            crop, _, mode = oracle.align_face(frames[b], lmk[ki], bbox=det[bi], with_mode=True)
            picked += 1
        else:
            crop, mode = None, 0
        assert bufs["align_mode"][b] == mode
        np.testing.assert_array_equal(bufs["crops"][b], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
        off += n
    assert picked >= B - 2
    if upload:   # preprocess rows + one face rectangle per image + heads, against whole frames + heads
        _, _, h2d_full, _ = ctx.pipeline_host(frames, heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4, select=True, is_enroll=is_enroll)
        assert h2d < 0.75 * h2d_full


def test_pipeline_host_zero_copy_heads(ctx, oracle):
    """heads_zero_copy: the bbox / landmark tensors stay in pinned host memory and the detect kernel reads the passing anchors'
    values from there — same outputs, fewer bytes over PCIe; pageable buffers silently take the copy."""
    from rs_face_detection_b200.ffi import pinned_like
    B = 4
    frames = [synth.make_frame(1080, 1920, 2500 + i) for i in range(B)]
    heads, _ = synth.make_heads(B, seed=3300, n_faces=12, content_hw=(360, 640))
    ref, total, h2d_copy, _ = ctx.pipeline_host(frames, heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4)
    pinned = [pinned_like(h) for h in heads]
    for mode_heads in ([p.array for p in pinned], heads):
        got, total2, h2d, _ = ctx.pipeline_host(frames, mode_heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4, heads_zero_copy=True)
        assert total2 == total > 0
        np.testing.assert_array_equal(got["counts"], ref["counts"])
        np.testing.assert_array_equal(got["det"][:total], ref["det"][:total])
        np.testing.assert_array_equal(got["lmk"][:total], ref["lmk"][:total])
        np.testing.assert_array_equal(got["crops"][:total], ref["crops"][:total])
        if mode_heads is not heads:
            assert h2d < h2d_copy - 0.8 * sum(h.nbytes for i, h in enumerate(heads) if i % 3)
        else:
            assert h2d == h2d_copy
    _check_all_faces(oracle, frames, heads, got, total, 0.7, 0.4)
    for p in pinned:
        p.free()


def test_device_resident_sequence(ctx, oracle):
    """The benchmarked call sequence: preprocess_batch -> detect_batch -> align_detections, inputs resident in HBM."""
    B = 3
    frames = [synth.make_frame(1080, 1920, 10 + i) for i in range(B)]
    heads, _ = synth.make_heads(B, seed=42, n_faces=15, content_hw=(360, 640))
    fdev = [ctx.to_device(f) for f in frames]
    hdev = [ctx.to_device(h) for h in heads]
    fl = [(d.ptr, 1080, 1920, 5760) for d in fdev]
    tensor = ctx.alloc(B * 3 * 640 * 640 * 4)
    cap = B * 64
    crops = ctx.alloc(cap * 112 * 112 * 3)
    for _ in range(2):   # twice: workspace reuse
        ds = ctx.preprocess_batch(fl, tensor)
        ctx.detect_batch(hdev, B, ds, 0.7, 0.4)
        ctx.align_detections(fl, crops, cap)
        counts, det, lmk = ctx.detect_fetch(B)
    got = crops.download((cap, 112, 112, 3), np.uint8)
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.4)
    off = 0
    for b in range(B):
        _, edet, elmk, _ = _oracle_frame(oracle, cfg, frames[b], [h[b] for h in heads])
        assert counts[b] == len(edet)
        _check_rows(cfg, [h[b] for h in heads], ds[b], det[off:off + counts[b]], lmk[off:off + counts[b]], edet, elmk, "image %d" % b)
        for i in range(counts[b]):
            crop, _ = oracle.align_face(frames[b], lmk[off + i])
            np.testing.assert_array_equal(got[off + i], crop)
        off += counts[b]
    assert ctx.launch_count() > 0


def test_retinaface_detection_class(ctx, oracle):
    """Mirror of RetinaFaceDetection::call with the CNN stubbed by synthetic head tensors."""
    from rs_face_detection_b200.pipeline import RetinaFaceDetection
    heads, _ = synth.make_heads(1, seed=8, n_faces=10, content_hw=(360, 640))
    det = RetinaFaceDetection(infer=lambda t: [h[0] for h in heads], confidence_threshold=0.7, iou_threshold=0.45, ctx=ctx)
    img = synth.make_frame(1080, 1920, 1)
    d, l = det.call(img)
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.45)
    ed, el, _ = oracle.detect_post(cfg, [h[0] for h in heads], np.float32(360 / 1080))
    _check_rows(cfg, [h[0] for h in heads], np.float32(360 / 1080), d, l, ed, el)
