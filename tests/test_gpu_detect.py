"""Decode + sort + NMS + rescale parity (face_detection.rs:319-493) through the C ABI vs the oracle."""
import numpy as np
import pytest

from detect_ref import check_image
from rs_face_detection_b200.utils import synth

pytestmark = pytest.mark.gpu


def _check_image(oracle, cfg, heads_b, det_scale, det, lmk):
    """GPU rows vs the oracle, bit for bit: scores and landmarks equal the oracle's, boxes equal a restatement with a
    correctly rounded exp and differ from the oracle's only where its libm expf misrounds (tests/detect_ref.py)."""
    return check_image(oracle, cfg, heads_b, det_scale, det, lmk)


@pytest.mark.parametrize("conf,iou", [(0.7, 0.4), (0.7, 0.45), (0.02, 0.4)])
def test_c1_single_image(ctx, oracle, conf, iou):
    """BASELINE config 1: 640x640 single image, synthetic heads for strides 32/16/8 (16,800 anchors)."""
    heads, _ = synth.make_heads(1, seed=1234, n_faces=20)
    hb = [h[0] for h in heads]
    cfg = oracle.make_det_cfg(conf_thr=conf, iou_thr=iou)
    det, lmk = ctx.detect(hb, 1.0, conf, iou)
    K = _check_image(oracle, cfg, hb, 1.0, det, lmk)
    assert K > (4096 if conf < 0.1 else 20)   # conf 0.02 exceeds the single-CTA capacity -> big path


def test_decode_candidates_and_exact_keep(ctx, oracle):
    """Stage-level: the keep list of the oracle's own candidates, and the rows bit for bit."""
    heads, _ = synth.make_heads(3, seed=99, n_faces=25)
    devs = [ctx.to_device(h) for h in heads]
    ctx.detect_batch(devs, 3, np.ones(3, np.float32), 0.5, 0.4)
    counts, det, lmk = ctx.detect_fetch(3)
    cfg = oracle.make_det_cfg(conf_thr=0.5, iou_thr=0.4)
    off = 0
    for b in range(3):
        hb = [h[b] for h in heads]
        box, score, clmk, idx = oracle.decode_candidates(cfg, hb)
        d = det[off:off + counts[b]]
        # every GPU detection is one of the oracle's candidates, in the oracle's keep order
        order = oracle.argsort_descending(score)
        pre = np.concatenate([box[order], score[order, None]], 1)
        keep = oracle.nms(pre, 0.4)
        np.testing.assert_array_equal(d[:, 4], pre[keep, 4])
        _check_image(oracle, cfg, hb, 1.0, d, lmk[off:off + counts[b]])
        off += counts[b]
    assert off == len(det)


def test_batch_with_ragged_and_empty_images(ctx, oracle):
    heads, _ = synth.make_heads(6, seed=7, n_faces=12)
    for h in heads[0::3]:
        h[2, 2:] = 0.0           # image 2: no foreground at all -> (0,5), (0,5,2)   (face_detection.rs:413-419)
        h[2, :2] = 1.0
    scales = np.array([1.0, 0.5, 0.33333334, 0.25, 0.16666667, 1.5], np.float32)
    devs = [ctx.to_device(h) for h in heads]
    ctx.detect_batch(devs, 6, scales, 0.7, 0.45)
    counts, det, lmk = ctx.detect_fetch(6)
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.45)
    assert counts[2] == 0
    off = 0
    for b in range(6):
        _check_image(oracle, cfg, [h[b] for h in heads], scales[b], det[off:off + counts[b]], lmk[off:off + counts[b]])
        off += counts[b]
    v = ctx.detect_view()
    assert v.det_dev and v.landmarks_dev and v.offsets_dev


def test_all_anchors_pass_big_path_in_batch(ctx, oracle):
    """conf 0.02 with every anchor above threshold: K = 16800 per image -> the per-image big path (radix + peel)."""
    heads = synth.make_dense_heads(2, seed=3)
    devs = [ctx.to_device(h) for h in heads]
    ctx.detect_batch(devs, 2, np.ones(2, np.float32), 0.02, 0.4)
    counts, det, lmk = ctx.detect_fetch(2)
    cfg = oracle.make_det_cfg(conf_thr=0.02, iou_thr=0.4)
    off = 0
    for b in range(2):
        K = _check_image(oracle, cfg, [h[b] for h in heads], 1.0, det[off:off + counts[b]], lmk[off:off + counts[b]])
        assert K == 16800
        off += counts[b]


@pytest.mark.parametrize("conf", [0.7, 0.2, 0.05])
def test_mixed_candidate_counts_in_one_batch(oracle, conf):
    """A batch mixing images with few candidates (K <= 1024: resolved inside the fused kernel) and crowded ones.  On a fresh
    ctx the fused kernel defers the crowded images (fd_detect_fetch completes them: general single-CTA NMS for K <= 4096,
    radix + spatial path beyond); once the ctx has met one, later launches keep K <= 4096 on the device.  Same rows, in
    frame order, both ways."""
    from rs_face_detection_b200 import Context
    crowded, _ = synth.make_heads(2, seed=21, n_faces=60)      # K ~ 1150 / 2250 / 5000 at conf 0.7 / 0.2 / 0.05
    sparse, _ = synth.make_heads(2, seed=22, n_faces=5)
    heads = [np.ascontiguousarray(np.stack([c[0], s_[0], c[1], s_[1]])) for c, s_ in zip(crowded, sparse)]
    scales = np.array([1.0, 0.5, 0.33333334, 2.0], np.float32)
    c = Context(0)
    try:
        devs = [c.to_device(h) for h in heads]
        c.detect_batch(devs, 4, scales, conf, 0.4)
        counts, det, lmk = c.detect_fetch(4)               # first meeting: deferred images completed here
        cfg = oracle.make_det_cfg(conf_thr=conf, iou_thr=0.4)
        off, Ks = 0, []
        for b in range(4):
            Ks.append(_check_image(oracle, cfg, [h[b] for h in heads], scales[b], det[off:off + counts[b]], lmk[off:off + counts[b]]))
            off += counts[b]
        assert off == len(det)
        assert max(Ks) > 1024 and (conf < 0.7 or min(Ks) <= 1024)
        # second call on the same ctx: images with K <= 4096 never leave the device, K > 4096 is still completed at fetch
        crops = c.alloc(len(det) * 112 * 112 * 3 + 16)
        frames = [synth.make_frame(360, 640, 7 + i) for i in range(4)]
        fdev = [c.to_device(f) for f in frames]
        fl = [(d.ptr, 360, 640, 1920) for d in fdev]
        c.detect_batch(devs, 4, scales, conf, 0.4)
        c.align_detections(fl, crops, len(det))           # consumes the device-side results before any fetch
        counts2, det2, lmk2 = c.detect_fetch(4)
        np.testing.assert_array_equal(counts, counts2)
        np.testing.assert_array_equal(det, det2)
        np.testing.assert_array_equal(lmk, lmk2)
        got = crops.download((len(det), 112, 112, 3), np.uint8)
        off = 0
        for b in range(4):
            for i in range(off, off + min(counts[b], 3)):   # a few crops per image against the oracle
                crop, _ = oracle.align_face(frames[b], lmk[i])
                if crop is not None:
                    np.testing.assert_array_equal(got[i], crop)
            off += counts[b]
    finally:
        c.close()


def test_score_ties_follow_concat_order(ctx, oracle):
    """Equal scores across strides: the stable order is stride32 | stride16 | stride8, then (h,w,a) (face_detection.rs:410)."""
    heads, _ = synth.make_heads(1, seed=5, n_faces=0, bg=False)
    rng = np.random.default_rng(1)
    for s in range(3):
        n = heads[3 * s].shape[-1]
        pick = rng.integers(0, n, (12, 2))
        for (hh, ww) in pick:
            a = int(rng.integers(0, 2))
            heads[3 * s][0, 2 + a, hh, ww] = 0.875
            heads[3 * s][0, a, hh, ww] = 0.125
    hb = [h[0] for h in heads]
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.45)
    det, lmk = ctx.detect(hb, 1.0, 0.7, 0.45)
    edet, elmk, K = oracle.detect_post(cfg, hb, 1.0)
    assert K >= 30
    _check_image(oracle, cfg, hb, 1.0, det, lmk)                   # same rows in the same order


def test_nan_score_is_dropped_like_the_reference(ctx, oracle):
    """face_detection.rs:375 keeps `s >= confidence_threshold`; NaN fails the comparison, so a NaN foreground score is
    dropped before argsort_descending could ever see it (no panic, no error) — same rows as the oracle."""
    heads, _ = synth.make_heads(3, seed=5, n_faces=4)
    heads[3][0, 2, 3, 3] = np.nan          # fg channel of stride 16, image 0
    heads[0][1, 3, 7, 2] = np.nan          # fg channel of stride 32, image 1
    heads[6][2, 2, 40, 41] = -np.nan
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.45)
    for b in range(3):
        hb = [h[b] for h in heads]
        det, lmk = ctx.detect(hb, 1.0, 0.7, 0.45)
        edet, elmk, _ = oracle.detect_post(cfg, hb, 1.0)
        assert len(det) == len(edet) > 0
        _check_image(oracle, cfg, hb, 1.0, det, lmk)


def test_detect_from_raw_output_contents(ctx, oracle):
    """SURVEY 8(f) N2: Triton raw_output_contents (little-endian f32 bytes at arbitrary host alignment) straight into the
    decode kernel; same results as the f32 path, the reference's shape check reproduced (face_detection.rs:286-312)."""
    from rs_face_detection_b200 import FdError
    B = 3
    heads, _ = synth.make_heads(B, seed=31, n_faces=10)
    ds = np.array([1.0, 0.5, 0.25], np.float32)
    raw, shapes = [], []
    for i, h in enumerate(heads):
        buf = np.empty(h.nbytes + 7, np.uint8)
        view = buf[1 + (i % 3):1 + (i % 3) + h.nbytes]          # deliberately unaligned
        view[:] = np.frombuffer(h.astype("<f4").tobytes(), np.uint8)
        raw.append(view)
        shapes.append(h.shape)
    ctx.detect_batch_raw(raw, shapes, ds, 0.7, 0.45)
    counts, det, lmk = ctx.detect_fetch(B)
    devs = [ctx.to_device(h) for h in heads]
    ctx.detect_batch(devs, B, ds, 0.7, 0.45)
    counts2, det2, lmk2 = ctx.detect_fetch(B)
    np.testing.assert_array_equal(counts, counts2)
    np.testing.assert_array_equal(det, det2)
    np.testing.assert_array_equal(lmk, lmk2)
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.45)
    off = 0
    for b in range(B):
        _check_image(oracle, cfg, [h[b] for h in heads], ds[b], det[off:off + counts[b]], lmk[off:off + counts[b]])
        off += counts[b]
    # trailing bytes that do not fill an f32 are ignored (chunks_exact) ...
    longer = [np.concatenate([r, np.zeros(3, np.uint8)]) for r in raw]
    ctx.detect_batch_raw(longer, shapes, ds, 0.7, 0.45)
    np.testing.assert_array_equal(ctx.detect_fetch(B)[1], det)
    # ... a shape whose product differs from the f32 count is an error, as is a foreign geometry
    bad = list(shapes)
    bad[0] = (B, 4, 20, 21)
    with pytest.raises(FdError):
        ctx.detect_batch_raw(raw, bad, ds, 0.7, 0.45)
    with pytest.raises(FdError):
        ctx.detect_batch_raw([r[:-4] for r in raw], shapes, ds, 0.7, 0.45)


def test_shared_sm_build_gives_identical_results(ctx):
    """fd_ctx_set_sharing(2) launches the 32-register build of the fused detect kernel: same bits out."""
    heads, _ = synth.make_heads(5, seed=41, n_faces=15)
    devs = [ctx.to_device(h) for h in heads]
    ds = np.array([1.0, 0.5, 0.25, 1 / 3, 2.0], np.float32)
    ctx.detect_batch(devs, 5, ds, 0.7, 0.4)
    ref = ctx.detect_fetch(5)
    ctx.set_sharing(2)
    try:
        ctx.detect_batch(devs, 5, ds, 0.7, 0.4)
        got = ctx.detect_fetch(5)
    finally:
        ctx.set_sharing(1)
    for a, b in zip(ref, got):
        np.testing.assert_array_equal(a, b)


def _random_heads(rng, B, A, fhw, hot=0.02):
    """head tensors for an arbitrary geometry: a few percent of the anchors above 0.7, plausible regression deltas"""
    heads = []
    for (fh, fw) in fhw:
        fg = rng.uniform(0, 0.6, (B, A, fh, fw)).astype(np.float32)
        hotm = rng.uniform(0, 1, fg.shape) < hot
        fg[hotm] = rng.uniform(0.7, 0.999, int(hotm.sum())).astype(np.float32)
        sc = np.concatenate([1 - fg, fg], 1)
        bb = rng.normal(0, 0.3, (B, 4 * A, fh, fw)).astype(np.float32)
        lm = rng.normal(0, 0.3, (B, 10 * A, fh, fw)).astype(np.float32)
        heads += [np.ascontiguousarray(sc), bb, lm]
    return heads


@pytest.mark.parametrize("image_wh,strides,A", [
    ((480, 320), (16, 8), 1),        # non-square, two strides, one anchor per position (runtime-A score scan)
    ((640, 640), (32, 16, 8), 3),    # three anchors per position
    ((328, 328), (8,), 2),           # 41 x 41 positions: no 128-bit score rows -> three-kernel path
])
def test_other_detector_geometries(oracle, image_wh, strides, A):
    """fd_config other than the reference's RetinaFace-640: anchors, strides and image size are configuration, not code."""
    from rs_face_detection_b200 import Context, default_config
    rng = np.random.default_rng(image_wh[0] + A)
    base = np.zeros((len(strides), A, 4), np.float32)
    for i, st in enumerate(strides):
        for a in range(A):
            half = st * (a + 1) * 1.5
            base[i, a] = [-half + st / 2, -half + st / 2, half + st / 2 - 1, half + st / 2 - 1]
    cfg = default_config()
    cfg.image_w, cfg.image_h = image_wh
    cfg.n_strides = len(strides)
    for i, st in enumerate(strides):
        cfg.strides[i] = st
    cfg.num_anchors = A
    for i in range(len(strides)):
        for a in range(A):
            for k in range(4):
                cfg.base_anchors[(i * 4 + a) * 4 + k] = float(base[i, a, k])     # [FD_MAX_STRIDES][FD_MAX_ANCHORS][4], flat
    cfg.bbox_stds[0], cfg.bbox_stds[1], cfg.bbox_stds[2], cfg.bbox_stds[3] = 0.1, 0.1, 0.2, 0.2
    cfg.landmark_std = 0.5
    c = Context(0, cfg)
    try:
        fhw = [((image_wh[1] + st - 1) // st, (image_wh[0] + st - 1) // st) for st in strides]
        B = 3
        heads = _random_heads(rng, B, A, fhw)
        ocfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.4, image_size=image_wh, strides=strides, base_anchors=base,
                                   bbox_stds=(0.1, 0.1, 0.2, 0.2), landmark_std=0.5)
        devs = [c.to_device(h) for h in heads]
        ds = np.array([1.0, 0.5, 0.75], np.float32)
        c.detect_batch(devs, B, ds, 0.7, 0.4)
        counts, det, lmk = c.detect_fetch(B)
        off = 0
        for b in range(B):
            K = _check_image(oracle, ocfg, [h[b] for h in heads], ds[b], det[off:off + counts[b]], lmk[off:off + counts[b]])
            assert K > 5
            off += counts[b]
        assert off == len(det) and off > 0
    finally:
        c.close()


def test_large_batch_more_images_than_sms(ctx, oracle):
    """B = 200 > 148 SMs: the fused kernel's CTAs run in more than one wave, so the epoch-tagged counts of later images wait
    for earlier tickets; rows must still come out in frame order, twice in a row (the tickets re-arm themselves)."""
    B = 200
    heads, _ = synth.make_heads(B, seed=123, n_faces=6)
    devs = [ctx.to_device(h) for h in heads]
    ds = (1.0 / (1 + np.arange(B) % 4)).astype(np.float32)
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.45)
    for rep in range(2):
        ctx.detect_batch(devs, B, ds, 0.7, 0.45)
        counts, det, lmk = ctx.detect_fetch(B)
        assert counts.sum() == len(det)
        off = 0
        for b in range(B):
            _check_image(oracle, cfg, [h[b] for h in heads], ds[b], det[off:off + counts[b]], lmk[off:off + counts[b]])
            off += counts[b]


def test_property_random_heads(ctx, oracle):
    """Random head tensors through the fused kernel: quantised scores (many exact ties across strides and anchors), hot
    fractions from nothing to crowded, random batch sizes and det_scales; rows and order must match the oracle."""
    hypothesis = pytest.importorskip("hypothesis")
    from hypothesis import given, settings, strategies as st

    fhw = [(20, 20), (40, 40), (80, 80)]

    @settings(max_examples=25, deadline=None, derandomize=True)
    @given(st.integers(0, 10 ** 6), st.integers(1, 4), st.sampled_from([0.0, 0.001, 0.01, 0.04, 0.1]), st.sampled_from([None, 64, 8]),
           st.sampled_from([0.3, 0.4, 0.45, 0.6]))
    def prop(seed, B, hot, levels, iou):
        rng = np.random.default_rng(seed)
        heads = _random_heads(rng, B, 2, fhw, hot=hot)
        if levels:                                   # quantise the fg scores: exact ties, bg = 1 - fg stays consistent
            for s in range(3):
                fg = np.round(heads[3 * s][:, 2:] * levels) / levels
                heads[3 * s][:, 2:] = fg
                heads[3 * s][:, :2] = 1 - fg
        ds = rng.choice(np.float32([1.0, 0.5, 0.33333334, 0.25, 1.5]), B).astype(np.float32)
        cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=iou)
        devs = [ctx.to_device(h) for h in heads]
        ctx.detect_batch(devs, B, ds, 0.7, iou)
        counts, det, lmk = ctx.detect_fetch(B)
        off = 0
        for b in range(B):
            _check_image(oracle, cfg, [h[b] for h in heads], ds[b], det[off:off + counts[b]], lmk[off:off + counts[b]])
            off += counts[b]
        assert off == len(det)
        for d in devs:
            d.free()

    prop()
