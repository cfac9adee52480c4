"""Drop-in single operators (processing::bbox_transform, rcnn::anchors, rcnn::bbox) through the C ABI vs the oracle."""
import numpy as np
import pytest

from detect_ref import assert_bitwise, nonlinear_transform_ref, pred_ref

pytestmark = pytest.mark.gpu
# Boxes from bbox_pred / nonlinear_pred and the log of nonlinear_transform are compared bit for bit with a restatement
# that rounds exp and log correctly (tests/detect_ref.py), not with the oracle: the oracle's expf / logf come from the
# platform's libm, which is not correctly rounded.  Everything else is compared with the oracle, bit for bit.


def _boxes(n, seed):
    rng = np.random.default_rng(seed)
    x, y = rng.uniform(-50, 600, n), rng.uniform(-50, 600, n)
    w, h = rng.uniform(1, 300, n), rng.uniform(1, 300, n)
    return np.stack([x, y, x + w, y + h], 1).astype(np.float32)


def test_anchors_plane(ctx, oracle):
    from rs_face_detection_b200.utils import synth
    from rs_face_detection_b200.rcnn.anchors import anchors
    for s, stride in enumerate((32, 16, 8)):
        n = 640 // stride
        np.testing.assert_array_equal(ctx.anchors_plane(n, n, stride, synth.BASE_ANCHORS[s]), oracle.anchors_plane(n, n, stride, synth.BASE_ANCHORS[s]))
    base = np.array([[0, 0, 15, 15], [0, 0, 31, 31]], np.float32)           # anchors.rs:30-37
    np.testing.assert_array_equal(anchors(2, 2, 16, base, ctx), oracle.anchors_plane(2, 2, 16, base))
    np.testing.assert_array_equal(ctx.anchors_plane(3, 7, 8, base), oracle.anchors_plane(3, 7, 8, base))


def test_bbox_and_landmark_pred(ctx, oracle):
    rng = np.random.default_rng(0)
    b = _boxes(5000, 1)
    d = rng.normal(0, 0.4, (5000, 4)).astype(np.float32)
    assert_bitwise(ctx.bbox_pred(b, d), pred_ref(b, d, False))
    d8 = rng.normal(0, 0.4, (5000, 8)).astype(np.float32)
    assert_bitwise(ctx.bbox_pred(b, d8), pred_ref(b, d8, False))                                            # cols >=4 copied
    assert_bitwise(ctx.nonlinear_pred(b, d8), pred_ref(b, d8, True))
    l = rng.normal(0, 0.4, (5000, 5, 2)).astype(np.float32)
    np.testing.assert_array_equal(ctx.landmark_pred(b, l), oracle.landmark_pred(b, l))                       # no exp: bit-exact
    assert ctx.bbox_pred(np.zeros((0, 4), np.float32), np.zeros((0, 4), np.float32)).shape == (0, 4)
    # reference test vectors (bbox_transform.rs:253-278)
    bx = np.array([[50, 50, 150, 150], [30, 30, 200, 200]], np.float32)
    dl = np.array([[0.1, 0.2, 0.1, 0.2, 0.2, 0.1, 0.2, 0.1], [0.2, 0.1, 0.2, 0.1, 0.1, 0.2, 0.1, 0.2]], np.float32)
    assert_bitwise(ctx.nonlinear_pred(bx, dl), pred_ref(bx, dl, True))
    pd = np.array([[0.1, 0.2, 0.1, 0.2, 0.2, 0.1, 0.2, 0.1, 0.3, 0.3], [0.2, 0.1, 0.2, 0.1, 0.1, 0.2, 0.1, 0.2, 0.3, 0.3]], np.float32)
    np.testing.assert_array_equal(ctx.landmark_pred(bx, pd), oracle.landmark_pred(bx, pd))


def test_clip_iou_transform_overlaps(ctx, oracle):
    rng = np.random.default_rng(2)
    b8 = rng.uniform(-100, 800, (777, 8)).astype(np.float32)
    np.testing.assert_array_equal(ctx.clip_boxes(b8, (640, 600)), oracle.clip_boxes(b8, (640, 600)))
    p = rng.uniform(-100, 800, (333, 10)).astype(np.float32)
    np.testing.assert_array_equal(ctx.clip_points(p, (100, 120)), oracle.clip_points(p, (100, 120)))
    b = _boxes(400, 3)
    d = rng.normal(0, 3, (400, 8)).astype(np.float32)
    np.testing.assert_array_equal(ctx.iou_pred(b, d, 2), oracle.iou_pred(b, d, 2))
    g = _boxes(400, 4)
    assert_bitwise(ctx.nonlinear_transform(b, g), nonlinear_transform_ref(b, g))
    q = _boxes(123, 5)
    np.testing.assert_array_equal(ctx.bbox_overlaps(b, q), oracle.bbox_overlaps(b, q))
    from rs_face_detection_b200.rcnn.bbox import bbox_overlaps
    bb = np.array([[10, 20, 50, 60], [15, 25, 55, 65]], np.float32)           # bbox.rs:40-48
    qq = np.array([[12, 22, 52, 62], [18, 28, 58, 68]], np.float32)
    np.testing.assert_array_equal(bbox_overlaps(bb, qq, ctx), oracle.bbox_overlaps(bb, qq))
