"""The 4:2:0 -> BGR reference of the YUV tests (tests/yuv420_ref.py) equals cv2.cvtColor for NV21, I420 and YV12."""
import numpy as np
import pytest

from yuv420_ref import I420, NV21, YV12, bgr_to_yuv420, yuv420_to_bgr

cv2 = pytest.importorskip("cv2")
LAYOUTS = [NV21, I420, YV12]
CODE = {NV21: "COLOR_YUV2BGR_NV21", I420: "COLOR_YUV2BGR_I420", YV12: "COLOR_YUV2BGR_YV12"}


def _cv2(y, chroma, layout):
    """cv2 on the single tight buffer it reads: the Y rows, then the chroma bytes (planar: (H/2) * (W/2) per plane)"""
    H, W = y.shape
    buf = np.concatenate([np.ascontiguousarray(y).reshape(-1), np.ascontiguousarray(chroma).reshape(-1)]).reshape(H * 3 // 2, W)
    return cv2.cvtColor(buf, getattr(cv2, CODE[layout]))


def _tight(u, v, layout):
    """U and V (H/2, W/2) planes as the layout's tight chroma buffer and its pitch"""
    h2, w2 = u.shape
    if layout == NV21:
        c = np.empty((h2, 2 * w2), np.uint8)
        c[:, 0::2], c[:, 1::2] = v, u
        return c, 2 * w2
    return np.concatenate([u, v] if layout == I420 else [v, u], 0), w2


@pytest.mark.parametrize("layout", LAYOUTS)
def test_every_yuv_triple_matches_cv2(layout):
    """one 4096 x 4096 frame: each of the 65536 U,V pairs covers 64 2x2 blocks carrying 256 distinct Y values"""
    uvid = np.arange(65536, dtype=np.uint32)
    U = np.repeat((uvid & 255).astype(np.uint8), 64).reshape(2048, 2048)
    V = np.repeat((uvid >> 8).astype(np.uint8), 64).reshape(2048, 2048)
    k = np.tile(np.arange(64, dtype=np.uint32), 65536).reshape(2048, 2048)
    y = np.empty((4096, 4096), np.uint8)
    y[0::2, 0::2], y[0::2, 1::2], y[1::2, 0::2], y[1::2, 1::2] = 4 * k, 4 * k + 1, 4 * k + 2, 4 * k + 3
    chroma, pitch = _tight(U, V, layout)
    np.testing.assert_array_equal(yuv420_to_bgr(y, chroma, layout, 4096, 4096, pitch), _cv2(y, chroma, layout))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("hw,pad", [((2, 2), 1), ((6, 10), 3), ((34, 4), 2), ((362, 646), 5), ((100, 642), 7), ((1080, 1920), 13)])
def test_pitched_planes_match_cv2(layout, hw, pad):
    """noisy padding, an odd pitch and an odd start; (362, 646) and (34, 4) have H/2 odd"""
    H, W = hw
    rng = np.random.default_rng(H * 7 + layout)
    u, v = (rng.integers(0, 256, (H // 2, W // 2), np.uint8) for _ in range(2))
    y = rng.integers(0, 256, (H, W), np.uint8)
    chroma, tight = _tight(u, v, layout)
    pitch = tight + pad
    rows = chroma.shape[0]
    buf = rng.integers(0, 256, 1 + rows * pitch + 16, np.uint8)
    buf[1:1 + rows * pitch].reshape(rows, pitch)[:, :tight] = chroma
    ybuf = rng.integers(0, 256, (H, W + pad), np.uint8)
    ybuf[:, :W] = y
    np.testing.assert_array_equal(yuv420_to_bgr(ybuf[:, :W], buf[1:], layout, H, W, pitch), _cv2(y, chroma, layout))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("hw", [(3, 4), (4, 3), (5, 5)])
def test_odd_sizes_are_rejected_like_cv2(layout, hw):
    H, W = hw
    with pytest.raises(cv2.error):
        cv2.cvtColor(np.zeros((H + (H + 1) // 2, W), np.uint8), getattr(cv2, CODE[layout]))
    with pytest.raises(ValueError):
        yuv420_to_bgr(np.zeros((H, W), np.uint8), np.zeros(H * W, np.uint8), layout, H, W, W)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_round_trip_inputs_are_what_cv2_decodes(layout):
    bgr = np.random.default_rng(0).integers(0, 256, (66, 96, 3), np.uint8)
    y, chroma = bgr_to_yuv420(bgr, layout)
    assert y.shape == (66, 96) and chroma.shape == ((33, 96) if layout == NV21 else (66, 48))
    np.testing.assert_array_equal(yuv420_to_bgr(y, chroma, layout, 66, 96, chroma.shape[1]), _cv2(y, chroma, layout))
