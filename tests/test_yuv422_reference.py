"""The packed 4:2:2 -> BGR reference of the YUV 4:2:2 tests (tests/yuv422_ref.py) equals cv2.cvtColor for YUY2, UYVY and YVYU."""
import numpy as np
import pytest

from yuv422_ref import UYVY, YUY2, YVYU, bgr_to_yuv422, yuv422_to_bgr

cv2 = pytest.importorskip("cv2")
LAYOUTS = [YUY2, UYVY, YVYU]
CODE = {YUY2: "COLOR_YUV2BGR_YUY2", UYVY: "COLOR_YUV2BGR_UYVY", YVYU: "COLOR_YUV2BGR_YVYU"}


def _cv2(rows, layout):
    """cv2 on the tight (H, W, 2) array it reads"""
    H, W2 = rows.shape
    return cv2.cvtColor(np.ascontiguousarray(rows).reshape(H, W2 // 2, 2), getattr(cv2, CODE[layout]))


def test_every_yuv_triple_matches_cv2():
    """one 4096 x 4096 YUY2 frame: each of the 65536 U,V pairs is carried by 128 macropixels holding 256 distinct Y values"""
    m = np.arange(1 << 23, dtype=np.uint32)
    uv, k = m >> 7, m & 127
    mp = np.stack([2 * k, uv & 255, 2 * k + 1, uv >> 8], -1).astype(np.uint8)   # Y0 U Y1 V
    rows = mp.reshape(4096, 8192)
    np.testing.assert_array_equal(yuv422_to_bgr(rows, YUY2, 4096, 4096, 8192), _cv2(rows, YUY2))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("hw,pad", [((1, 2), 1), ((3, 4), 3), ((7, 10), 2), ((361, 646), 5), ((1080, 1920), 13)])
def test_pitched_rows_match_cv2(layout, hw, pad):
    """noisy padding, an odd pitch and an odd start; odd heights are accepted"""
    H, W = hw
    rng = np.random.default_rng(H * 7 + layout)
    rows = rng.integers(0, 256, (H, 2 * W), np.uint8)
    pitch = 2 * W + pad
    buf = rng.integers(0, 256, 1 + H * pitch + 16, np.uint8)
    buf[1:1 + H * pitch].reshape(H, pitch)[:, :2 * W] = rows
    np.testing.assert_array_equal(yuv422_to_bgr(buf[1:], layout, H, W, pitch), _cv2(rows, layout))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("hw", [(2, 3), (4, 5), (1, 1)])
def test_odd_widths_are_rejected_like_cv2(layout, hw):
    H, W = hw
    with pytest.raises(cv2.error):
        cv2.cvtColor(np.zeros((H, W, 2), np.uint8), getattr(cv2, CODE[layout]))
    with pytest.raises(ValueError):
        yuv422_to_bgr(np.zeros(H * 2 * W + 8, np.uint8), layout, H, W, 2 * W)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_round_trip_inputs_are_what_cv2_decodes(layout):
    bgr = np.random.default_rng(0).integers(0, 256, (67, 96, 3), np.uint8)
    rows = bgr_to_yuv422(bgr, layout)
    assert rows.shape == (67, 192)
    np.testing.assert_array_equal(yuv422_to_bgr(rows, layout, 67, 96, 192), _cv2(rows, layout))
