"""The RGB-family -> BGR reference of the RGB tests (tests/rgb_ref.py) equals cv2.cvtColor for RGB24, RGBA, BGRA and GRAY8."""
import numpy as np
import pytest

from rgb_ref import BGRA, BPP, GRAY8, RGB24, RGBA, bgr_to_rgb, place, rgb_to_bgr

cv2 = pytest.importorskip("cv2")
LAYOUTS = [RGB24, RGBA, BGRA, GRAY8]
CODE = {RGB24: "COLOR_RGB2BGR", RGBA: "COLOR_RGBA2BGR", BGRA: "COLOR_BGRA2BGR", GRAY8: "COLOR_GRAY2BGR"}


def _cv2(rows, layout):
    """cv2 on the tight (H, W, channels) array it reads"""
    H, R = rows.shape
    bpp = BPP[layout]
    src = np.ascontiguousarray(rows).reshape(H, R // bpp, bpp) if bpp > 1 else np.ascontiguousarray(rows)
    return cv2.cvtColor(src, getattr(cv2, CODE[layout]))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("hw,pad", [((1, 1), 1), ((1, 3), 0), ((3, 4), 3), ((7, 9), 2), ((361, 645), 5), ((1080, 1920), 13)])
def test_pitched_rows_match_cv2(layout, hw, pad):
    """noisy padding, an odd pitch and an odd start"""
    H, W = hw
    rng = np.random.default_rng(H * 7 + W + layout)
    rows = rng.integers(0, 256, (H, BPP[layout] * W), np.uint8)
    pitch = BPP[layout] * W + pad
    _, frame = place(rows, pitch, offset=1, seed=H + layout)
    np.testing.assert_array_equal(rgb_to_bgr(frame, layout, H, W, pitch), _cv2(rows, layout))


@pytest.mark.parametrize("layout", [RGBA, BGRA])
def test_the_fourth_byte_changes_nothing(layout):
    rng = np.random.default_rng(layout)
    bgr = rng.integers(0, 256, (33, 47, 3), np.uint8)
    a = bgr_to_rgb(bgr, layout, alpha=rng.integers(0, 256, (33, 47), np.uint8))
    b = bgr_to_rgb(bgr, layout, alpha=0)
    assert not np.array_equal(a, b)
    np.testing.assert_array_equal(_cv2(a, layout), _cv2(b, layout))
    np.testing.assert_array_equal(rgb_to_bgr(a, layout, 33, 47, 4 * 47), bgr)
    np.testing.assert_array_equal(rgb_to_bgr(b, layout, 33, 47, 4 * 47), bgr)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_builders_make_what_cv2_converts_back(layout):
    """bgr_to_rgb builds the frame whose cvtColor is the BGR frame (GRAY8: the frame of its G channel)"""
    bgr = np.random.default_rng(0).integers(0, 256, (67, 95, 3), np.uint8)
    rows = bgr_to_rgb(bgr, layout)
    assert rows.shape == (67, 95 * BPP[layout])
    want = np.repeat(bgr[..., 1:2], 3, -1) if layout == GRAY8 else bgr
    np.testing.assert_array_equal(_cv2(rows, layout), want)
    np.testing.assert_array_equal(rgb_to_bgr(rows, layout, 67, 95, 95 * BPP[layout]), want)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_bad_geometry_is_rejected(layout):
    bpp = BPP[layout]
    with pytest.raises(ValueError):
        rgb_to_bgr(np.zeros(64, np.uint8), layout, 2, 4, bpp * 4 - 1)
    with pytest.raises(ValueError):
        rgb_to_bgr(np.zeros(64, np.uint8), layout, 0, 4, bpp * 4)
    with pytest.raises(ValueError):
        rgb_to_bgr(np.zeros(64, np.uint8), layout, 2, 0, bpp * 4)
    with pytest.raises(ValueError):
        rgb_to_bgr(np.zeros(64, np.uint8), 4, 2, 4, 16)
