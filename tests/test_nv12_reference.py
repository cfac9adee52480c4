"""The NV12 -> BGR reference of the NV12 tests (tests/nv12_ref.py) equals cv2.cvtColor(COLOR_YUV2BGR_NV12)."""
import numpy as np
import pytest

from nv12_ref import bgr_to_nv12, nv12_to_bgr

cv2 = pytest.importorskip("cv2")


def _cv2(y, uv):
    return cv2.cvtColor(np.concatenate([np.ascontiguousarray(y), np.ascontiguousarray(uv)], 0), cv2.COLOR_YUV2BGR_NV12)


def test_every_yuv_triple_matches_cv2():
    """one 4096 x 4096 frame: each of the 65536 U,V pairs covers 64 2x2 blocks carrying 256 distinct Y values"""
    uvid = np.arange(65536, dtype=np.uint32)
    U = np.repeat((uvid & 255).astype(np.uint8), 64).reshape(2048, 2048)
    V = np.repeat((uvid >> 8).astype(np.uint8), 64).reshape(2048, 2048)
    k = np.tile(np.arange(64, dtype=np.uint32), 65536).reshape(2048, 2048)
    y = np.empty((4096, 4096), np.uint8)
    y[0::2, 0::2], y[0::2, 1::2], y[1::2, 0::2], y[1::2, 1::2] = 4 * k, 4 * k + 1, 4 * k + 2, 4 * k + 3
    uv = np.empty((2048, 4096), np.uint8)
    uv[:, 0::2], uv[:, 1::2] = U, V
    np.testing.assert_array_equal(nv12_to_bgr(y, uv), _cv2(y, uv))


@pytest.mark.parametrize("hw,pad", [((2, 2), 1), ((6, 10), 3), ((362, 646), 5), ((1080, 1920), 13)])
def test_pitched_planes_match_cv2(hw, pad):
    H, W = hw
    rng = np.random.default_rng(H)
    ybuf = rng.integers(0, 256, (H, W + pad), np.uint8)
    uvbuf = rng.integers(0, 256, (H // 2, W + pad + 2), np.uint8)
    y, uv = ybuf[:, :W], uvbuf[:, 1:W + 1]          # views with odd pitches and an odd start
    np.testing.assert_array_equal(nv12_to_bgr(y, uv), _cv2(y, uv))


@pytest.mark.parametrize("hw", [(3, 4), (4, 3), (5, 5)])
def test_odd_sizes_are_rejected_like_cv2(hw):
    H, W = hw
    with pytest.raises(cv2.error):
        cv2.cvtColor(np.zeros((H + (H + 1) // 2, W), np.uint8), cv2.COLOR_YUV2BGR_NV12)
    with pytest.raises(ValueError):
        nv12_to_bgr(np.zeros((H, W), np.uint8), np.zeros(((H + 1) // 2, W), np.uint8))


def test_round_trip_inputs_are_what_cv2_decodes():
    bgr = np.random.default_rng(0).integers(0, 256, (64, 96, 3), np.uint8)
    y, uv = bgr_to_nv12(bgr)
    assert y.shape == (64, 96) and uv.shape == (32, 96)
    np.testing.assert_array_equal(nv12_to_bgr(y, uv), _cv2(y, uv))
