"""NV12 <-> BGR for the NV12 tests.

nv12_to_bgr restates cv2.cvtColor(COLOR_YUV2BGR_NV12) (BT.601 limited range, OpenCV's 20-bit fixed point) in integers;
tests/test_nv12_reference.py pins it against live cv2 on every (Y, U, V) triple.  It is the reference the GPU tests compose
with the BGR oracle.  bgr_to_nv12 makes test inputs the way a decoder would hand them over (I420, U and V interleaved)."""
import numpy as np

CY, CVR, CVG, CUG, CUB = 1220542, 1673527, -852492, -409993, 2116026


def nv12_to_bgr(y, uv):
    """y (H, W) u8, uv (H/2, W) u8 interleaved U,V (any strides) -> (H, W, 3) u8 BGR"""
    y, uv = np.asarray(y, np.uint8), np.asarray(uv, np.uint8)
    H, W = y.shape
    if H % 2 or W % 2 or uv.shape != (H // 2, W):
        raise ValueError("NV12 needs an even width and height and an (H/2, W) UV plane")
    yy = np.maximum(y.astype(np.int32) - 16, 0) * CY + (1 << 19)
    u = np.repeat(np.repeat(uv[:, 0::2].astype(np.int32) - 128, 2, 0), 2, 1)
    v = np.repeat(np.repeat(uv[:, 1::2].astype(np.int32) - 128, 2, 0), 2, 1)
    b = (yy + CUB * u) >> 20
    g = (yy + CVG * v + CUG * u) >> 20
    r = (yy + CVR * v) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def bgr_to_nv12(bgr):
    """(H, W, 3) u8 with even H, W -> (y (H, W), uv (H/2, W)) via cv2 COLOR_BGR2YUV_I420"""
    import cv2
    H, W = bgr.shape[:2]
    i420 = cv2.cvtColor(np.ascontiguousarray(bgr), cv2.COLOR_BGR2YUV_I420)
    y = i420[:H].copy()
    c = i420[H:].reshape(-1)           # U then V, (H/2) x (W/2) each: not whole rows of W when H/2 is odd
    n = (H // 2) * (W // 2)
    u, v = c[:n].reshape(H // 2, W // 2), c[n:2 * n].reshape(H // 2, W // 2)
    uv = np.empty((H // 2, W), np.uint8)
    uv[:, 0::2], uv[:, 1::2] = u, v
    return y, uv
