"""Packed 4:2:2 frames in the layouts of the *_yuv422 calls <-> BGR, with tests/nv12_ref.py's conversion arithmetic.

A frame is H rows of W/2 macropixels of 4 bytes, `pitch` bytes apart: Y0 U Y1 V (YUY2), U Y0 V Y1 (UYVY) or Y0 V Y1 U (YVYU).
Pixel x takes its own Y and the U, V of its pair x & ~1; there is no vertical subsampling.  yuv422_to_bgr restates
cv2.cvtColor(COLOR_YUV2BGR_<layout>); tests/test_yuv422_reference.py pins it against live cv2 for every layout."""
import numpy as np

from nv12_ref import CUB, CUG, CVG, CVR, CY

YUY2, UYVY, YVYU = 0, 1, 2          # FD_YUV422_* of include/fd_b200.h
NAMES = {YUY2: "yuy2", UYVY: "uyvy", YVYU: "yvyu"}
# byte positions of Y0, U, Y1, V in a macropixel
ORDER = {YUY2: (0, 1, 2, 3), UYVY: (1, 0, 3, 2), YVYU: (0, 3, 2, 1)}


def _bgr(y, u, v):
    """BT.601 limited range as nv12_ref.nv12_to_bgr: OpenCV's 20-bit fixed point, round half up, saturate"""
    yy = np.maximum(y.astype(np.int32) - 16, 0) * CY + (1 << 19)
    u, v = u.astype(np.int32) - 128, v.astype(np.int32) - 128
    b = (yy + CUB * u) >> 20
    g = (yy + CVG * v + CUG * u) >> 20
    r = (yy + CVR * v) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def yuv422_to_bgr(rows, layout, H, W, pitch):
    """rows: the packed plane from its first byte (any array; read flat), H rows of 2W bytes `pitch` apart -> (H, W, 3) u8:
    cv2.cvtColor(COLOR_YUV2BGR_<layout>)"""
    if layout not in NAMES:
        raise ValueError("unknown layout %r" % (layout,))
    if H < 1 or W < 2 or W % 2:
        raise ValueError("packed 4:2:2 needs an even width and a height of at least 1")
    if pitch < 2 * W:
        raise ValueError("pitch below twice the width")
    buf = np.ascontiguousarray(rows, np.uint8).reshape(-1)
    if (H - 1) * pitch + 2 * W > buf.size:
        raise ValueError("packed buffer too short")
    m = np.lib.stride_tricks.as_strided(buf, (H, W // 2, 4), (pitch, 4, 1))
    y0, u, y1, v = (m[..., k] for k in ORDER[layout])
    y = np.stack([y0, y1], -1).reshape(H, W)
    return _bgr(y, np.repeat(u, 2, 1), np.repeat(v, 2, 1))


def bgr_to_yuv422(bgr, layout):
    """(H, W, 3) u8 with even W -> (H, 2W) u8 packed rows via cv2 COLOR_BGR2YUV_YUY2 / _UYVY / _YVYU"""
    import cv2
    code = {YUY2: cv2.COLOR_BGR2YUV_YUY2, UYVY: cv2.COLOR_BGR2YUV_UYVY, YVYU: cv2.COLOR_BGR2YUV_YVYU}[layout]
    H, W = bgr.shape[:2]
    return cv2.cvtColor(np.ascontiguousarray(bgr), code).reshape(H, 2 * W)
