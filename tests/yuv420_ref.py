"""4:2:0 frames in the layouts of the *_yuv420 calls <-> BGR, on top of tests/nv12_ref.py.

A frame is a Y plane and a chroma buffer that starts where the descriptor's `uv` points, its rows `pitch_uv` bytes apart:
NV12 / NV21 hold H/2 rows of W interleaved U,V / V,U bytes; I420 / YV12 hold H/2 rows of W/2 U / V bytes followed, at
(H/2) * pitch_uv, by as many rows of the other plane.  yuv420_to_bgr re-interleaves the chroma as U,V and converts with
nv12_to_bgr; tests/test_yuv420_reference.py pins it against live cv2 for every layout."""
import numpy as np

from nv12_ref import bgr_to_nv12, nv12_to_bgr

NV12, NV21, I420, YV12 = 0, 1, 2, 3          # FD_YUV420_* of include/fd_b200.h
NAMES = {NV12: "nv12", NV21: "nv21", I420: "i420", YV12: "yv12"}
PLANAR = (I420, YV12)


def _rows(buf, first, n, pitch, width):
    """n rows of `width` bytes, `pitch` apart, from byte `first` of the flat buffer"""
    if n and first + (n - 1) * pitch + width > buf.size:
        raise ValueError("chroma buffer too short")
    return np.lib.stride_tricks.as_strided(buf[first:], (n, width), (pitch, 1)).copy()


def yuv420_to_uv(chroma, layout, H, W, pitch_uv):
    """the chroma of an H x W frame in `layout` (a buffer with rows pitch_uv bytes apart) as NV12's (H/2, W) U,V plane"""
    if H % 2 or W % 2:
        raise ValueError("4:2:0 needs an even width and height")
    if layout not in NAMES:
        raise ValueError("unknown layout %r" % (layout,))
    buf = np.ascontiguousarray(chroma, np.uint8).reshape(-1)
    h2 = H // 2
    if layout in (NV12, NV21):
        if pitch_uv < W:
            raise ValueError("pitch_uv below the width")
        c = _rows(buf, 0, h2, pitch_uv, W)
        if layout == NV12:
            return c
        uv = np.empty_like(c)
        uv[:, 0::2], uv[:, 1::2] = c[:, 1::2], c[:, 0::2]
        return uv
    if pitch_uv < W // 2:
        raise ValueError("pitch_uv below half the width")
    a, b = _rows(buf, 0, h2, pitch_uv, W // 2), _rows(buf, h2 * pitch_uv, h2, pitch_uv, W // 2)
    u, v = (a, b) if layout == I420 else (b, a)
    uv = np.empty((h2, W), np.uint8)
    uv[:, 0::2], uv[:, 1::2] = u, v
    return uv


def yuv420_to_bgr(y, chroma, layout, H, W, pitch_uv):
    """y (H, W) u8 (any strides), chroma as in yuv420_to_uv -> (H, W, 3) u8: cv2.cvtColor(COLOR_YUV2BGR_<layout>)"""
    return nv12_to_bgr(np.asarray(y, np.uint8)[:H, :W], yuv420_to_uv(chroma, layout, H, W, pitch_uv))


def bgr_to_yuv420(bgr, layout):
    """(H, W, 3) u8 with even H, W -> (y (H, W), chroma) with tight rows: (H/2, W) for NV12/NV21, (H, W/2) for I420/YV12
    (the first plane's H/2 rows, then the second's)"""
    y, uv = bgr_to_nv12(bgr)
    if layout == NV12:
        return y, uv
    if layout == NV21:
        vu = np.empty_like(uv)
        vu[:, 0::2], vu[:, 1::2] = uv[:, 1::2], uv[:, 0::2]
        return y, vu
    if layout not in PLANAR:
        raise ValueError("unknown layout %r" % (layout,))
    u, v = uv[:, 0::2], uv[:, 1::2]
    return y, np.ascontiguousarray(np.concatenate([u, v] if layout == I420 else [v, u], 0))
