"""Interleaved RGB-family frames in the layouts of the *_rgb calls <-> BGR.

A frame is H rows of W pixels, `pitch` bytes apart: R,G,B (RGB24, 3 bytes), R,G,B,A (RGBA) or B,G,R,A (BGRA, 4 bytes; the
fourth byte is ignored), or one grey byte (GRAY8, B = G = R).  rgb_to_bgr restates cv2.cvtColor(COLOR_RGB2BGR /
COLOR_RGBA2BGR / COLOR_BGRA2BGR / COLOR_GRAY2BGR); tests/test_rgb_reference.py pins it against live cv2 for every layout."""
import numpy as np

RGB24, RGBA, BGRA, GRAY8 = 0, 1, 2, 3     # FD_RGB_* of include/fd_b200.h
NAMES = {RGB24: "rgb24", RGBA: "rgba", BGRA: "bgra", GRAY8: "gray8"}
BPP = {RGB24: 3, RGBA: 4, BGRA: 4, GRAY8: 1}
# byte positions of B, G, R in a pixel
ORDER = {RGB24: (2, 1, 0), RGBA: (2, 1, 0), BGRA: (0, 1, 2), GRAY8: (0, 0, 0)}


def rgb_to_bgr(rows, layout, H, W, pitch):
    """rows: the frame from its first byte (any array; read flat), H rows of BPP*W bytes `pitch` apart -> (H, W, 3) u8"""
    if layout not in NAMES:
        raise ValueError("unknown layout %r" % (layout,))
    if H < 1 or W < 1:
        raise ValueError("the frame needs a height and a width of at least 1")
    bpp = BPP[layout]
    if pitch < bpp * W:
        raise ValueError("pitch below the bytes per pixel times the width")
    buf = np.ascontiguousarray(rows, np.uint8).reshape(-1)
    if (H - 1) * pitch + bpp * W > buf.size:
        raise ValueError("frame buffer too short")
    px = np.lib.stride_tricks.as_strided(buf, (H, W, bpp), (pitch, bpp, 1))
    return np.ascontiguousarray(px[..., list(ORDER[layout])])


def bgr_to_rgb(bgr, layout, alpha=None):
    """(H, W, 3) u8 -> (H, W * BPP) u8 tight rows in `layout`.  GRAY8 keeps the G channel (cv2's BGR2GRAY would not give
    back a frame whose GRAY2BGR is `bgr`; the tests compare against the BGR call on GRAY2BGR of the grey frame).  alpha:
    the fourth byte of RGBA / BGRA ((H, W) u8 or a scalar; default 255)."""
    bgr = np.ascontiguousarray(bgr, np.uint8)
    H, W = bgr.shape[:2]
    if layout == GRAY8:
        return np.ascontiguousarray(bgr[..., 1])
    px = np.empty((H, W, BPP[layout]), np.uint8)
    for c, k in enumerate(ORDER[layout]):
        px[..., k] = bgr[..., c]
    if BPP[layout] == 4:
        px[..., 3] = 255 if alpha is None else alpha
    return px.reshape(H, W * BPP[layout])


def place(rows, pitch, offset=0, seed=0):
    """tight rows (H, R) -> a noisy u8 buffer holding them `pitch` bytes apart from byte `offset` (padding and the bytes
    before and after are random); returns (buf, view of the first frame byte onward)"""
    H, R = rows.shape
    rng = np.random.default_rng(seed)
    buf = rng.integers(0, 256, offset + (H - 1) * pitch + R + 16, np.uint8)
    for y in range(H):
        buf[offset + y * pitch:offset + y * pitch + R] = rows[y]
    return buf, buf[offset:]
