"""TEST INFRASTRUCTURE — CPU restatement (numpy, int32 arithmetic) of cv::cvtColor(bgr, out, COLOR_BGR2YUV_I420) for an
8-bit BGR image of even width and height, as OpenCV 4.13 computes it (imgproc/src/color_yuv.simd.hpp, RGB888toYUV420pInvoker):

    SHIFT = 20, HALF = 1 << 19
    Y[y][x] = sat_u8(( 269484 R + 528482 G + 102760 B + HALF + (16 << 20)) >> 20)      every pixel
    U[i][j] = sat_u8((-155188 R - 305135 G + 460324 B + HALF + (128 << 20)) >> 20)     R, G, B of pixel (2i, 2j) only
    V[i][j] = sat_u8(( 460324 R - 385875 G -  74448 B + HALF + (128 << 20)) >> 20)     R, G, B of pixel (2i, 2j) only

with `>>` an arithmetic shift. Chroma is the top-left pixel of each 2 x 2 block, not an average. The result is an
(3H/2) x W uint8 array: the Y plane (H rows of W), then U and V, (W/2) x (H/2) bytes each, tightly packed, the way cv2 returns
it. BT.601 limited range (Y 16-235). Equal to cv2 on every 24-bit colour and on random images (tests/test_i420.py). Only tests
and tools may import this module."""
from __future__ import annotations

import numpy as np

SHIFT = 20
HALF = 1 << (SHIFT - 1)
Y_COEF = (269484, 528482, 102760)           # R, G, B
U_COEF = (-155188, -305135, 460324)
V_COEF = (460324, -385875, -74448)


def _mix(coef, r, g, b, offset):
    v = (np.int32(coef[0]) * r + np.int32(coef[1]) * g + np.int32(coef[2]) * b + np.int32(HALF + (offset << SHIFT))) >> SHIFT
    return np.clip(v, 0, 255).astype(np.uint8)


def restate(bgr: np.ndarray) -> np.ndarray:
    """cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420) of one H x W x 3 uint8 frame, or of a stack (..., H, W, 3) of them:
    returns (..., 3H/2, W). ValueError for an odd H or W (cv2 throws)."""
    bgr = np.asarray(bgr)
    if bgr.dtype != np.uint8 or bgr.ndim < 3 or bgr.shape[-1] != 3:
        raise ValueError("expected (..., H, W, 3) uint8")
    h, w = bgr.shape[-3:-1]
    if h % 2 or w % 2 or h == 0 or w == 0:
        raise ValueError(f"I420 needs an even frame size, got {w}x{h}")
    b, g, r = (bgr[..., c].astype(np.int32) for c in range(3))
    lead = bgr.shape[:-3]
    y = _mix(Y_COEF, r, g, b, 16)
    rs, gs, bs = r[..., 0::2, 0::2], g[..., 0::2, 0::2], b[..., 0::2, 0::2]
    u = _mix(U_COEF, rs, gs, bs, 128).reshape(lead + (-1,))
    v = _mix(V_COEF, rs, gs, bs, 128).reshape(lead + (-1,))
    chroma = np.concatenate([u, v], axis=-1).reshape(lead + (h // 2, w))
    return np.concatenate([y, chroma], axis=-2)
