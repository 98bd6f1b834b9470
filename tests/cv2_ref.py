"""The reference's stage formulas composed from cv2 calls and float32 numpy arithmetic: an independent pin of the CPU
restatement (oracle/poppy_oracle.cpp, oracle/margin.py) and of the CUDA stages where the reference library is not built.

numpy rounds every float32 operation on its own, as the reference's expressions compiled with -ffp-contract=off do.
cv2 is OpenCV 4.13 where the reference vendors 4.6.0. The two differ in two places:
  * GaussianBlur of 32F data (unsharp's blur): 4.13 runs the first 4 elements of the scalar row tail as one more vector
    step, so those elements may differ wherever (w * cn) % 8 >= 4. tail_positions() names them;
  * cvtColor(BGR2GRAY) of 32F data: 4.13 evaluates the scalar association on every column, 4.6.0 runs an 8-lane vector
    body with another association. The gray of the blend mask is therefore not restated here.
Importing this module skips the importing test module when cv2 is not installed."""
from __future__ import annotations

import math

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

f32 = np.float32


def tail_positions(w: int, cn: int) -> np.ndarray:
    """Element indices x * cn + c of a row where 4.13's 32F GaussianBlur may differ from 4.6.0's: the first 4 elements of
    the scalar tail, when the tail has at least 4."""
    n = w * cn
    start, rem = n - n % 8, n % 8
    return np.arange(start, start + 4) if rem >= 4 and w > 1 else np.zeros(0, np.int64)


def pyr_down(src, dsize=None):
    """cv::pyrDown, BORDER_DEFAULT."""
    return cv2.pyrDown(np.ascontiguousarray(src, f32), dstsize=dsize) if dsize else cv2.pyrDown(np.ascontiguousarray(src, f32))


def pyr_up(src, dsize):
    """cv::pyrUp to dsize = (width, height), BORDER_DEFAULT."""
    return cv2.pyrUp(np.ascontiguousarray(src, f32), dstsize=tuple(dsize))


def _blend(a, b, m):
    """a * m + b * (1 - m) per channel, each product and sum rounded to float (reference src/blend.hpp:68-73)."""
    m = m[..., None]
    return a * m + b * (f32(1) - m)


def _size(img):
    return img.shape[1], img.shape[0]


def lap_blend(l, r, m, levels):
    """LaplacianBlending::blend (reference src/blend.hpp:11-91): Gaussian pyramids of l, r and the mask, Laplacian
    pyramids of l and r, a blended pyramid, collapsed from the blended top level down."""
    gl, gr, gm = [np.ascontiguousarray(l, f32)], [np.ascontiguousarray(r, f32)], [np.ascontiguousarray(m, f32)]
    for _ in range(levels):
        gl.append(pyr_down(gl[-1]))
        gr.append(pyr_down(gr[-1]))
        gm.append(pyr_down(gm[-1]))
    cur = _blend(gl[levels], gr[levels], gm[levels])
    for k in range(levels - 1, -1, -1):
        lap_l = gl[k] - pyr_up(gl[k + 1], _size(gl[k]))
        lap_r = gr[k] - pyr_up(gr[k + 1], _size(gr[k]))
        cur = pyr_up(cur, _size(gl[k])) + _blend(lap_l, lap_r, gm[k])
    return cur


def gaussian9(src):
    """cv::GaussianBlur(src, Size(), 1.0): 9 taps, BORDER_DEFAULT."""
    return cv2.GaussianBlur(np.ascontiguousarray(src, f32), (0, 0), 1.0)


def median3(src):
    return cv2.medianBlur(np.ascontiguousarray(src, f32), 3)


def unsharp(src, amount, threshold=0.3):
    """poppy::unsharp_mask (reference src/util.cpp:113-148) with sigma 1: blur, subtract, 3 x 3 median, and where the
    double norm of the 3-channel median is >= threshold, add amount times it."""
    src = np.ascontiguousarray(src, f32)
    med = median3(src - gaussian9(src))
    norm = np.sqrt((med.astype(np.float64) ** 2).sum(-1))
    sharp = src + f32(amount) * med
    return np.where((norm >= float(f32(threshold)))[..., None], sharp, src)


def to_u8(v):
    """convertTo(CV_8U, 255) (reference src/algo.cpp:265): cvRound(v * 255) saturated; NaN gives 0."""
    r = np.rint(np.asarray(v, f32) * f32(255))
    return np.clip(np.nan_to_num(r, nan=0.0), 0, 255).astype(np.uint8)


def u8_to_f32(v):
    """convertTo(CV_32F, 1 / 255.0) (reference src/algo.cpp:245-248): one rounding of float(v) * float(1 / 255.0)."""
    return np.asarray(v, np.uint8).astype(f32) * f32(1 / 255.0)


def remap_u8c3(src, mapx, mapy):
    """cv::remap 8UC3, INTER_LINEAR, BORDER_CONSTANT 0 (reference src/algo.cpp:233,238)."""
    return cv2.remap(src, np.ascontiguousarray(mapx, f32), np.ascontiguousarray(mapy, f32), cv2.INTER_LINEAR,
                     borderMode=cv2.BORDER_CONSTANT, borderValue=(0, 0, 0))


def paint_triangles(w, h, tri_xy):
    """The triangle-ID map (reference src/algo.cpp:95-106,222-223): fillConvexPoly of triangle i with label i + 1, LINE_8, in
    painter's order on a zeroed 32SC1 image. tri_xy: T x 6 integer vertex coordinates (x0, y0, x1, y1, x2, y2)."""
    img = np.zeros((h, w), np.int32)
    for i, t in enumerate(np.asarray(tri_xy, np.int32).reshape(-1, 3, 2)):
        cv2.fillConvexPoly(img, np.ascontiguousarray(t), i + 1, lineType=cv2.LINE_8)
    return img


GABOR = dict(angles=16, ksize=13, sigma=5.0, lambd=10.0, gamma=0.04, psi=math.pi / 4)


def gabor_filter(src):
    """poppy::gabor_filter with its defaults (reference src/util.cpp:40-60, src/poppy.hpp:122): the mean over 16 angles
    theta_i = i * float(180 / 16) (integer division; degrees handed to an argument in radians) of filter2D with
    getGaborKernel(13 x 13), each response clamped to [0, 1]."""
    src = np.ascontiguousarray(src, f32)
    step = float(f32(180 // GABOR["angles"]))
    dst = np.zeros_like(src)
    for i in range(GABOR["angles"]):
        k = cv2.getGaborKernel((GABOR["ksize"],) * 2, GABOR["sigma"], i * step, GABOR["lambd"], GABOR["gamma"],
                               GABOR["psi"], ktype=cv2.CV_32F)
        plane = cv2.filter2D(src, -1, k)
        dst += np.clip(plane.reshape(src.shape), f32(0), f32(1))
    return dst / f32(GABOR["angles"])


def blur_margin(src, union_size):
    """poppy::blur_margin (reference src/util.cpp:574-602): src centred on a black canvas of union_size = (width, height);
    the left, right, top and bottom margins, each cut from the unblurred canvas, GaussianBlur(127 x 127, sigma 6) and
    written back in that order."""
    uw, uh = int(union_size[0]), int(union_size[1])
    rows, cols = src.shape[:2]
    margin = (cols + rows) / 100.0
    dx, dy = abs(cols - uw) / 2.0, abs(rows - uh) / 2.0
    canvas = np.zeros((uh, uw, 3), np.uint8)
    canvas[int(dy):int(dy) + rows, int(dx):int(dx) + cols] = src
    dx = 1.3 if dx == 0 else dx + margin
    dy = 1.3 if dy == 0 else dy + margin
    out = canvas.copy()
    for x, y, w, h in ((0, 0, int(dx), uh), (int(uw - dx), 0, int(dx), uh), (0, 0, uw, int(dy)), (0, int(uh - dy), uw, int(dy))):
        out[y:y + h, x:x + w] = cv2.GaussianBlur(np.ascontiguousarray(canvas[y:y + h, x:x + w]), (127, 127), 6.0)
    return out
