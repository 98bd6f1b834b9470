"""TEST INFRASTRUCTURE — CPU restatement (numpy, integer arithmetic) of cv::fastNlMeansDenoising for 8-bit BGR images,
the --denoise step the reference's run() applies to every input image (src/poppy.cpp:172, 269-311).

OpenCV runs FastNlMeansDenoisingInvoker<Vec3b, int, unsigned, DistSquared, int> (photo/src/fast_nlmeans_denoising_invoker.hpp):
  * windows: th = tw // 2, sh = sw // 2, then tw = 2 th + 1, sw = 2 sh + 1 (even sizes round up);
  * border: the source extended by sh + th on every side, BORDER_REFLECT_101 (cv::borderInterpolate: reflect repeatedly,
    index 0 on a length-1 axis), so the extension may be larger than the image;
  * weights: mult = INT_MAX // (sw^2 * 255); shift = least p with 2^p >= tw^2, m = 2^shift / tw^2; for a < int(3 * 255^2 / m + 1):
    w = exp(-a m / den) with den = float32(float32(h * h) * 3), 1 where that is NaN (h = 0), lut[a] = cvRound(mult * w)
    (half to even), and 0 where lut[a] < 0.001 * mult;
  * per pixel p, for every offset o of the search window: D = sum over the template around p of sum_c (I(q) - I(q + o))^2,
    wt = lut[D >> shift], W += wt, E_c += wt * I_c(p + o); out_c = (E_c + W // 2) // W.
Everything but the table is integer arithmetic, so the order of summation is immaterial. Checked against cv2 byte for byte
(tests/test_denoise.py). One numpy pass per offset: fine up to about 640 x 360. Only tests may import this module."""
from __future__ import annotations

import math

import numpy as np

INT_MAX = 2 ** 31 - 1
CHANNELS = 3


def reflect101(n: int, lo: int, hi: int) -> np.ndarray:
    """cv::borderInterpolate(p, n, BORDER_REFLECT_101) for p in [lo, hi)."""
    out = []
    for p in range(lo, hi):
        if n == 1:
            out.append(0)
            continue
        while p < 0 or p >= n:
            p = -p if p < 0 else 2 * (n - 1) - p
        out.append(p)
    return np.array(out, np.int64)


def windows(template_window_size: int, search_window_size: int) -> tuple[int, int]:
    """Half sizes (th, sh) after rounding even sizes up."""
    return template_window_size // 2, search_window_size // 2


def weight_table(h: float, template_window_size: int = 7, search_window_size: int = 21) -> tuple[np.ndarray, int]:
    """(lut, shift): the invoker's fixed-point weight table (int(3 * 255^2 / m + 1) entries). The weights fall with the
    index, so the entries past the first zero are 0 and are not evaluated."""
    th, sh = windows(template_window_size, search_window_size)
    tw, sw = 2 * th + 1, 2 * sh + 1
    mult = min(INT_MAX // (sw * sw * 255), INT_MAX)
    shift = 0
    while (1 << shift) < tw * tw:
        shift += 1
    m = float(1 << shift) / (tw * tw)
    amax = int(255 * 255 * CHANNELS / m + 1)
    hf = np.float32(h)
    with np.errstate(over="ignore"):                # h * h may overflow float to inf, as it does in OpenCV: every weight 1
        den = float(np.float32(hf * hf) * np.float32(CHANNELS))
    lut = np.zeros(amax, np.int64)
    for a in range(amax):
        d = a * m
        if den != 0.0:
            w = math.exp(-d / den)
        else:
            w = 1.0 if d == 0.0 else 0.0           # -d / 0: NaN (-> 1) at d = 0, -inf (-> exp 0) elsewhere
        v = int(np.rint(mult * w))
        if v < 0.001 * mult:
            v = 0
        lut[a] = v
        if v == 0:                                  # the weights fall with a: every later entry is 0 as well
            break
    return lut, shift


def nonzero_prefix(lut: np.ndarray) -> int:
    """Index of the table's first zero (its length if it has none)."""
    z = np.flatnonzero(lut == 0)
    return int(z[0]) if z.size else int(lut.size)


def denoise(src: np.ndarray, h: float = 3.0, template_window_size: int = 7, search_window_size: int = 21) -> np.ndarray:
    """cv::fastNlMeansDenoising(src, h, template_window_size, search_window_size) of an H x W x 3 uint8 image."""
    src = np.asarray(src)
    assert src.dtype == np.uint8 and src.ndim == 3 and src.shape[2] == CHANNELS
    th, sh = windows(template_window_size, search_window_size)
    tw = 2 * th + 1
    B = sh + th
    H, W, _ = src.shape
    ext = src[reflect101(H, -B, H + B)][:, reflect101(W, -B, W + B)].astype(np.int64)
    lut, shift = weight_table(h, template_window_size, search_window_size)
    n = nonzero_prefix(lut)
    lut = np.append(lut[:n], 0)                     # entries past the first zero are all 0: clamp the index there
    ws = np.zeros((H, W), np.int64)
    est = np.zeros((H, W, CHANNELS), np.int64)
    cen = ext[sh:sh + H + 2 * th, sh:sh + W + 2 * th]
    for dy in range(-sh, sh + 1):
        for dx in range(-sh, sh + 1):
            oth = ext[sh + dy:sh + dy + H + 2 * th, sh + dx:sh + dx + W + 2 * th]
            d = ((cen - oth) ** 2).sum(-1)
            c = np.cumsum(np.cumsum(np.pad(d, ((1, 0), (1, 0))), 0), 1)
            box = c[tw:, tw:] - c[:-tw, tw:] - c[tw:, :-tw] + c[:-tw, :-tw]
            wgt = lut[np.minimum(box >> shift, n)]
            ws += wgt
            est += wgt[..., None] * oth[th:th + H, th:th + W]
    out = (est + (ws // 2)[..., None]) // ws[..., None]
    return np.clip(out, 0, 255).astype(np.uint8)
