#!/usr/bin/env python
"""Writes tests/golden/conditioning/denoise.npz with OpenCV's cv2.fastNlMeansDenoising (8-bit BGR, NORM_L2), the call the
reference's run() makes under --denoise (src/poppy.cpp:172, 269-311). The content is a blurred base with noise of +-8 to
+-25, on which denoising moves most pixels (a low h on strong noise would change nothing); one image also holds pixels at 0
and 255. Sizes include images smaller than the border (1 x 1, 5 x 3, 2 x 7) and odd sizes."""
import os

import cv2
import numpy as np

rng = np.random.default_rng(2026)


def noisy(h, w, amp, sigma=2.0):
    base = cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), sigma)
    return np.clip(base.astype(np.int32) + rng.integers(-amp, amp + 1, base.shape), 0, 255).astype(np.uint8)


def saturated(h, w):
    img = noisy(h, w, 20)
    img[: h // 3, : w // 2] = np.clip(img[: h // 3, : w // 2].astype(np.int32) - 200, 0, 255).astype(np.uint8)
    img[-(h // 3):, w // 2:] = np.clip(img[-(h // 3):, w // 2:].astype(np.int32) + 200, 0, 255).astype(np.uint8)
    img[h // 2, :, 1] = 255
    img[:, w // 3, 2] = 0
    return img


# (image, h, template_window_size, search_window_size)
cases = [
    (noisy(37, 53, 25), 10.0, 7, 21),
    (noisy(40, 29, 8, sigma=8.0), 3.0, 7, 21),
    (noisy(1, 1, 20), 10.0, 7, 21),
    (noisy(5, 3, 20), 10.0, 7, 21),
    (noisy(2, 7, 25), 25.0, 5, 15),
    (noisy(31, 45, 15), 0.0, 7, 21),
    (noisy(33, 27, 20), 10.0, 5, 15),
    (noisy(26, 39, 25), 25.0, 3, 35),
    (noisy(29, 34, 12), 10.0, 8, 20),
    (noisy(65, 33, 18), 10.0, 7, 21),
    (saturated(35, 41), 25.0, 7, 21),
]
out = {"n": np.int32(len(cases))}
for i, (img, h, tw, sw) in enumerate(cases):
    out[f"src{i}"] = img
    out[f"params{i}"] = np.array([h, tw, sw], np.float64)
    out[f"dst{i}"] = cv2.fastNlMeansDenoising(img, None, h, tw, sw)
    print(i, img.shape, h, tw, sw, "changed", float((out[f"dst{i}"] != img).mean()))
out["opencv_version"] = np.array(cv2.__version__)
path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "denoise.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path), "bytes")
