#!/usr/bin/env python
"""Writes tests/golden/output/i420.npz with OpenCV's cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420): the conversion of rendered BGR
frames to I420 (YUV 4:2:0) that MorphRenderer.download_i420 reproduces on the GPU. Cases: the smallest frame (2 x 2), an odd
number of chroma rows (34 x 18: 9 rows) and an odd chroma width (2 x 10: 1 column), widths where 3 * W % 4 != 0, saturated
content (pure primaries, black and white in 2 x 2 blocks and split across them), and one image holding every byte value in
every channel, with the three channels permuted differently so that all three appear at the chroma sample positions."""
import os

import cv2
import numpy as np

rng = np.random.default_rng(420)


def noise(h, w):
    return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)


def saturated(h, w):
    img = rng.choice(np.array([0, 255], np.uint8), (h, w, 3))
    blocks = np.array([[0, 0, 0], [255, 255, 255], [255, 0, 0], [0, 255, 0], [0, 0, 255], [255, 255, 0], [0, 255, 255],
                       [255, 0, 255]], np.uint8)
    for k, c in enumerate(blocks):                     # uniform 2 x 2 blocks along the top rows
        img[0:2, 2 * k:2 * k + 2] = c
    return img


def every_byte(h, w):
    """Each channel holds every value 0..255, at the chroma sample positions (even row, even column) and at the others;
    the channels are permuted independently. (h / 2) * (w / 2) must be a multiple of 256."""
    img = np.empty((h, w, 3), np.uint8)
    n_sample = (h // 2) * (w // 2)
    for c in range(3):
        img[..., c] = rng.permutation(np.arange(h * w) % 256).reshape(h, w)
        img[0::2, 0::2, c] = rng.permutation(np.arange(n_sample) % 256).reshape(h // 2, w // 2)
    assert all(len(np.unique(img[0::2, 0::2, c])) == 256 for c in range(3))
    return img


cases = [
    noise(2, 2),
    noise(18, 34),
    noise(10, 2),
    noise(6, 4),
    noise(4, 18),
    noise(2, 640),
    noise(480, 2),
    saturated(8, 16),
    saturated(18, 34),
    every_byte(64, 64),
]
out = {"n": np.int32(len(cases))}
for i, img in enumerate(cases):
    out[f"bgr{i}"] = img
    out[f"i420_{i}"] = cv2.cvtColor(img, cv2.COLOR_BGR2YUV_I420)
    print(i, img.shape, "->", out[f"i420_{i}"].shape)
out["opencv_version"] = np.array(cv2.__version__)
path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "i420.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path), "bytes")
