"""Writes cv2_64x48.mkv and frames.npz here: two 64 x 48 frames written by cv2.VideoWriter with fourcc FFV1 into
Matroska (libavcodec's encoder: version 3, micro 4, Golomb-Rice coder, RGB with alpha, slice CRCs), and their BGR pixels.
tests/test_ffv1.py reads libavcodec's configuration record and slice headers from it with the restated range decoder.

    python tests/golden/output/ffv1/make_golden_ffv1.py
"""
import os

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    rng = np.random.default_rng(20261022)
    smooth = cv2.GaussianBlur(rng.integers(0, 256, (48, 64, 3), dtype=np.uint8), (0, 0), 2)
    frames = np.stack([smooth, smooth[::-1, ::-1].copy()])
    path = os.path.join(HERE, "cv2_64x48.mkv")
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"FFV1"), 30, (64, 48))
    assert w.isOpened()
    for f in frames:
        w.write(f)
    w.release()
    np.savez_compressed(os.path.join(HERE, "frames.npz"), frames=frames)
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
