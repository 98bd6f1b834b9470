"""Shared helpers of the parity tests."""
from __future__ import annotations

import numpy as np


def reference():
    """What the parity tests compare with: the reference library (oracle/ref.py) where oracle/_ref is built, else the CPU
    restatement (oracle/port.py) with the same morph_images / chain / stages entry points, which tests/test_golden.py
    pins bit for bit to vectors stored from the reference library. The restatement triangulates with the product's own
    host stage (poppy_b200.host), so on that path a test checks everything after the triangle lists against an independent
    implementation but not the lists themselves: those are pinned to cv::Subdiv2D only by tests/golden/topology.npz and
    the golden frames (tests/test_host_topology.py, tests/test_golden.py)."""
    from oracle import port, ref
    return ref if ref.available() else port


def any_size_inputs(w, h, seed=0, smooth=False):
    """(bgr1, bgr2, gabor2, pts1, pts2) at any frame size, down to 1 x 1 (poppy_b200.synth needs about 8 x 8).
    Images: seeded random bytes, or with smooth=True slow sinusoids in 70..190, whose lapBlend leaves most strip chunks
    calm for the calm unsharp route. gabor2: a smooth field. Points: a few interior ones, points outside the frame
    (clip_points moves them to the border), repeated points where w or h is 1, and the four corners."""
    rng = np.random.Generator(np.random.PCG64(seed * 7919 + w * 31 + h))
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    if smooth:
        bgr1, bgr2 = (np.stack([130 + 60 * np.sin(x / (17.0 + 4 * c + k) + y / (23.0 + 3 * c) + c + 2 * k) for c in range(3)],
                               -1).round().astype(np.uint8) for k in range(2))
    else:
        bgr1 = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        bgr2 = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    gab = np.stack([0.5 + 0.45 * np.sin(x / (7.0 + 3 * c) + y / (5.0 + 2 * c) + c) for c in range(3)], -1).astype(np.float32)
    corners = np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float32)
    inner = rng.uniform(0.0, 1.0, (6, 2)) * [w - 1, h - 1]
    outside = np.array([[-2.5, 0.3 * (h - 1)], [w + 3.25, 0.6 * (h - 1)], [0.5 * (w - 1), -1.75], [0.4 * (w - 1), h + 2.5]])
    pts1 = np.concatenate([inner, outside]).astype(np.float32)
    pts2 = (pts1 + rng.uniform(-2.0, 2.0, pts1.shape)).astype(np.float32)
    pts2[:len(inner)] = np.clip(pts2[:len(inner)], 0, [w - 1, h - 1])
    if w == 1 or h == 1:
        pts1 = np.concatenate([pts1, pts1[:2]])
        pts2 = np.concatenate([pts2, pts2[:2]])
    pts1 = np.concatenate([pts1, corners])
    pts2 = np.concatenate([pts2, corners])
    return bgr1, bgr2, gab, pts1, pts2


def bits_differ(a: np.ndarray, b: np.ndarray) -> int:
    """Number of elements whose bit patterns differ (floats compared as uint32, so -0/+0 and NaNs count)."""
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.dtype.kind == "f":
        return int((np.ascontiguousarray(a).view(np.uint32) != np.ascontiguousarray(b).view(np.uint32)).sum())
    return int((a != b).sum())


def psnr(a: np.ndarray, b: np.ndarray) -> float:
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return float("inf") if mse == 0 else 10.0 * np.log10(255.0 ** 2 / mse)


def frame_report(got: np.ndarray, want: np.ndarray) -> dict:
    d = np.abs(got.astype(np.int32) - want.astype(np.int32))
    return {"differing_bytes": int((d != 0).sum()), "within_1": float((d <= 1).mean()), "max_abs": int(d.max()),
            "psnr": psnr(got, want)}


def assert_frame_parity(got: np.ndarray, want: np.ndarray, what=""):
    """North-star tolerance (BASELINE.json): >= 99.9 % of 8-bit values within +-1 LSB, max abs error <= 2,
    PSNR >= 50 dB per frame."""
    r = frame_report(got, want)
    assert r["within_1"] >= 0.999 and r["max_abs"] <= 2 and r["psnr"] >= 50.0, (what, r)
    return r


def flat_tri(tri_lists):
    """list of (T_f x 3) arrays -> (concatenated, offsets)."""
    offs = np.zeros(len(tri_lists) + 1, np.int32)
    offs[1:] = np.cumsum([len(t) for t in tri_lists])
    cat = np.concatenate(tri_lists).astype(np.int32) if len(tri_lists) else np.zeros((0, 3), np.int32)
    return cat, offs


def frame_checksum(frame: np.ndarray) -> int:
    """Position-weighted 64-bit checksum of a frame's bytes: the function of k_checksum (device) and of the
    full-pipeline harness (oracle/ref_full_harness.cpp)."""
    b = np.ascontiguousarray(frame).reshape(-1).astype(np.uint64)
    i = np.arange(b.size, dtype=np.uint64)
    with np.errstate(over="ignore"):
        k = (i + np.uint64(0x9E3779B97F4A7C15)) * np.uint64(0xBF58476D1CE4E5B9)
        k ^= k >> np.uint64(29)
        return int(((b + np.uint64(1)) * (k | np.uint64(1))).sum(dtype=np.uint64))
