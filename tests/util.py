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
