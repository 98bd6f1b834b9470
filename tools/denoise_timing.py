#!/usr/bin/env python
"""poppy_cuda_denoise (cv::fastNlMeansDenoising, h = 10, 7 / 21) at 1080p and 4K (GPU only). Per size:
  * kernel: device duration of k_denoise from a torch.profiler trace (CUPTI kernel records), after two warm-up calls; the C
    call is stand-alone (allocation, copies and the launch inside), so the kernel alone is read from the trace. Median of
    `calls` launches. The working set (source tile rows + table) is far below L2 and is read once per CTA.
  * wall: api.denoise through the C ABI with pageable host arrays (host clock; the call ends in a synchronous copy back),
    taken with the profiler off.
  * pixel-offsets per second (pixels x 21^2 / kernel time), and the kernel against a model of ~12 lane instructions per
    pixel-offset at 1.17e12 warp instructions per second for the whole GPU (DESIGN.md section 7's issue model).
  * cv2.fastNlMeansDenoising on this host's cores, if cv2 imports, and whether its bytes equal the GPU's.
Input: a smooth seeded image with +-20 noise, on which the call moves most pixels. The card's name and power limit are read
in the same run. Writes one JSON line to `out` (default profiles/denoise_timing_b200.json) and prints it.
usage: python tools/denoise_timing.py [calls (10)] [out]"""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

from poppy_b200 import api

SIZES = {"1080p": (1920, 1080), "4k": (3840, 2160)}
H, TW, SW = 10.0, 7, 21
LANE_INSTR_PER_PIXEL_OFFSET = 12
WARP_INSTR_PER_S = 1.17e12


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": limit}
    except Exception as e:          # the numbers are still reported, marked as such
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def image(w, h, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([96 + 60 * np.sin(xx / 37.0 + c) * np.cos(yy / 53.0 - c) for c in range(3)], -1)
    return np.clip(base + rng.integers(-20, 21, base.shape), 0, 255).astype(np.uint8)


def stats(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "n": len(v)}


def kernel_ms(src, calls):
    """Device durations (ms) of the k_denoise launches of `calls` api.denoise calls, from a profiler trace."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            api.denoise(src, H, TW, SW)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        events = json.load(open(path))["traceEvents"]
    durs = [e["dur"] / 1e3 for e in events if e.get("cat") == "kernel" and "k_denoise" in e.get("name", "")]
    if len(durs) != calls:
        raise RuntimeError(f"expected {calls} k_denoise kernels in the trace, found {len(durs)}")
    return durs


def run(w, h, calls):
    src = image(w, h, w)
    out = api.denoise(src, H, TW, SW)
    api.denoise(src, H, TW, SW)                             # warm-up: module load, allocator
    wall = []
    for _ in range(calls):
        t0 = time.perf_counter()
        api.denoise(src, H, TW, SW)
        wall.append((time.perf_counter() - t0) * 1e3)
    kern = kernel_ms(src, calls)
    pixel_offsets = w * h * SW * SW
    model_ms = pixel_offsets * LANE_INSTR_PER_PIXEL_OFFSET / 32 / WARP_INSTR_PER_S * 1e3
    res = {"width": w, "height": h, "kernel": stats(kern), "wall_c_abi_pageable": stats(wall),
           "pixel_offsets": pixel_offsets, "pixel_offsets_per_s": pixel_offsets / (np.median(kern) / 1e3),
           "issue_model_ms": model_ms, "share_of_issue_model": model_ms / float(np.median(kern)),
           "pixels_changed": float((out != src).mean())}
    try:
        import cv2
    except ImportError:
        res["cv2"] = "cv2 does not import"
        return res
    t = []
    for _ in range(2):
        t0 = time.perf_counter()
        want = cv2.fastNlMeansDenoising(src, None, H, TW, SW)
        t.append((time.perf_counter() - t0) * 1e3)
    res["cv2"] = {"version": cv2.__version__, "threads": cv2.getNumThreads(), "host_cores": os.cpu_count(), **stats(t),
                  "bytes_differing_from_gpu": int((want != out).sum())}
    return res


def main():
    calls = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    path = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "profiles", "denoise_timing_b200.json")
    res = {"tool": "denoise_timing", "card": card(), "h": H, "template_window_size": TW, "search_window_size": SW,
           "sizes": {k: run(w, h, calls) for k, (w, h) in SIZES.items()}}
    line = json.dumps(res)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
