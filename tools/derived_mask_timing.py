#!/usr/bin/env python
"""Conditioning of one pair for the renderer, by two routes, alternating in one process (GPU only):
  (a) explicit: gabor2 = api.gabor_filter(corrected2 * float32(1/255)) through host memory, then MorphRenderer.set_pair
      with it;
  (b) derived:  MorphRenderer.set_pair(corrected1, corrected2, None) - k_gabor_mask_basis on the device.
Inputs: a seeded synth.noise_image pair (pageable host arrays) at 1080p and 4K. Both routes end in a synchronise
(gabor_filter copies back, set_pair waits for its uploads), so the host clock around them is the wall time per pair.
Device time of k_gabor_mask_basis: the CUDA events the context's stage timing records around it (kernel class "misc",
the only timed launch of set_pair), after one warm-up pair. PCIe bytes per pair are computed from the shapes. The card's
name and power limit are read in the same run. Prints one JSON line.
usage: python tools/derived_mask_timing.py [pairs per route (10)]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from poppy_b200 import api, synth
from poppy_b200.renderer import MorphRenderer

SIZES = {"1080p": (1920, 1080), "4k": (3840, 2160)}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": limit}
    except Exception as e:          # the numbers are still reported, marked as such
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def pcie_bytes(w, h):
    px = w * h
    return {"explicit": {"gabor_filter_in": 12 * px, "gabor_filter_out": 12 * px, "set_pair": 3 * px + 3 * px + 12 * px,
                         "total": 42 * px},
            "derived": {"set_pair": 6 * px, "total": 6 * px}}


def misc_ms(r):
    return r.stage_times()["misc"]["ms"]


def run(w, h, pairs):
    c1, c2 = synth.noise_image(w, h, 101), synth.noise_image(w, h, 102)
    inv255 = np.float32(1 / 255.0)
    with MorphRenderer(w, h, 6, 64, 64, 1, stage_timing=True) as r:
        def explicit():
            r.set_pair(c1, c2, api.gabor_filter(c2.astype(np.float32) * inv255))

        def derived():
            r.set_pair(c1, c2, None)

        explicit(), derived()                       # warm-up: module load, taps upload, staging allocation
        wall = {"explicit": [], "derived": []}
        kernel = []
        for _ in range(pairs):
            for name, fn in (("explicit", explicit), ("derived", derived)):
                before = misc_ms(r)
                t0 = time.perf_counter()
                fn()
                wall[name].append((time.perf_counter() - t0) * 1e3)
                if name == "derived":
                    kernel.append(misc_ms(r) - before)
    stats = lambda v: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "n": len(v)}
    return {"width": w, "height": h, "wall_per_pair": {k: stats(v) for k, v in wall.items()},
            "k_gabor_mask_basis_device": stats(kernel),
            "speedup_wall_median": float(np.median(wall["explicit"]) / np.median(wall["derived"])),
            "pcie_bytes_per_pair": pcie_bytes(w, h)}


def main():
    pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    res = {"tool": "derived_mask_timing", "card": card(), "pairs_per_route": pairs,
           "sizes": {k: run(w, h, pairs) for k, (w, h) in SIZES.items()}}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
