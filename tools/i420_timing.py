"""What downloading frames as I420 (converted on the GPU, 1.5 bytes per pixel) saves against BGR (3 bytes per pixel). Prints one
JSON line and writes it to --out, with the card's name and power limit read by nvidia-smi in the same run.

1. Downloads of a rendered ring (1920 x 1080: 120 frames, 3840 x 2160: 60 frames), BGR against I420, into pageable numpy
   memory and into pinned memory: the four variants alternate within each of --rounds rounds, each timed by a host clock
   around a call that ends in a device sync; medians are reported.
2. The device time of k_bgr_to_i420 in a separate torch.profiler run (downloads of the same ring), with the bytes it must move
   (3 read + 1.5 written per pixel) over that time, against the 7.7 TB/s of HBM3e on the B200 data sheet.
3. api.morph_segments end to end with pixel_format "bgr" against "i420", at the shapes of tools/segments_devices_timing.py
   (1080p N = 120, K in {8, 16, 32}; 4K N = 60, K in {8, 16}), alternating within each of --reps rounds; medians.

Frames come from synthetic content (poppy_b200.synth noise images, 400 matched points, gabor2 derived on the device)."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from poppy_b200 import _lib, api, host, synth  # noqa: E402
from poppy_b200.renderer import MorphRenderer, device_count  # noqa: E402

LEVELS = 64
HBM_BYTES_PER_S = 7.7e12


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out or ["unknown"]
    except Exception as e:
        return [f"unknown ({e})"]


def rendered_ring(w, h, frames):
    p1, p2 = synth.matched_points(w, h, 400, 8.0, 7)
    phases = np.linspace(0.0, 1.0, frames, dtype=np.float32)
    plan = host.SequencePlan(p1, p2, w, h, phases)
    r = MorphRenderer(w, h, LEVELS, len(p1), plan.max_triangles, frames)
    r.set_pair(synth.noise_image(w, h, 1), synth.noise_image(w, h, 2))
    r.set_points(p1, p2)
    r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
    plan.close()
    r.sync()
    return r


def pinned(nbytes):
    lib = _lib.load()
    p = C.c_void_p()
    if lib.poppy_cuda_alloc_pinned(nbytes, C.byref(p)) != 0:
        raise RuntimeError("pinned allocation failed")
    return p


def downloads(w, h, frames, rounds):
    lib = _lib.load()
    r = rendered_ring(w, h, frames)
    bgr_bytes, i420_bytes = w * h * 3, w * h * 3 // 2
    page_bgr = np.ones((frames, h, w, 3), np.uint8)
    page_i420 = np.ones((frames, h * 3 // 2, w), np.uint8)
    pin_bgr, pin_i420 = pinned(frames * bgr_bytes), pinned(frames * i420_bytes)
    variants = {
        "bgr_pageable": lambda: r.download(0, frames, out=page_bgr),
        "i420_pageable": lambda: r.download_i420(0, frames, out=page_i420),
        "bgr_pinned": lambda: (r.download_async(0, frames, pin_bgr.value, w * 3, bgr_bytes), r.sync()),
        "i420_pinned": lambda: (r._check(lib.poppy_cuda_download_i420(r._ctx, 0, frames, pin_i420, i420_bytes)), r.sync()),
    }
    for f in variants.values():             # warm-up: staging allocation, first touch of the host pages
        f()
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, f in variants.items():
            t = time.perf_counter()
            f()
            times[k].append(time.perf_counter() - t)
    out = {"frames": frames}
    for k, ts in times.items():
        s = statistics.median(ts)
        nbytes = frames * (bgr_bytes if k.startswith("bgr") else i420_bytes)
        out[k] = {"median_s": round(s, 5), "frames_per_s": round(frames / s, 1), "host_GB_per_s": round(nbytes / s / 1e9, 2),
                  "all_s": [round(t, 5) for t in ts]}
    out["i420_speedup_pageable"] = round(out["bgr_pageable"]["median_s"] / out["i420_pageable"]["median_s"], 2)
    out["i420_speedup_pinned"] = round(out["bgr_pinned"]["median_s"] / out["i420_pinned"]["median_s"], 2)
    out["kernel"] = kernel_time(r, w, h, frames, pin_i420)
    lib.poppy_cuda_free_pinned(pin_bgr)
    lib.poppy_cuda_free_pinned(pin_i420)
    r.close()
    return out


def kernel_time(r, w, h, frames, pin_i420, calls=5):
    """k_bgr_to_i420 device time from torch.profiler (a run of its own, after the timed rounds)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    lib = _lib.load()
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            r._check(lib.poppy_cuda_download_i420(r._ctx, 0, frames, pin_i420, w * h * 3 // 2))
            r.sync()
    with tempfile.TemporaryDirectory() as d:     # the trace itself is not kept
        prof.export_chrome_trace(os.path.join(d, "trace.json"))
        events = json.load(open(os.path.join(d, "trace.json")))["traceEvents"]
    durs = [e["dur"] * 1e-6 for e in events if e.get("cat") == "kernel" and "k_bgr_to_i420" in e.get("name", "")]
    if not durs:
        return {"captured": False}
    per_frame = sum(durs) / (calls * frames)
    moved = w * h * 4.5
    return {"captured": True, "launches": len(durs), "name": next(e["name"] for e in events
                                                                   if e.get("cat") == "kernel" and "k_bgr_to_i420" in e.get("name", "")),
            "us_per_frame": round(per_frame * 1e6, 2), "bytes_per_frame": int(moved),
            "achieved_TB_per_s": round(moved / per_frame / 1e12, 2),
            "share_of_7_7_TB_per_s": round(moved / per_frame / HBM_BYTES_PER_S, 3)}


def synthetic_segments(K, w, h, pairs=8):
    images = [(synth.noise_image(w, h, 100 + i), synth.noise_image(w, h, 101 + i)) for i in range(min(K, pairs))]
    return [(images[i % pairs][0], images[i % pairs][1], None) + synth.matched_points(w, h, 400, 8.0, 103 + i) for i in range(K)]


def end_to_end(w, h, n_frames, Ks, reps):
    rows = []
    segs_all = synthetic_segments(max(Ks), w, h)
    for K in Ks:
        segs = segs_all[:K]
        for fmt in ("bgr", "i420"):          # creates and sizes the cached renderer
            api.morph_segments(segs, number_of_frames=n_frames, pixel_format=fmt)
        ts = {"bgr": [], "i420": []}
        for _ in range(reps):
            for fmt in ts:
                t = time.perf_counter()
                api.morph_segments(segs, number_of_frames=n_frames, pixel_format=fmt)
                ts[fmt].append(time.perf_counter() - t)
        frames = K * n_frames
        row = {"K": K, "frames": frames}
        for fmt, v in ts.items():
            s = statistics.median(v)
            row[fmt] = {"e2e_s": round(s, 4), "frames_per_s": round(frames / s, 1), "all_s": [round(t, 4) for t in v]}
        row["i420_speedup"] = round(row["bgr"]["e2e_s"] / row["i420"]["e2e_s"], 2)
        rows.append(row)
        api.release()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "i420_timing_b200.json"))
    args = ap.parse_args()
    if device_count() < 1:
        raise SystemExit("i420_timing: no CUDA device")
    api.Settings.instance().pyramid_levels = LEVELS
    res = {"gpus": gpu_info(), "host_cpus": os.cpu_count(), "levels": LEVELS, "rounds": args.rounds, "reps": args.reps}
    res["download_1920x1080"] = downloads(1920, 1080, 120, args.rounds)
    res["download_3840x2160"] = downloads(3840, 2160, 60, args.rounds)
    res["morph_segments_1920x1080_N120"] = end_to_end(1920, 1080, 120, [8, 16, 32], args.reps)
    res["morph_segments_3840x2160_N60"] = end_to_end(3840, 2160, 60, [8, 16], args.reps)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
