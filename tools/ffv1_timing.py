"""What encoding rendered frames as FFV1 on the GPU gives against BGR downloads and the host encoder cv2 uses. Prints one JSON
line and writes it to --out, with the card's name and power limit read by nvidia-smi in the same run.

1. MorphRenderer.download_ffv1 of a rendered ring (1920 x 1080: 64 frames, 3840 x 2160: 16 frames), timed by a host clock
   around the call (it returns after the packets are in host memory), medians of --rounds; and the device time of each FFV1
   kernel in a separate torch.profiler run, per frame.
2. Packet bytes against the BGR bytes and against what cv2.VideoWriter(fourcc FFV1) writes for the same frames (its
   Matroska packets, read back with oracle/ffv1.read_mkv), over 8 frames of each size.
3. End to end, alternating within each of --reps rounds, medians: api.morph_segments(..., pixel_format="ffv1",
   writer=api.MatroskaWriter) against api.morph_segments(...) BGR + cv2.VideoWriter(.mkv, FFV1) on this host's cores.

Frames are rendered from textured synthetic content (poppy_b200.synth noise images blurred at sigma 3, 400 matched points)."""
from __future__ import annotations

import argparse
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

from oracle import ffv1  # noqa: E402
from poppy_b200 import api, host, synth  # noqa: E402
from poppy_b200.renderer import MorphRenderer, device_count  # noqa: E402

LEVELS = 64


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


def encode_rate(r, frames, rounds):
    r.download_ffv1(0, frames)                   # staging allocated, modules loaded
    times = []
    for _ in range(rounds):
        t = time.perf_counter()
        r.download_ffv1(0, frames)
        times.append(time.perf_counter() - t)
    med = statistics.median(times)
    return {"frames": frames, "download_ffv1_s_median": med, "frames_per_s": frames / med}


def kernel_times(r, frames):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r.download_ffv1(0, frames)
        torch.cuda.synchronize()
    us = {}
    for e in prof.events():
        if "k_ffv1" in e.name:
            key = e.name.split("(")[0].split("::")[-1]
            us[key] = us.get(key, 0.0) + e.device_time
    return {k: v / frames for k, v in sorted(us.items())} | {"total_us_per_frame": sum(us.values()) / frames}


def cv2_ffv1_bytes(frames, w, h):
    import cv2
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "x.mkv")
        wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"FFV1"), 30, (w, h))
        for f in frames:
            wr.write(f)
        wr.release()
        return sum(len(p) for p in ffv1.read_mkv(path)["packets"])


def sizes(r, w, h):
    n = 8
    bgr = r.download(0, n)
    ours = sum(len(p) for p in r.download_ffv1(0, n))
    theirs = cv2_ffv1_bytes(bgr, w, h)
    return {"frames": n, "ffv1_bytes": ours, "bgr_bytes": int(bgr.nbytes), "cv2_ffv1_bytes": theirs,
            "ffv1_over_bgr": ours / bgr.nbytes, "ffv1_over_cv2_ffv1": ours / theirs, "slice_grid": ffv1.slice_grid(w, h)}


def segments(K, w, h):
    out = []
    for s in range(K):
        p1, p2 = synth.matched_points(w, h, 400, 8.0, 100 + s)
        out.append((synth.noise_image(w, h, 2 * s + 1), synth.noise_image(w, h, 2 * s + 2), None, p1, p2))
    return out


def end_to_end(w, h, n_frames, K, reps):
    import cv2
    segs = segments(K, w, h)
    frames = K * n_frames
    with tempfile.TemporaryDirectory() as d:
        def ours():
            with api.MatroskaWriter(os.path.join(d, "gpu.mkv"), w, h) as mw:
                api.morph_segments(segs, number_of_frames=n_frames, pixel_format="ffv1", writer=mw)

        def host_cv2():
            wr = cv2.VideoWriter(os.path.join(d, "cv2.mkv"), cv2.VideoWriter_fourcc(*"FFV1"), 30, (w, h))
            api.morph_segments(segs, number_of_frames=n_frames, writer=wr)
            wr.release()

        ours()
        t_ours, t_cv2 = [], []
        for _ in range(reps):
            for fn, acc in ((ours, t_ours), (host_cv2, t_cv2)):
                t = time.perf_counter()
                fn()
                acc.append(time.perf_counter() - t)
    a, b = statistics.median(t_ours), statistics.median(t_cv2)
    return {"K": K, "N": n_frames, "ffv1_gpu_mkv_frames_per_s": frames / a, "bgr_cv2_ffv1_frames_per_s": frames / b,
            "speedup": b / a}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ffv1_timing_b200.json"))
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if device_count() < 1:
        raise SystemExit("no CUDA device: this tool measures the GPU encoder and has nothing to measure without one")
    import cv2
    res = {"gpu": gpu_info(), "host_cores": os.cpu_count(), "cv2": cv2.__version__}
    for (w, h, n) in [(1920, 1080, 64), (3840, 2160, 16)]:
        r = rendered_ring(w, h, n)
        with r:
            key = f"{w}x{h}"
            res[f"encode_{key}"] = encode_rate(r, n, args.rounds)
            try:
                res[f"kernels_us_per_frame_{key}"] = kernel_times(r, n)
            except Exception as e:          # the profiler run is separate; its absence leaves the host-clock rates
                res[f"kernels_us_per_frame_{key}"] = f"not measured ({type(e).__name__}: {e})"
            res[f"bytes_{key}"] = sizes(r, w, h)
        api.release()
    res["end_to_end_1920x1080"] = end_to_end(1920, 1080, 15, 4, args.reps)
    res["end_to_end_3840x2160"] = end_to_end(3840, 2160, 6, 2, args.reps)
    api.release()
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
