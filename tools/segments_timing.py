"""Device time per frame of K segments rendered together (poppy_cuda_render_segments) against the same K chains rendered one
after another, on one context. Prints one JSON line (and writes it to --out).

  512 x 512, 64 levels: K in {1, 4, 16, 32}, 60 frames, segments derived from tests/golden/full/c1.npz (seeded point jitter,
                        the reversed pair every other segment)
  1920 x 1080, 64 levels: K in {1, 4, 8}, 120 frames, synthetic segments (synth.make_inputs)

The two routes run alternately, --reps times each; medians are reported. End-to-end frames/s adds the host planning
(SequencePlan per segment) and a device sync to the batched render, as api.morph_segments spends it apart from downloads."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from poppy_b200 import api, host, synth  # noqa: E402
from poppy_b200.renderer import MorphRenderer  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:
        return f"unknown ({e})"


def c1_segments(K):
    g = np.load(os.path.join(ROOT, "tests", "golden", "full", "c1.npz"))
    c1, c2 = g["corrected1"], g["corrected2"]
    rng = np.random.default_rng(2024)
    segs = []
    for i in range(K):
        p1 = (g["pts1"] + rng.normal(0, 2.0, g["pts1"].shape)).astype(np.float32)
        p2 = (g["pts2"] + rng.normal(0, 2.0, g["pts2"].shape)).astype(np.float32)
        segs.append((c1, c2, p1, p2) if i % 2 == 0 else (c2, c1, p2, p1))
    return segs


def synthetic_segments(K, w, h):
    segs = []
    for i in range(K):
        inp = synth.make_inputs(w, h, 400, seed=100 + i)
        segs.append((inp.bgr1, inp.bgr2, inp.pts1, inp.pts2))
    return segs


def measure(segs, n_frames, levels, reps):
    h, w = segs[0][0].shape[:2]
    K = len(segs)
    ratio = np.array([host.chain_ratio(j, n_frames) for j in range(n_frames)], np.float64)
    shape = ratio.astype(np.float32)
    plans = [host.SequencePlan(p1, p2, w, h, shape, chain=True) for _, _, p1, p2 in segs]
    n_max = max(p.n for p in plans)
    r = MorphRenderer(w, h, levels, n_max, max(max(p.max_triangles for p in plans), 2 * n_max + 16), K * n_frames)
    r.set_segments(K, n_frames)
    for s, (c1, c2, p1, p2) in enumerate(segs):
        r.set_segment(s, c1, c2, None, p1, p2)
    tri, offs = api.interleave_segment_plans(plans, n_frames)

    def batched():
        r.render_segments(0, shape, ratio, tri, offs)
        return r.last_render_ms()

    def sequential():
        ms = 0.0
        for (c1, c2, p1, p2), p in zip(segs, plans):
            r.set_pair(c1, c2, None)
            r.set_points(p1, p2)
            r.render(shape, ratio, p.tri_idx, p.tri_offsets, chain=True)
            ms += r.last_render_ms()
        return ms

    batched(), sequential()                           # warm-up of every shape
    b, q = [], []
    for _ in range(reps):
        b.append(batched())
        q.append(sequential())
    launches0 = r.launch_count()
    r.render_segments(0, shape, ratio, tri, offs)
    r.sync()
    launches = (r.launch_count() - launches0) / n_frames
    for p in plans:
        p.close()
    # end to end: plan every segment on the host, render the batch, sync
    e2e = []
    for _ in range(max(2, reps // 2)):
        t0 = time.perf_counter()
        pl = [host.SequencePlan(p1, p2, w, h, shape, chain=True) for _, _, p1, p2 in segs]
        t_i, o_i = api.interleave_segment_plans(pl, n_frames)
        r.render_segments(0, shape, ratio, t_i, o_i)
        r.sync()
        e2e.append(time.perf_counter() - t0)
        for p in pl:
            p.close()
    r.close()
    frames = K * n_frames
    mb, mq = statistics.median(b), statistics.median(q)
    return {"K": K, "frames": frames, "batched_ms": round(mb, 3), "sequential_ms": round(mq, 3),
            "batched_us_per_frame": round(1000 * mb / frames, 2), "sequential_us_per_frame": round(1000 * mq / frames, 2),
            "speedup": round(mq / mb, 2), "launches_per_step": launches,
            "e2e_frames_per_s": round(frames / statistics.median(e2e), 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "host_cpus": os.cpu_count(), "reps": args.reps, "512x512_L64_N60": [], "1920x1080_L64_N120": []}
    for K in (1, 4, 16, 32):
        res["512x512_L64_N60"].append(measure(c1_segments(K), 60, 64, args.reps))
    for K in (1, 4, 8):
        res["1920x1080_L64_N120"].append(measure(synthetic_segments(K, 1920, 1080), 120, 64, args.reps))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
