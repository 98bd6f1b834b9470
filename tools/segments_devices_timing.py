"""End-to-end frames/s of api.morph_segments with the segments sharded over 1, 2, 4 and 8 GPUs of one box (as many as it has),
frames returned to the host. Prints one JSON line and writes it to --out.

  1920 x 1080, 64 levels, N = 120: K in {8, 16, 32}
  3840 x 2160, 64 levels, N = 60:  K in {8, 16}

Synthetic segments as tools/segments_timing.py builds them (synth noise images, 400 matched points, gabor2 derived on the
device), except that the images come from 8 seeded pairs used in turn; every segment has its own seeded points, which is what
its host plan depends on.

Per shape, the device counts alternate within each of --reps rounds and medians are reported; one untimed call per count
first creates the cached renderers. Besides the end-to-end time of api.morph_segments, a second pass over the same
renderers splits a call into its parts: host planning (every segment's SequencePlan, as the call plans them before
rendering), rendering (segment uploads and render_segments up to a device sync, on the slowest device) and downloads into
host memory (on the slowest device)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from poppy_b200 import api, host, shard, synth  # noqa: E402
from poppy_b200.renderer import device_count  # noqa: E402

LEVELS = 64


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out or ["unknown"]
    except Exception as e:
        return [f"unknown ({e})"]


def synthetic_segments(K, w, h, pairs=8):
    images = [(synth.noise_image(w, h, 100 + i), synth.noise_image(w, h, 101 + i)) for i in range(min(K, pairs))]
    segs = []
    for i in range(K):
        p1, p2 = synth.matched_points(w, h, 400, 8.0, 103 + i)
        segs.append((images[i % pairs][0], images[i % pairs][1], None, p1, p2))
    return segs


def parts(segs, n_frames, devices):
    """(planning, slowest device's rendering, slowest device's downloads) in seconds: the steps of api.morph_segments."""
    K = len(segs)
    h, w = segs[0][0].shape[:2]
    t0 = time.perf_counter()
    ratio = np.array([host.chain_ratio(j, n_frames) for j in range(n_frames)], np.float64)
    shape = ratio.astype(np.float32)
    plans = [host.SequencePlan(p1, p2, w, h, shape, chain=True) for _, _, _, p1, p2 in segs]
    t_plan = time.perf_counter() - t0
    n_max, tri_max = max(p.n for p in plans), max(p.max_triangles for p in plans)
    G = min(len(devices), K)
    out = np.empty((K, n_frames, h, w, 3), np.uint8)
    render, download = [0.0] * G, [0.0] * G

    def run(g):
        lo, hi = shard.phase_range(g, G, K)
        per_batch = max(1, min(hi - lo, api._SEGMENT_RING_BYTES // (n_frames * w * h * 3)))
        d = devices[g]
        r = api._renderer(w, h, n_max, tri_max, per_batch * n_frames) if d == api.Settings.instance().cuda_device \
            else api._device_renderer(d, w, h, n_max, tri_max, per_batch * n_frames)
        for b0 in range(lo, hi, per_batch):
            batch = range(b0, min(hi, b0 + per_batch))
            t = time.perf_counter()
            r.set_segments(len(batch), n_frames)
            for i, s in enumerate(batch):
                c1, c2, _, p1, p2 = segs[s]
                r.set_segment(i, c1, c2, None, p1, p2)
            tri, offs = api.interleave_segment_plans([plans[s] for s in batch], n_frames)
            r.render_segments(0, shape, ratio, tri, offs)
            r.sync()
            render[g] += time.perf_counter() - t
            t = time.perf_counter()
            r.download(0, len(batch) * n_frames, out=out[b0:b0 + len(batch)].reshape(-1, h, w, 3))
            download[g] += time.perf_counter() - t
    threads = [threading.Thread(target=run, args=(g,)) for g in range(G)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for p in plans:
        p.close()
    return t_plan, max(render), max(download)


def measure(w, h, n_frames, Ks, counts, reps):
    rows = []
    segs_all = synthetic_segments(max(Ks), w, h)
    for K in Ks:
        segs = segs_all[:K]
        for G in counts:                                     # creates and sizes every renderer the timed calls use
            api.morph_segments(segs, number_of_frames=n_frames, devices=list(range(G)))
        e2e = {G: [] for G in counts}
        split = {G: [] for G in counts}
        for _ in range(reps):
            for G in counts:
                t = time.perf_counter()
                api.morph_segments(segs, number_of_frames=n_frames, devices=list(range(G)))
                e2e[G].append(time.perf_counter() - t)
                split[G].append(parts(segs, n_frames, list(range(G))))
        frames = K * n_frames
        for G in counts:
            s = statistics.median(e2e[G])
            rows.append({"K": K, "gpus": G, "frames": frames, "e2e_s": round(s, 4), "e2e_frames_per_s": round(frames / s, 1),
                         "plan_s": round(statistics.median(p[0] for p in split[G]), 4),
                         "render_s_slowest_gpu": round(statistics.median(p[1] for p in split[G]), 4),
                         "download_s_slowest_gpu": round(statistics.median(p[2] for p in split[G]), 4)})
            base = next(r for r in rows if r["K"] == K and r["gpus"] == counts[0])
            rows[-1]["speedup_vs_1"] = round(rows[-1]["e2e_frames_per_s"] / base["e2e_frames_per_s"], 2)
        api.release()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "segments_devices_timing_b200.json"))
    args = ap.parse_args()
    n = device_count()
    if n < 1:
        raise SystemExit("segments_devices_timing: no CUDA device")
    counts = [G for G in (1, 2, 4, 8) if G <= n]
    api.Settings.instance().pyramid_levels = LEVELS
    res = {"gpus": gpu_info(), "gpus_on_box": n, "host_cpus": os.cpu_count(), "reps": args.reps, "levels": LEVELS}
    res["1920x1080_N120"] = measure(1920, 1080, 120, [8, 16, 32], counts, args.reps)
    res["3840x2160_N60"] = measure(3840, 2160, 60, [8, 16], counts, args.reps)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
