#!/usr/bin/env python
"""Benchmark of the morph-render hot path (BASELINE.json metric: morphed frames/sec; HBM GB/s vs peak).

    python bench.py --gpus N --steps K --warmup W            # the CUDA path, one process per GPU (torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU morph_images on host cores

A *step* is one pass of the hot path over one batch of synthetic input: `--frames` independent frame phases
(direct mode) of the named workload, rendered into the HBM frame ring with the image pair, the point sets and the
per-frame triangle lists prepared beforehand. Default workload: BASELINE.json configs[3] — synthetic 3840x2160
pair, 20k matched points (~40k triangles), 6-level pyramid; 600 phases per step and rank.

    python bench.py --workload 1080p|4k|8k                     # the other points of the metric (default 4k = configs[3])
    python bench.py --workload 8k --total-frames 2400 --gpus N   # configs[4]: 2,400 8K phases sharded over N ranks (strong scaling)
    python bench.py --mode chain                                # configs[0]: the reference demo pair, 60 chained frames, 64 levels
    python bench.py --dump-outputs DIR                          # + a fixed sample of the last timed step's outputs, DIR/*.npy

JSON line (rank 0):
  value       whole-job frames/s with inputs resident in HBM, device time (CUDA events on the context's stream),
              max over ranks
  e2e         frames/s through the public API call (poppy_b200.api.render_phases semantics: host topology planning
              on host threads + H2D of the pair from pinned memory + render + D2H of every frame to pinned memory)
  roofline    whole-path algorithmic bytes (SURVEY.md section 8(d): 23 B x P0 + 132 B x sum P1..P(L-1) + 104 B x PL
              per frame) x frames/s against the measured HBM copy peak, plus the per-kernel-class time shares
  cpu_baseline  the reference library (oracle/_ref, unmodified reference code) timed on a bounded sample of the same
              workload on the host cores of rank 0, with the parity of those frames against the GPU frames
"""
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


# ------------------------------------------------------------------------------------------------------------------
def algorithmic_bytes_per_frame(w: int, h: int, levels: int) -> int:
    """SURVEY.md section 8(d) / BASELINE.md section 3."""
    px = []
    lw, lh = w, h
    for _ in range(levels + 1):
        px.append(lw * lh)
        lw, lh = (lw + 1) // 2, (lh + 1) // 2
    return 23 * px[0] + 132 * sum(px[1:levels]) + 104 * px[levels]


def ncu_traffic():
    """DRAM bytes per frame of every kernel class from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_summary.py traffic): dram__bytes_read.sum + dram__bytes_write.sum."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(path))
    except Exception:
        return None


def dominant_kernel_roofline(kern, W, H, F, chunk_frames, peak, traffic, levels=6):
    """roofline of the kernel class with the largest share of the step: algorithmic bytes of that stage per launch
    (DESIGN.md section 5) / its CUDA-event launch time measured in this run. A class made of several per-level launches
    is rated over the launch sequence of one chunk."""
    if not kern:
        return None
    P, lw, lh = [], W, H
    for _ in range(levels + 1):
        P.append(lw * lh)
        lw, lh = (lw + 1) // 2, (lh + 1) // 2
    px, mid = P[0], sum(P[1:levels])
    # compulsory bytes per frame of each kernel class as designed: every input read once, every output written once
    alg = {
        "raster_warp": 8 * px + 8 * px / max(chunk_frames, 1),     # warped pair written; both sources read once per chunk
        "unsharp_store": 15 * px,                                   # lapBlend 32FC3 read, 8UC3 frame written
        # level 0: warped pair 8 + mask 4 + coarse (24 + 12)/4 read, out 12 written; level k: 28 + 9 read, 12 written;
        # coarsest: 28 read, 12 written
        "blend_collapse": 33 * px + 49 * mid + 40 * P[levels],
        # level 0->1: warped 8 + basis 4 read, mask0 4 + 7 planes/4 written; level k->k+1: 28 read, 7 written
        "pyr_down": 23 * px + 35 * mid,
    }
    k = kern[0]
    name = k["kernel"]
    chunks = max(1, -(-F // max(chunk_frames, 1)))
    launches_per_chunk = max(1, round(k["launches_per_step"] / chunks))
    out = {"kernel": name, "share_of_step": k["share"], "launches_per_chunk": launches_per_chunk,
           "us_per_launch": k["us_per_launch"] * launches_per_chunk}
    if launches_per_chunk > 1:
        out["note"] = f"{launches_per_chunk} launches of one chunk rated together"
    if name in alg:
        b = alg[name] * F
        ach = b / (k["ms_per_step"] * 1e-3) / 1e9
        out.update({"algorithmic_bytes_per_launch": int(alg[name] * min(F, chunk_frames)), "achieved": ach, "peak": peak,
                    "unit": "GB/s", "frac": ach / peak})
    if traffic and name in traffic.get("bytes_per_frame", {}):
        out["traffic"] = int(traffic["bytes_per_frame"][name] * min(F, chunk_frames))
        out["traffic_source"] = traffic.get("source")
    return out


def issue_roofline(traffic, fps_per_gpu, clocks, sms=148, slots_per_sm=4):
    """The other roofline of this path: warp instructions per frame (ncu smsp__inst_executed.sum of every kernel,
    profiles/ncu_traffic.json) against the issue slots of the GPU at the SM clock sampled during the run."""
    if not traffic or "warp_instructions_per_frame" not in traffic:
        return None
    wi = float(sum(traffic["warp_instructions_per_frame"].values()))
    mhz = float((clocks or {}).get("sm_mhz") or 1965.0)
    peak = sms * slots_per_sm * mhz * 1e6
    return {"warp_instructions_per_frame": int(wi), "peak_warp_instructions_per_s": peak,
            "roofline_frames_per_s": peak / wi, "frac": fps_per_gpu * wi / peak}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def mirror_tile(img: np.ndarray, w: int, h: int) -> np.ndarray:
    """img repeated with alternating mirror images (no seams) up to h x w."""
    ih, iw = img.shape[:2]
    row = np.concatenate([img, img[:, ::-1]], axis=1)
    cell = np.concatenate([row, row[::-1]], axis=0)
    reps = (-(-h // (2 * ih)), -(-w // (2 * iw))) + (1,) * (img.ndim - 2)
    return np.ascontiguousarray(np.tile(cell, reps)[:h, :w])


# ------------------------------------------------------------------------------------------------------------------
class Job:
    """The workload of one rank: inputs, frame schedule, and the config dict both arms print."""

    def __init__(self, args, rank, world):
        from poppy_b200 import synth, shard, host
        self.mode = args.mode
        self.chain = args.mode == "chain"
        if self.chain:
            # BASELINE.json configs[0]: images/square.png -> images/circle.png through the reference front end (blur_margin,
            # extractor, matcher, gabor_filter): what it handed to morph_images() is the committed fixture
            g = np.load(os.path.join(ROOT, "tests", "golden", "full", "c1.npz"))
            self.W, self.H, self.L = int(g["width"]), int(g["height"]), int(g["levels"])
            self.bgr1, self.bgr2, self.gabor2 = g["corrected1"], g["corrected2"], g["gabor2"]
            self.pts1, self.pts2 = g["pts1"], g["pts2"]
            self.F = int(g["n_frames"])
            self.total = self.F * world                      # replicas: a chain does not shard (SURVEY.md 8(e))
            ratio = np.array([host.chain_ratio(j, self.F) for j in range(self.F)], np.float64)
            self.phases, self.masks = ratio.astype(np.float32), ratio
            self.hashes = g["hashes"]
            self.name = "config1-chain"
            self.data = "reference demo images"
            self.desc = (f"images/square.png -> images/circle.png (reference front end), {self.W}x{self.H}, {len(self.pts1)} matcher "
                         f"points, {self.F} chained frames, {self.L}-level pyramid (BASELINE.json configs[0])")
            self.scaling = "weak"
            self.parallelism = f"chain replicas x{world} (a chain is a recurrence: it does not shard), no collective"
        else:
            wl = dict(synth.WORKLOADS[args.workload])
            self.W, self.H, self.L = wl["w"], wl["h"], wl["levels"]
            inp = synth.make_inputs(self.W, self.H, wl["n_points"], wl["jitter"], wl["seed"])
            self.bgr1, self.bgr2, self.gabor2, self.pts1, self.pts2 = inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2
            content = "synthetic (band-limited noise, full 8-bit range)"
            if args.content == "photo":
                # secondary line: the same geometry over photographic content - the reference's own demo pair
                # (tests/golden/full/c1.npz: images/square.png, images/circle.png after its front end) mirror-tiled to size
                g = np.load(os.path.join(ROOT, "tests", "golden", "full", "c1.npz"))
                self.bgr1, self.bgr2, self.gabor2 = (mirror_tile(g[k], self.W, self.H) for k in ("corrected1", "corrected2", "gabor2"))
                content = "the reference's demo pair (config 1 fixture) mirror-tiled"
            self.data = "synthetic" if args.content == "synthetic" else "reference demo images, tiled; synthetic points"
            if args.total_frames:
                self.total = args.total_frames
                self.scaling = "strong"
            else:
                per_rank = args.frames or (300 if args.workload == "8k" else wl["frames"])
                self.total = per_rank * world
                self.scaling = "weak"
            sched = shard.phase_schedule(self.total)
            lo, hi = shard.phase_range(rank, world, self.total)
            self.phases = np.ascontiguousarray(sched[lo:hi])
            self.masks = self.phases.astype(np.float64)
            self.F = hi - lo
            self.name = args.workload
            cfg = {"1080p": "the 1080p point of the metric", "4k": "BASELINE.json configs[3]", "8k": "BASELINE.json configs[4]"}[args.workload]
            self.desc = (f"synthetic {self.W}x{self.H} BGR pair, {wl['n_points']}+4 matched points, {self.L}-level pyramid, "
                         if args.content == "synthetic" else
                         f"{self.W}x{self.H} BGR pair = {content}, {wl['n_points']}+4 synthetic matched points, {self.L}-level pyramid, ")
            self.desc += f"{self.total} independent phases over {world} rank(s) ({cfg})"
            self.parallelism = f"phase-sharded x{world}, no collective"
        self.frame_bytes = self.W * self.H * 3
        # frames resident in the HBM ring at once: the whole shard where it fits (8K: 300-frame slices, 30 GB)
        cap = args.ring or (300 if self.W * self.H > 3840 * 2160 else 1 << 30)
        self.ring = max(1, min(self.F, cap))
        self.slices = [(a, min(a + self.ring, self.F)) for a in range(0, self.F, self.ring)]

    def config(self):
        return {"workload": self.desc,
                "mode": "chain (frame j sources frame j-1, reference src/poppy.hpp:177-243)" if self.chain
                        else "direct (independent phases, reference '-f 1 -p s')",
                "total_frames_per_step": self.total, "parallelism": self.parallelism,
                "l2_policy": "inputs larger than L2: every frame streams its scratch (>1 GB at 4K) through HBM; consecutive frames "
                             "write different ring slots",
                "timing": "CUDA events on the renderer's stream, max over ranks"}


DUMP_FRAMES, DUMP_PIXELS = 8, 1 << 19     # 8 frames x 2^19 pixels x 3 channels x 4 bytes = 48 MiB


def dump_outputs(out_dir, r, job):
    """What the last timed step handed back, as float32 .npy files in out_dir: the frames still resident in the ring (the
    step's last ring slice) and their morphed points. A 4K frame alone is 100 MB in float32, so the files hold a fixed
    sample: up to DUMP_FRAMES frames spread evenly over the slice, and in each the same seeded set of at most DUMP_PIXELS
    pixel positions. Inputs and sample depend on the arguments only, so two builds can be compared file for file."""
    a, b = job.slices[-1]
    ks = np.unique(np.linspace(0, b - a - 1, min(b - a, DUMP_FRAMES)).round().astype(int))
    px = job.W * job.H
    sel = np.sort(np.random.default_rng(0).choice(px, DUMP_PIXELS, replace=False)) if px > DUMP_PIXELS else slice(None)
    frames = np.stack([r.download(int(k), 1)[0].reshape(px, 3)[sel] for k in ks]).astype(np.float32)
    points = np.stack([r.morphed_points(int(k)) for k in ks]).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frames.npy"), frames)                  # (frames, pixels, BGR) values 0..255
    np.save(os.path.join(out_dir, "morphed_points.npy"), points)          # (frames, points, xy)


def _kproc_worker(q, path, w, h, levels, phases):
    """One process of the K-process CPU baseline: the reference library on one OpenCV thread."""
    try:
        sys.path.insert(0, ROOT)
        from oracle import ref
        d = np.load(path)
        ref.set_threads(1)
        ref.morph_images(d["bgr1"], d["bgr2"], d["gabor2"], d["pts1"], d["pts2"], 0.5, 0.5, levels)      # warm-up
        t0 = time.perf_counter()
        for s in phases:
            ref.morph_images(d["bgr1"], d["bgr2"], d["gabor2"], d["pts1"], d["pts2"], float(s), float(s), levels)
        q.put((len(phases), time.perf_counter() - t0))
    except Exception as e:          # pragma: no cover
        q.put((0, repr(e)))


def kprocess_baseline(job, procs, frames_per_proc=1):
    """Best case of the reference on the box (BASELINE.md 4.3): K independent single-threaded processes over disjoint
    phases. Returns frames/s over the slowest process."""
    import multiprocessing as mp
    import tempfile
    ctx = mp.get_context("spawn")
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "inputs.npz")
        np.savez(path, bgr1=job.bgr1, bgr2=job.bgr2, gabor2=job.gabor2, pts1=job.pts1, pts2=job.pts2)
        q = ctx.Queue()
        ps = []
        for i in range(procs):
            ph = [float(job.phases[(7 + 13 * (i * frames_per_proc + j)) % job.F]) for j in range(frames_per_proc)]
            ps.append(ctx.Process(target=_kproc_worker, args=(q, path, job.W, job.H, job.L, ph)))
        for pr in ps:
            pr.start()
        res = [q.get(timeout=900) for _ in ps]
        for pr in ps:
            pr.join()
    if any(n == 0 for n, _ in res):
        return {"error": str([t for n, t in res if n == 0][:1])}
    slowest = max(t for _, t in res)
    return {"value": sum(n for n, _ in res) / slowest, "unit": "frames/s", "processes": procs, "threads_per_process": 1,
            "sample": f"{frames_per_proc} frame(s) per process after one warm-up frame; rate = all frames / slowest process"}


def reference_arm(args, rank, world):
    """The reference's own CPU implementation of the path (oracle/_ref/libpoppy_ref.so = unmodified reference
    sources + vendored OpenCV 4.6.0), all host threads; each step is a bounded sample of the workload."""
    if rank != 0:
        return
    from oracle import ref
    if not ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libpoppy_ref.so not built"}))
        return
    job = Job(args, 0, world)
    total = args.warmup + args.steps
    times = []
    if job.chain:
        per_step = job.F
        for i in range(total):
            t0 = time.perf_counter()
            ref.chain(job.bgr1, job.bgr2, job.gabor2, job.pts1, job.pts2, job.F, job.L)
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
        sample = f"the whole {job.F}-frame chain per step, {len(times)} steps after {args.warmup} warm-up"
    else:
        per_step = 1
        picks = [int(round(i * (job.F - 1) / max(total - 1, 1))) for i in range(total)]
        for i, k in enumerate(picks):
            s = float(job.phases[k])
            t0 = time.perf_counter()
            ref.morph_images(job.bgr1, job.bgr2, job.gabor2, job.pts1, job.pts2, s, s, job.L)
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
        sample = f"{len(times)} frames of the workload (phases spread over [0,1]), 1 frame per step, after {args.warmup} warm-up frames"
    fps = per_step * len(times) / sum(times)
    cores = ref.get_threads()
    out = {
        "impl": "reference", "metric": "morphed frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sum(times) / len(times),
        "higher_is_better": True, "scaling": job.scaling, "vs_baseline": None, "dtype": "u8/f32", "data": job.data,
        "config": job.config(),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.kprocs and not job.chain:
        out["cpu_baseline"]["k_process"] = kprocess_baseline(job, args.kprocs)
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--mode", default="direct", choices=["direct", "chain"])
    ap.add_argument("--workload", default="4k", choices=["1080p", "4k", "8k"])
    ap.add_argument("--content", default="synthetic", choices=["synthetic", "photo"],
                    help="pixel content of the pair: the synthetic texture (headline) or the reference's demo pair tiled to size")
    ap.add_argument("--frames", type=int, default=0, help="frame phases per step and rank (weak scaling; default: workload's)")
    ap.add_argument("--total-frames", type=int, default=0, help="frame phases per step over ALL ranks (strong scaling)")
    ap.add_argument("--ring", type=int, default=0, help="frames resident in the HBM ring (default: the shard, 300 at 8K)")
    ap.add_argument("--chunk", type=int, default=0, help="frames per kernel batch (0 = library default)")
    ap.add_argument("--unsharp-mode", type=int, default=0, choices=[0, 1, 2], help="0 adaptive, 1 dense, 2 calm route")
    ap.add_argument("--cpu-frames", type=int, default=4, help="reference frames timed for cpu_baseline (0 = skip)")
    ap.add_argument("--kprocs", type=int, default=-1, help="processes of the K-process CPU baseline (-1: one per core up to 16, 0: skip)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-slice", type=int, default=64, help="frames per planned/rendered/downloaded slice of the e2e pipeline")
    ap.add_argument("--no-stage-pass", action="store_true",
                    help="profiling runs (under ncu): skip the per-kernel-class timing pass and the e2e leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write a fixed sample of the frames and morphed points of the last timed step (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA path; the reference arm does not dump")
    if args.kprocs < 0:
        args.kprocs = min(os.cpu_count() or 1, 16) if args.cpu_frames > 0 and args.mode == "direct" and args.workload != "8k" else 0

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from poppy_b200 import build, host, shard
    from poppy_b200.renderer import MorphRenderer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the morph renderer has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()           # the other ranks load the library only after rank 0 has (re)built it

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs (identical on every rank), this rank's frames, host topology plan -------------------------------
    job = Job(args, rank, world)
    F, W, H, L = job.F, job.W, job.H, job.L
    phases, masks = job.phases, job.masks
    ncores = os.cpu_count() or 1
    plan_threads = max(1, ncores // world)
    t0 = time.perf_counter()
    plan = host.SequencePlan(job.pts1, job.pts2, W, H, phases, chain=job.chain, threads=plan_threads)
    plan_s = time.perf_counter() - t0

    r = MorphRenderer(W, H, L, len(job.pts1), plan.max_triangles, job.ring, device=local_rank,
                      chunk_frames=args.chunk or None)
    r.set_unsharp_mode(args.unsharp_mode)
    # pinned host copies of the pair (source of the e2e H2D)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_bgr1, h_bgr2, h_gab = pin(job.bgr1), pin(job.bgr2), pin(job.gabor2)
    r.set_pair(h_bgr1.numpy(), h_bgr2.numpy(), h_gab.numpy())
    r.set_points(job.pts1, job.pts2)
    stream = torch.cuda.ExternalStream(r.stream(), device=torch.device("cuda", local_rank))
    # per ring slice: schedule + triangle lists rebased to the slice
    offs = plan.tri_offsets
    slice_args = [(phases[a:b], masks[a:b], plan.tri_idx[offs[a]:offs[b]], np.ascontiguousarray(offs[a:b + 1] - offs[a]))
                  for a, b in job.slices]

    # `value` is measured with its inputs resident in HBM: the pair, the points and the plan's triangle lists (validated and
    # uploaded once here; the e2e leg below plans, validates and uploads them inside its timed region)
    r.set_plan(plan.tri_idx, plan.tri_offsets)

    def step(checksums=None):
        for (a, b), (ph, mk, ti, to) in zip(job.slices, slice_args):
            r.render_planned(ph, mk, plan_first=a, chain=job.chain)
            if checksums is not None:
                checksums.append(r.checksum(0, len(ph)))

    for _ in range(args.warmup):
        step()
    r.sync()
    r.unsharp_stats()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = r.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    e1.synchronize()
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = r.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r, job)
    exact_chunks, all_chunks = r.unsharp_stats()
    sums = []
    if len(job.slices) > 1:
        step(sums)                 # frames of earlier slices are gone from the ring: checksum every slice as it is rendered
    else:
        sums.append(r.checksum(0, F))
    checksum = shard.combine_checksums(sums) if len(sums) > 1 else sums[0]

    # ---- per-kernel-class shares: one more step with CUDA-event stage timing -------------------------------------
    stage, stage_total_ms = {}, None
    if not args.no_stage_pass:
        r._check(r._lib.poppy_cuda_set_stage_timing(r._ctx, 1))
        acc = {}
        stage_total_ms = 0.0
        for ph, mk, ti, to in slice_args:
            r.render(ph, mk, ti, to, chain=job.chain)
            for k, v in r.stage_times().items():
                a = acc.setdefault(k, {"ms": 0.0, "launches": 0})
                a["ms"] += v["ms"]; a["launches"] += v["launches"]
            stage_total_ms += r.last_render_ms()
        stage = acc
        r._check(r._lib.poppy_cuda_set_stage_timing(r._ctx, 0))

    # ---- e2e: the public-API path with host buffers --------------------------------------------------------------
    ring_frames = job.ring
    host_ring = min(ring_frames, max(64, args.e2e_slice))      # pinned host ring: at least one slice
    h_ring = torch.empty((host_ring, H, W, 3), dtype=torch.uint8).pin_memory()
    frame_bytes = job.frame_bytes
    e2e_times, e2e_parts = [], None
    barrier()
    # The sequence streams through the renderer slice by slice: a planner thread triangulates slice k+1 on the host
    # cores while slice k renders and slice k-1 is copied to pinned memory (copy stream) - the reference's frame loop
    # (src/poppy.hpp:172-243) with its three stages overlapped instead of run back to back. A chain is one slice: its
    # point recurrence is planned ahead of the render, its frames leave in order afterwards.
    import queue
    slice_frames = F if job.chain else max(1, min(F, args.e2e_slice, ring_frames))
    slices = [(a, min(a + slice_frames, F)) for a in range(0, F, slice_frames)]
    for it in range(0 if args.no_stage_pass or args.e2e_steps <= 0 else args.e2e_steps + 1):
        plans = queue.Queue(maxsize=3)
        plan_busy = [0.0]

        def planner():
            for a, b in slices:
                t0 = time.perf_counter()
                p = host.SequencePlan(job.pts1, job.pts2, W, H, phases[a:b], chain=job.chain, threads=plan_threads, copy=False)
                plan_busy[0] += time.perf_counter() - t0
                plans.put((a, b, p))

        t_a = time.perf_counter()
        th = threading.Thread(target=planner, daemon=True)
        th.start()
        r.set_pair(h_bgr1.numpy(), h_bgr2.numpy(), h_gab.numpy())
        r.set_points(job.pts1, job.pts2)
        t_c = time.perf_counter()
        dev_slot = 0
        for _ in slices:
            a, b, p = plans.get()
            n = b - a
            if dev_slot + n > ring_frames:
                dev_slot = 0
            r.render(phases[a:b], masks[a:b], p.tri_idx, p.tri_offsets, chain=job.chain, first_slot=dev_slot)
            # frames leave through the pinned host ring in pieces of at most its size
            for c0 in range(0, n, host_ring):
                cn = min(host_ring, n - c0)
                r.download_async(dev_slot + c0, cn, h_ring.data_ptr(), W * 3, frame_bytes)
            dev_slot += n
            p.close()
        r.sync()
        t_d = time.perf_counter()
        th.join()
        if it > 0:        # first pass is warm-up
            e2e_times.append(t_d - t_a)
            e2e_parts = {"total_s": t_d - t_a, "h2d_s": t_c - t_a, "planner_busy_s": plan_busy[0], "plan_threads": plan_threads,
                         "planner_frames_per_s_per_core": F / max(plan_busy[0], 1e-9) / plan_threads,
                         "slice_frames": slice_frames, "slices": len(slices)}
    e2e_s = statistics.median(e2e_times) if e2e_times else float("inf")

    # ---- the drop-in call itself: one morph_images() per frame, exactly the reference's signature and calling pattern
    # (src/poppy.hpp:215: images, points and ratios in, dst and morphedPoints out; every call uploads the pair,
    # triangulates on ONE host thread, renders one frame and downloads it)
    single_call = None
    if rank == 0 and world == 1 and not args.no_stage_pass and args.e2e_steps > 0 and not job.chain:
        from poppy_b200 import api
        api.Settings.instance().pyramid_levels = L
        ts = []
        for k in range(min(8, F)):
            sk = float(phases[(F // 3 + k) % F])          # consecutive frames of the sequence, as the reference's loop calls it
            t0 = time.perf_counter()
            api.morph_images(job.bgr1, job.bgr2, job.bgr1, job.bgr2, job.gabor2, job.pts1, job.pts2, sk, sk)
            ts.append(time.perf_counter() - t0)
        api.release()
        single_call = {"value": 1.0 / statistics.median(ts[1:]), "unit": "frames/s",
                       "what": "poppy_b200.api.morph_images() called once per frame on consecutive frames (pair staged once, "
                               "single-thread Delaunay predicted by the previous call's walks + render + D2H per call), the "
                               "reference's own calling pattern"}
    h2d_bytes = job.bgr1.nbytes + job.bgr2.nbytes + job.gabor2.nbytes + job.pts1.nbytes + job.pts2.nbytes + \
        plan.tri_idx.nbytes + plan.tri_offsets.nbytes + phases.nbytes + masks.nbytes
    d2h_bytes = F * frame_bytes

    # ---- reduce over ranks ---------------------------------------------------------------------------------------
    frames_all = F
    rank_ms = [dev_ms / args.steps]
    if world > 1:
        per_rank = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(per_rank, torch.tensor([dev_ms / args.steps], dtype=torch.float64, device="cuda"))
        rank_ms = [float(v[0]) for v in per_rank]
        t = torch.tensor([dev_ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_s = float(t[0]), float(t[1])
        l = torch.tensor([launches, F, exact_chunks, all_chunks], dtype=torch.int64, device="cuda")
        dist.all_reduce(l, op=dist.ReduceOp.SUM)
        launches, frames_all, exact_chunks, all_chunks = (int(v) for v in l)
        gsums = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(gsums, torch.tensor([checksum & 0x7FFFFFFFFFFFFFFF], dtype=torch.int64, device="cuda"))
        checksum_all = shard.combine_checksums([int(v[0]) for v in gsums])
    else:
        checksum_all = shard.combine_checksums([checksum & 0x7FFFFFFFFFFFFFFF])

    if rank == 0:
        total_frames = frames_all * args.steps
        fps = total_frames / (dev_ms / 1000.0)
        alg = algorithmic_bytes_per_frame(W, H, L)
        peak, peak_src = measured_peaks()
        traffic = ncu_traffic() if (W, H, L) == (3840, 2160, 6) else None      # the committed capture is of configs[3]
        chunk_used = args.chunk or min(32, job.ring)
        if job.chain:
            chunk_used = 1
        achieved = alg * (fps / world) / 1e9            # per GPU
        kern = []
        tot = sum(v["ms"] for v in stage.values()) or 1.0
        for name, v in sorted(stage.items(), key=lambda kv: -kv[1]["ms"]):
            if v["launches"]:
                kern.append({"kernel": name, "ms_per_step": round(v["ms"], 3), "share": round(v["ms"] / tot, 4),
                             "launches_per_step": v["launches"], "us_per_launch": round(1000 * v["ms"] / v["launches"], 2)})
        out = {
            "metric": "morphed frames/sec", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "ms_per_step_by_rank": [round(v, 2) for v in rank_ms],
            "higher_is_better": True, "scaling": job.scaling,
            "vs_baseline": None, "dtype": "u8/f32", "data": job.data,
            "config": job.config(),
            "e2e": {"value": frames_all / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": int(d2h_bytes), "breakdown": e2e_parts, "single_call": single_call,
                    "what": "H2D pair/points + per slice: host Delaunay planning (threads), H2D triangles, render, D2H of every frame to "
                            "pinned memory; the three stages of consecutive slices overlap"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (int(sum(traffic["bytes_per_frame"].values()) * F) if traffic else None),
                         "traffic_what": "ncu dram__bytes_read+write of all kernels of one step (profiles/ncu_traffic.json)",
                         "dominant_kernel": dominant_kernel_roofline(kern, W, H, F, chunk_used, peak, traffic, L),
                         "issue": issue_roofline(traffic, fps / world, clocks),
                         "peak_source": peak_src,
                         "scope": "whole render path per GPU (SURVEY.md 8(d) algorithmic bytes/frame x frames/s)",
                         "algorithmic_bytes_per_frame": alg, "kernels": kern,
                         "stage_timed_step_ms": stage_total_ms},
            "clocks": clocks,
            "unsharp": {"mode": ["adaptive", "dense", "calm"][args.unsharp_mode],
                        "exact_chunk_share": (exact_chunks / all_chunks) if all_chunks else None,
                        "what": "share of 120x24-pixel strip chunks of the timed frames that ran the exact GaussianBlur + medianBlur "
                                "path of unsharp_mask(); the rest is provably untouched by it (see DESIGN.md)"},
            "host_plan": {"seconds": plan_s, "threads": plan_threads, "frames_per_s": F / plan_s,
                          "frames_per_s_per_core": F / plan_s / plan_threads},
            "frames_checksum": f"{checksum_all:016x}",
        }
        # ---- CPU baseline + parity on the sampled frames (rank 0, N=1 only) --------------------------------------
        if world == 1 and args.cpu_frames > 0:
            from oracle import ref
            if not ref.available():
                out["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference",
                                       "sample": "oracle/_ref not built"}
            elif job.chain:
                t0 = time.perf_counter()
                want, _ = ref.chain(job.bgr1, job.bgr2, job.gabor2, job.pts1, job.pts2, F, L)
                dt = time.perf_counter() - t0
                got = r.download(0, F)
                d = np.abs(got.astype(np.int16) - np.asarray(want).astype(np.int16))
                out["cpu_baseline"] = {"value": F / dt, "unit": "frames/s", "cores": ref.get_threads(), "kind": "reference",
                                       "sample": f"the whole {F}-frame chain, unmodified reference frame recurrence on all host threads"}
                out["parity_vs_reference"] = {"frames": F, "differing_bytes": int((d != 0).sum()), "max_abs": int(d.max()),
                                              "min_fraction_within_1": float((d <= 1).mean())}
            else:
                last_a, last_b = job.slices[-1]                   # frames still resident in the ring
                idx = [last_a + int(round(i * (last_b - last_a - 1) / max(args.cpu_frames - 1, 1))) for i in range(args.cpu_frames)]
                ref.morph_images(job.bgr1, job.bgr2, job.gabor2, job.pts1, job.pts2, 0.5, 0.5, L)   # warm-up
                times, worst, diff_bytes, within1 = [], 0, 0, 1.0
                for k in idx:
                    s_ = float(phases[k])
                    t0 = time.perf_counter()
                    want, _ = ref.morph_images(job.bgr1, job.bgr2, job.gabor2, job.pts1, job.pts2, s_, s_, L)
                    times.append(time.perf_counter() - t0)
                    got = r.download(k - last_a, 1)[0]
                    d = np.abs(got.astype(np.int16) - want.astype(np.int16))
                    worst = max(worst, int(d.max())); diff_bytes += int((d != 0).sum())
                    within1 = min(within1, float((d <= 1).mean()))
                out["cpu_baseline"] = {"value": len(times) / sum(times), "unit": "frames/s", "cores": ref.get_threads(),
                                       "kind": "reference",
                                       "sample": f"{len(times)} frames of the same workload (phases {[round(float(phases[k]), 3) for k in idx]}), "
                                                 "unmodified reference morph_images() on all host threads"}
                out["parity_vs_reference"] = {"frames": len(idx), "differing_bytes": diff_bytes, "max_abs": worst,
                                              "min_fraction_within_1": within1}
                # how much of the frame takes the median / sharpen branch of the dense unsharp kernel (its speed is data
                # dependent): from the reference's own lapBlend of one sampled frame, x - GaussianBlur(x, sigma 1) against the
                # kernel's group test (a 4-pixel group is flagged when any |diff| >= 0.17; a group runs the exact median when a
                # flagged group touches its 3x3 windows)
                try:
                    kmid = min(idx, key=lambda k: abs(float(phases[k]) - 0.5))        # the sampled frame nearest mid-morph
                    st = ref.stages(job.bgr1, job.bgr2, job.gabor2, job.pts1, job.pts2, float(phases[kmid]), float(phases[kmid]), L)
                    dmag = np.abs(st.lap_blend - ref.gaussian_blur(st.lap_blend, 1.0)).max(axis=2)
                    wg = (W // 4) * 4
                    grp = (dmag[:, :wg].reshape(H, wg // 4, 4) >= 0.17).any(axis=2)
                    near = grp.copy()
                    near[:, 1:] |= grp[:, :-1]; near[:, :-1] |= grp[:, 1:]
                    med = near.copy()
                    med[1:] |= near[:-1]; med[:-1] |= near[1:]
                    out["unsharp"]["dense_kernel_branching"] = {
                        "frame_phase": round(float(phases[kmid]), 3),
                        "pixels_over_0.17": float((dmag >= 0.17).mean()), "groups_flagged": float(grp.mean()),
                        "groups_running_the_median": float(med.mean()),
                        "pixels_sharpened": float((st.dst != np.clip(np.rint(st.lap_blend * 255.0), 0, 255).astype(np.uint8)).any(axis=2).mean())}
                except Exception as e:      # diagnostics only
                    out["unsharp"]["dense_kernel_branching"] = {"error": str(e)[:200]}
                if args.kprocs:
                    r.close()               # give the host memory back before K processes load the pair
                    out["cpu_baseline"]["k_process"] = kprocess_baseline(job, args.kprocs)
        print(json.dumps(out))
    r.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
