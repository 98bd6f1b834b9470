#!/usr/bin/env python
"""Host planning throughput (Delaunay per frame) for a thread count. usage: plan_timing.py frames threads"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from poppy_b200 import host, shard, synth
F = int(sys.argv[1]); thr = int(sys.argv[2])
c = synth.WORKLOADS["4k"]; inp = synth.make_inputs(c["w"], c["h"], c["n_points"], c["jitter"], c["seed"])
ph = np.ascontiguousarray(shard.phase_schedule(600))[:F]
best = 1e9
for _ in range(2):
    t = time.perf_counter(); p = host.SequencePlan(inp.pts1, inp.pts2, c["w"], c["h"], ph, threads=thr); dt = time.perf_counter() - t; p.close()
    best = min(best, dt)
print(f"threads={thr} frames={F}: {best:.3f} s -> {F/best:.1f} frames/s", flush=True)
