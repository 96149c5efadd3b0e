#!/usr/bin/env python
"""Time the perspective-grid build of bench.py's value leg (cfg5 inputs, one GPU): gvpm_build_points_for_rays over the
10 M staged photons, with the camera rays uploaded once.

    python tools/time_build.py [--builds 50] [--warmup 5]            CUDA events, no profiler
    python tools/time_build.py --profile [--builds 20]                average time of each build kernel (torch.profiler)
    python tools/time_build.py --traced [--profile]                   the same over records traced on the device
                                                                      (gvpm_trace_photons_direct + gvpm_generate_rays)

The two modes belong in separate runs: the profiler slows the host.  GVPM_B200_LIB=<other build of libgvpm_b200.so>
times another build of the library on the same inputs.
"""
import argparse
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import gvpm_b200 as g  # noqa: E402
from gvpm_b200.api import Context  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--photons", type=int, default=10_000_000)
ap.add_argument("--scale", type=float, default=0.1)
ap.add_argument("--w", type=int, default=1920)
ap.add_argument("--h", type=int, default=1080)
ap.add_argument("--builds", type=int, default=50)
ap.add_argument("--warmup", type=int, default=5)
ap.add_argument("--profile", action="store_true", help="list each build kernel's average time (torch.profiler)")
ap.add_argument("--traced", action="store_true", help="photons traced into records and rays generated on the device "
                "(the device_traced leg of bench.py) instead of the staged cfg5 inputs")
a = ap.parse_args()


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=20).stdout.strip()
    except Exception as e:   # the numbers stay valid; the card line is then missing
        return f"nvidia-smi unavailable ({e})"


# the inputs of bench.py cfg5 at N = 1 (same seeds)
seed = 0xC0FFEE + 5
med = g.make_medium()
radius = g.bre_radius(a.scale)
ctx = Context(0)
ctx.set_medium(med)
ctx.set_config(g.make_config(a.w, a.h))
ctx.set_occluders(g.synth_occluders())
if a.traced:
    ctx.trace_photons(g.box_scene_default(), a.photons, seed + 100, direct=True)
    ctx.generate_rays(g.box_scene_default(), g.pinhole_camera(a.w, a.h), seed + 200, block=-32)
    n_rays = a.w * a.h
else:
    ph, _ = g.synth_photons(a.photons, med, seed=seed, threads=min(32, os.cpu_count() or 8))
    rays = g.synth_rays(a.w, a.h, seed=seed + 1, block=-32)
    ctx.upload_photons(ph)
    ctx.upload_rays(rays)
    n_rays = rays.n
kept = ctx.build_points_for_rays(radius, want_kept=True)
assert ctx.accel_kind() == "frustum", ctx.accel_kind()
for _ in range(a.warmup):
    ctx.build_points_for_rays(radius, want_kept=False)
ctx.sync()
lib = os.environ.get("GVPM_B200_LIB") or "in-tree libgvpm_b200.so"
print(f"card: {card()}")
print(f"library: {lib}; {'traced records' if a.traced else 'staged photons'}: {a.photons} photons, {n_rays} rays, "
      f"radius {radius:.6g}, kept {kept}")

if not a.profile:
    per_build = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(a.builds):
        ctx.build_points_for_rays(radius, want_kept=False)
        per_build.append(ctx.last_timings()[0])   # events around the build's own launches (synchronises)
    e1.record()
    torch.cuda.synchronize()
    b = np.array(per_build)
    print(f"build_ms: mean {b.mean():.4f} median {np.median(b):.4f} min {b.min():.4f} max {b.max():.4f} over {a.builds} builds; "
          f"loop {e0.elapsed_time(e1) / a.builds:.4f} ms per build (host read-back of each build's timing included)")
    print(f"card after: {card()}")
else:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.builds):
            ctx.build_points_for_rays(radius, want_kept=False)
        ctx.sync()
    rows = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            rows.append((e.key, e.count, t / e.count / 1e3, t / a.builds / 1e3))
    rows.sort(key=lambda r: -r[3])
    print(f"{'kernel':<60} {'calls':>6} {'ms/call':>9} {'ms/build':>9}")
    for k, c, per_call, per_build in rows:
        print(f"{k[:60]:<60} {c:>6} {per_call:>9.4f} {per_build:>9.4f}")
    print(f"sum of device time per build: {sum(r[3] for r in rows):.4f} ms")
ctx.close()
