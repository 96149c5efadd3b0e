#!/usr/bin/env python
"""Time the G-BRE gather on the perspective grid (k_bre_grid_traverse + k_bre_shade) on bench.py's cfg5 inputs:
gvpm_build_points_for_rays once, then gvpm_gather_bre_into (the filters applied in the traversal, as bench.py runs it).
tools/time_gather.py times the box-hierarchy path instead.

    python tools/time_grid_traverse.py [--gathers 50] [--warmup 5]      CUDA events, no profiler
    python tools/time_grid_traverse.py --profile [--gathers 20]          average time of each gather kernel (torch.profiler)

GVPM_B200_LIB=<other build of libgvpm_b200.so> times another build of the library on the same inputs.
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
ap.add_argument("--gathers", type=int, default=50)
ap.add_argument("--warmup", type=int, default=5)
ap.add_argument("--profile", action="store_true", help="list each gather kernel's average time (torch.profiler)")
a = ap.parse_args()


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=20).stdout.strip()
    except Exception as e:   # the numbers stay valid; the card line is then missing
        return f"nvidia-smi unavailable ({e})"


seed = 0xC0FFEE + 5   # bench.py cfg5 at N = 1
med = g.make_medium()
radius = g.bre_radius(a.scale)
ctx = Context(0)
ctx.set_medium(med)
ctx.set_config(g.make_config(a.w, a.h))
ctx.set_occluders(g.synth_occluders())
ph, _ = g.synth_photons(a.photons, med, seed=seed, threads=min(32, os.cpu_count() or 8))
rays = g.synth_rays(a.w, a.h, seed=seed + 1, block=-32)
ctx.upload_photons(ph)
ctx.upload_rays(rays)
kept = ctx.build_points_for_rays(radius, want_kept=True)
assert ctx.accel_kind() == "frustum", ctx.accel_kind()
out = torch.zeros(rays.n * 27, dtype=torch.float32, device="cuda")
for _ in range(a.warmup):
    ctx.gather_bre_into(out.data_ptr(), None)
ctx.sync()
lib = os.environ.get("GVPM_B200_LIB") or "in-tree libgvpm_b200.so"
print(f"card: {card()}")
print(f"library: {lib}; {a.photons} photons, {rays.n} rays, radius {radius:.6g}, kept {kept}")

if not a.profile:
    tr, sh, gm = [], [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.gathers):
        e0.record(torch.cuda.current_stream())
        ctx.gather_bre_into(out.data_ptr(), None)
        ctx.sync()
        e1.record(torch.cuda.current_stream())
        torch.cuda.synchronize()
        t, s, pairs = ctx.last_gather_detail()
        tr.append(t)
        sh.append(s)
        gm.append(ctx.last_timings()[1])
    for name, v in (("traverse_ms", tr), ("shade_ms", sh), ("gather_ms", gm)):
        v = np.array(v)
        print(f"{name}: median {np.median(v):.4f} min {v.min():.4f} max {v.max():.4f} over {a.gathers} gathers")
    print(f"pairs {pairs}; checksum {float(out.double().sum()):.9e}")
    print(f"card after: {card()}")
else:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.gathers):
            ctx.gather_bre_into(out.data_ptr(), None)
        ctx.sync()
    rows = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            rows.append((e.key, e.count, t / e.count / 1e3, t / a.gathers / 1e3))
    rows.sort(key=lambda r: -r[3])
    print(f"{'kernel':<60} {'calls':>6} {'ms/call':>9} {'ms/gather':>9}")
    for k, c, per_call, per_g in rows:
        print(f"{k[:60]:<60} {c:>6} {per_call:>9.4f} {per_g:>9.4f}")
ctx.close()
