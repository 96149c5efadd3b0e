#!/usr/bin/env python
"""A progressive G-BRE render with the per-pixel accumulators on the device against the same render folding on the
host.  Prints one JSON object.

    python tools/time_progressive.py [--w 1920 --h 1080 --photons 10000000 --iters 8 --reps 3]

Workload (cfg5 size by default): every iteration traces the photons straight into the gather records
(gvpm_trace_photons_direct), generates the camera rays (gvpm_generate_rays, block -32), builds over the photons the
rays can reach (gvpm_build_points_for_rays) at the APA radius of that iteration (3-D schedule, alpha 0.7, from
initialScaleVolume --scale = 0.1 as bench.py's cfg5), gathers and folds.  Two loops of --iters iterations alternate --reps times after one untimed run of each:
  device: gvpm_gather_bre_device + gvpm_accum_add + gvpm_accum_fold;
  host:   gvpm_gather_bre into page-locked host memory + the same fold in vectorised numpy.
ms_per_iteration is a host clock around a whole loop, over --iters; the loop ends in a synchronise.  add_ms and fold_ms
are CUDA events around gvpm_accum_add and gvpm_accum_fold on the context's stream (per call).  After the last loop,
gvpm_reconstruct_accum (L2D) is timed against gvpm_reconstruct on the downloaded accumulators (host clock, both end in
a synchronise).  Medians with min and max.  The GPU's name and power limit are read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import gvpm_b200 as g  # noqa: E402
from gvpm_b200.api import Context  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def stats(v):
    return {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v))}


def run_loop(ctx, a, device, host_out, events):
    import torch
    w, h = a.w, a.h
    scene, cam = g.box_scene_default(), g.pinhole_camera(w, h)
    stream = torch.cuda.ExternalStream(ctx.stream())
    acc = None if device else np.zeros((h * w, 27), dtype=np.float32)
    if device:
        ctx.accum_reset(w, h)
    scale = a.scale
    t0 = time.perf_counter()
    for it in range(1, a.iters + 1):
        n_paths = ctx.trace_photons(scene, a.photons, 0xC0FFEE + it, direct=True)
        ctx.generate_rays(scene, cam, 0x5EED + it, block=-32)
        ctx.build_points_for_rays(g.bre_radius(scale), want_kept=False)
        if device:
            ctx.gather_bre_device()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record(stream)
            ctx.accum_add()
            ev[1].record(stream)
            ctx.accum_fold(it, n_paths)
            ev[2].record(stream)
            events.append(ev)
        else:
            out, _ = ctx.gather_bre(out=host_out, counts=False)
            if it == 1:
                rays = ctx.download_rays()
                pix_of_ray = rays.py.astype(np.int64) * w + rays.px
            pix = np.zeros_like(acc)
            pix[pix_of_ray] = out          # one ray per pixel
            rnb, rit = np.float32(1.0) / np.float32(n_paths), np.float32(1.0) / np.float32(it)
            acc = (acc * np.float32(it - 1) + pix * rnb) * rit
        scale *= ((it - 1 + 0.7) / it) ** (1.0 / 3.0)
    ctx.sync()
    ms = (time.perf_counter() - t0) * 1e3 / a.iters
    return ms, acc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--w", type=int, default=1920)
    ap.add_argument("--h", type=int, default=1080)
    ap.add_argument("--photons", type=int, default=10_000_000)
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=0.1, help="initialScaleVolume of the first iteration (bench.py cfg5)")
    a = ap.parse_args()
    import torch
    ctx = Context(0)
    ctx.set_medium(g.make_medium())
    ctx.set_config(g.make_config(a.w, a.h))
    ctx.set_occluders(g.synth_occluders())
    host_out = torch.empty(a.w * a.h * 27, dtype=torch.float32, pin_memory=True).numpy()
    runs = {True: [], False: []}
    events = []
    host_acc = None
    for rep in range(a.reps + 1):   # rep 0: warm-up of both loops
        for device in (True, False):
            ms, acc = run_loop(ctx, a, device, host_out, events if rep else [])
            if rep:
                runs[device].append(ms)
            if not device:
                host_acc = acc
    torch.cuda.synchronize()
    add_ms = [e[0].elapsed_time(e[1]) for e in events]
    fold_ms = [e[1].elapsed_time(e[2]) for e in events]
    dev_acc, smoke, _ = ctx.accum_read()
    diff = float(np.abs(dev_acc.reshape(-1, 27).astype(np.float64) - host_acc).max() /
                 max(float(np.abs(host_acc).max()), 1e-30))
    rec = {"device": [], "host": []}
    for _ in range(a.reps):
        t = time.perf_counter()
        ctx.reconstruct_accum(preset="L2D")
        rec["device"].append((time.perf_counter() - t) * 1e3)
        t = time.perf_counter()
        acc_h, _, _ = ctx.accum_read()
        ctx.reconstruct(acc_h, a.w, a.h, preset="L2D")
        rec["host"].append((time.perf_counter() - t) * 1e3)
    npix = a.w * a.h
    result = {
        "gpu": gpu_info(), "w": a.w, "h": a.h, "photons": a.photons, "iters": a.iters, "reps": a.reps, "scale": a.scale,
        "device_ms_per_iteration": stats(runs[True]), "host_ms_per_iteration": stats(runs[False]),
        "add_ms": stats(add_ms), "fold_ms": stats(fold_ms),
        # bytes the add (read the ray outputs and px/py, read-modify-write the iteration sum) and the fold (read and
        # write the accumulators and the sum) must move at least
        "add_bytes": npix * (27 * 4 * 3 + 8 + 1), "fold_bytes": npix * 27 * 4 * 4,
        "reconstruct_accum_ms": stats(rec["device"]), "read_then_reconstruct_ms": stats(rec["host"]),
        "pixels_reached": int(smoke.sum()), "device_vs_host_fold_max_rel_diff": diff,
    }
    ctx.close()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
