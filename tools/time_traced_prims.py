#!/usr/bin/env python
"""Beams and planes made on the device against the host path, at bench sizes.  Prints one JSON object.

    python tools/time_traced_prims.py [--reps 3] [--shapes cfg3,beams1080,cfg4]

Per shape, the two ways of getting an iteration's primitives onto the device alternate (after one untimed warm-up of
each):
  device: gvpm_trace_beams (+ gvpm_planes_from_beams for planes);
  host:   gvpm_synth_beams on every host core + gvpm_upload_beams (+ gvpm_synth_planes + gvpm_upload_planes).
trace / planes / synth / upload are host-clock times around calls that end in a stream synchronise; build and gather
are the context's CUDA events around gvpm_build_* and gvpm_gather_* of the same primitives (cfg4: the camera inside the
medium, planes without bench.py's sheet squeeze).  Medians over --reps, with min and max.  The GPU's name and power limit
are read in the same process.
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
from gvpm_b200 import records as R  # noqa: E402
from gvpm_b200.api import Context  # noqa: E402

SHAPES = {  # technique, width, height, primitives, initialScaleVolume (bench.py TECHNIQUES)
    "cfg3": ("beams", 1280, 720, 500_000, 0.1),
    "beams1080": ("beams", 1920, 1080, 1_000_000, 0.1),
    "cfg4": ("planes", 1280, 720, 200_000, 0.1),
}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fn):
    t = time.perf_counter()
    r = fn()
    return r, (time.perf_counter() - t) * 1e3


def run_once(ctx, tech, n, seed, medium, radius, device, threads):
    t = {}
    if device:
        paths, t["trace_ms"] = timed(lambda: ctx.trace_beams(g.box_scene_default(), n, seed))
        if tech == "planes":
            _, t["planes_ms"] = timed(lambda: ctx.planes_from_beams(seed + 7))
    else:
        (beams, paths), t["synth_beams_ms"] = timed(lambda: R.synth_beams(n, medium, seed=seed, threads=threads))
        if tech == "beams":
            _, t["upload_ms"] = timed(lambda: ctx.upload_beams(beams))
        else:
            planes, t["synth_planes_ms"] = timed(lambda: R.synth_planes(beams, medium, seed=seed + 7))
            _, t["upload_ms"] = timed(lambda: ctx.upload_planes(planes))
    if tech == "beams":
        ctx.build_beams(radius)
        out, _ = ctx.gather_beams(counts=False)
    else:
        ctx.build_planes()
        out, _ = ctx.gather_planes(counts=False)
    t["build_ms"], t["gather_ms"] = ctx.last_timings()
    t["paths"] = paths
    t["checksum"] = float(out.astype(np.float64).sum())
    return t


def summary(runs):
    out = {}
    for k in runs[0]:
        v = [r[k] for r in runs]
        out[k] = v[0] if k == "paths" else {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="cfg3,beams1080,cfg4")
    a = ap.parse_args()
    threads = os.cpu_count() or 8
    result = {"gpu": gpu_info(), "host_threads": threads, "reps": a.reps, "shapes": {}}
    for name in a.shapes.split(","):
        tech, w, h, n, scale = SHAPES[name]
        seed = 0xC0FFEE + {"cfg3": 3, "cfg4": 4, "beams1080": 6}[name]
        medium = g.make_medium()
        if tech == "planes":
            rays = g.synth_rays(w, h, seed=seed + 1, block=-32, cam_dist=-0.05, cover=0.45)
        else:
            rays = g.synth_rays(w, h, seed=seed + 1, block=-32)
        ctx = Context(0)
        ctx.set_medium(medium)
        ctx.set_config(g.make_config(w, h))
        ctx.set_occluders(g.synth_occluders())
        ctx.upload_rays(rays)
        radius = g.bre_radius(scale)
        runs = {True: [], False: []}
        for rep in range(a.reps + 1):
            for device in (True, False):
                t = run_once(ctx, tech, n, seed, medium, radius, device, threads)
                if rep:
                    runs[device].append(t)
        ctx.close()
        result["shapes"][name] = {"technique": tech, "rays": rays.n, "primitives": n,
                                  "device": summary(runs[True]), "host": summary(runs[False])}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
