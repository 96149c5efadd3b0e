#!/usr/bin/env python
"""Occluder BVH timings (profiles/r5_occluder_bvh.md): BVH build per occluder set, gvpm_occluded throughput per path,
and the cfg5-sized G-BRE / cfg3-sized G-Beams gathers with the 12 walls (the list path) and with 1 k, 100 k and 1 M
extra triangles (BVH; the list where it finishes in reasonable time).

    python tools/time_occluders.py [--quick] [--list-gathers N] [--out FILE]

--list-gathers: the list path is timed up to N extra triangles (default 1000).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gvpm_b200 as g  # noqa: E402
import occluder_sets as S  # noqa: E402
from gvpm_b200 import records as R  # noqa: E402
from gvpm_b200.api import Context  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal of the script, not a measurement)")
ap.add_argument("--list-gathers", type=int, default=1000)
ap.add_argument("--out", help="also write the results as JSON to this file")
a = ap.parse_args()


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # noqa: BLE001
        return "unknown"


res = {"gpu": gpu_name(), "build": {}, "occluded": {}, "gathers": {}}
print("gpu:", res["gpu"], flush=True)
q = a.quick
sets = {
    "walls_12": S.walls,
    "blocker_24": lambda: np.concatenate([S.walls(), S.blocker_sheets()]),
    "blocker_grid_49k": lambda: S.blocker_sheets(cells=16 if q else 64),
    "sphere_20k": lambda: S.uv_sphere(32, 20) if q else S.uv_sphere(128, 80),
    "soup_100k": lambda: S.soup(5000 if q else 100000),
    "soup_100k_shifted": lambda: S.soup(5000 if q else 100000, shift=1000.0),
    "height_field_1m": lambda: S.height_field(64 if q else 708),
}

ctx = Context(0)
# ---- build and any-hit throughput ---------------------------------------------------------------------------------------
rng = np.random.default_rng(1)
n_rays = 20000 if q else 1 << 20
o = rng.uniform(0.0, 1.0, (n_rays, 3)).astype(np.float32)
d = rng.normal(size=(n_rays, 3))
d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
maxt = rng.uniform(1e-3, 1.0, n_rays).astype(np.float32)
for name, make in sets.items():
    tri = make()
    shift = 1000.0 if "shifted" in name else 0.0
    ro = o + np.float32(shift)
    ctx.set_occluder_accel("list")
    t0 = time.perf_counter(); ctx.set_occluders(tri); t_list = time.perf_counter() - t0
    walls = []
    for _ in range(3):
        ctx.set_occluder_accel("list")
        ctx.set_occluders(tri)
        t0 = time.perf_counter(); ctx.set_occluder_accel("bvh"); walls.append(time.perf_counter() - t0)
    b = dict(n_tri=len(tri), bvh_build_ms=1e3 * min(walls), set_occluders_upload_ms=1e3 * t_list)
    res["build"][name] = b
    print(f"build {name}: {b}", flush=True)
    row = {}
    for path in ("bvh", "list"):
        ctx.set_occluder_accel(path)
        m = n_rays if path == "bvh" else int(min(n_rays, max(4096, 4e9 / max(1, len(tri)))))
        ctx.occluded(ro[:1024], d[:1024], 1e-4, maxt[:1024])   # warm-up
        t0 = time.perf_counter()
        hit = ctx.occluded(ro[:m], d[:m], 1e-4, maxt[:m])
        dt = time.perf_counter() - t0
        row[path] = dict(rays=m, ms=1e3 * dt, rays_per_s=m / dt, hit_fraction=float(hit.mean()))
    res["occluded"][name] = row
    print(f"occluded {name}: {row}", flush=True)

# ---- gathers --------------------------------------------------------------------------------------------------------------
extras = [0, 1000, 100000, 1000000] if not q else [0, 1000, 20000]


def timed(fn, reps=3):
    """median of reps runs after a warm-up; a warm-up over 2 s is reported as it is (one run)"""
    first = fn()
    if first > 2000.0:
        return first
    return float(np.median([fn() for _ in range(reps)]))


SLOW_MS = 20000.0   # a path whose gather took longer than this is not run at the next (larger) size


w, h, nph, scale = (1920, 1080, 10_000_000, 0.1) if not q else (256, 144, 200_000, 0.5)
med = g.make_medium()
ph, _ = g.synth_photons(nph, med, seed=0xC0FFEE + 5, threads=os.cpu_count() or 8)
rays = g.synth_rays(w, h, seed=0xC0FFEE + 6, block=-32)
ctx.set_medium(med)
ctx.set_config(g.make_config(w, h))
ctx.upload_photons(ph)
ctx.upload_rays(rays)
r = g.bre_radius(scale)
slow = set()
for extra in extras:
    tri = np.concatenate([S.walls(), S.soup(extra, seed=17)]) if extra else S.walls()
    for path in ("auto", "list"):
        if path == "list" and extra > a.list_gathers:
            continue
        if path in slow:
            res["gathers"][f"bre_cfg5_walls+{extra}_{path}"] = "not measured: the previous size took > 20 s"
            continue
        ctx.set_occluder_accel(path)
        ctx.set_occluders(tri)
        kind = ctx.occluder_accel()
        if path == "list" and extra == 0:
            continue   # AUTO on the 12 walls is the list already
        ctx.build_points(r)
        out_ptr, _ = ctx.gather_bre_device()

        def run():
            ctx.gather_bre_into(out_ptr, None)
            ctx.sync()
            return ctx.last_timings()[1]
        ms = timed(run)
        key = f"bre_cfg5_walls+{extra}_{kind}"
        if ms > SLOW_MS:
            slow.add(path)
        res["gathers"][key] = dict(gather_ms=ms, pairs=int(ctx.last_gather_detail()[2]))
        print(key, res["gathers"][key], flush=True)

wb, hb, nb, sb = (1280, 720, 500_000, 0.1) if not q else (256, 144, 20_000, 0.5)
beams, _ = R.synth_beams(nb, med, seed=0xC0FFEE + 3, threads=os.cpu_count() or 8)
brays = g.synth_rays(wb, hb, seed=0xC0FFEE + 4, block=-32)
ctx.set_config(g.make_config(wb, hb))
ctx.upload_beams(beams)
ctx.build_beams(g.bre_radius(sb))
ctx.upload_rays(brays)
slow = set()
for extra in extras:
    tri = np.concatenate([S.walls(), S.soup(extra, seed=17)]) if extra else S.walls()
    for path in ("auto", "list"):
        if path == "list" and (extra > a.list_gathers or extra == 0):
            continue
        if path in slow:
            res["gathers"][f"beams_cfg3_walls+{extra}_{path}"] = "not measured: the previous size took > 20 s"
            continue
        ctx.set_occluder_accel(path)
        ctx.set_occluders(tri)
        kind = ctx.occluder_accel()

        def run():
            t0 = time.perf_counter()
            ctx.gather_beams_device()
            ctx.sync()
            return 1e3 * (time.perf_counter() - t0)
        ms = timed(run)
        key = f"beams_cfg3_walls+{extra}_{kind}"
        if ms > SLOW_MS:
            slow.add(path)
        res["gathers"][key] = dict(gather_ms_host_clock=ms)
        print(key, res["gathers"][key], flush=True)
ctx.close()
if a.out:
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
print(json.dumps(res))
