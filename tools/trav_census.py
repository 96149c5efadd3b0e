#!/usr/bin/env python
"""Census of the perspective-grid traversal (k_bre_grid_traverse) on bench.py's cfg5 inputs: photons per footprint class,
and per 32-ray tile the classes that hold candidates for it, the candidates per lane, and the batch slots the traversal
issues against the candidates it tests.

    python tools/trav_census.py [--scale 0.1] [--w 1920 --h 1080] [--photons 10000000]

The grid and its cell_start come from the library (Context.frustum_grid); the rays' cells are recomputed here in fp32
with the kernel's arithmetic (not necessarily bit-exact: a census).  'per-class rounds' is the traversal that visits
every class holding a photon anywhere and runs ceil(max_lane(candidates) / kTileBatch) batches per class and grid;
'one stream' runs ceil(max_lane(sum over classes) / kTileBatch) batches per tile over the classes the tile's census keeps.
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import gvpm_b200 as g  # noqa: E402
from gvpm_b200.api import Context  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--photons", type=int, default=10_000_000)
ap.add_argument("--scale", type=float, default=0.1)
ap.add_argument("--w", type=int, default=1920)
ap.add_argument("--h", type=int, default=1080)
ap.add_argument("--batch", type=int, default=16, help="kTileBatch")
a = ap.parse_args()
B = a.batch

seed = 0xC0FFEE + 5   # bench.py cfg5 at N = 1
med = g.make_medium()
radius = g.bre_radius(a.scale)
cfg = g.make_config(a.w, a.h)
ctx = Context(0)
ctx.set_medium(med)
ctx.set_config(cfg)
ph, _ = g.synth_photons(a.photons, med, seed=seed, threads=min(32, os.cpu_count() or 8))
rays = g.synth_rays(a.w, a.h, seed=seed + 1, block=-32)
ctx.upload_photons(ph)
ctx.upload_rays(rays)
kept = ctx.build_points_for_rays(radius, want_kept=True)
assert ctx.accel_kind() == "frustum", ctx.accel_kind()
G, cs = ctx.frustum_grid()
ctx.close()
cs = cs.astype(np.int64)
ncl, ncell = G.classes, G.n_cells
grids = 2 if G.parity_split else 1
near = int(cs[grids * ncell + 1] - cs[grids * ncell])
print(f"rays {rays.n}, photons {a.photons}, kept {kept}, radius {radius:.6g}, classes {ncl}, cells per grid {ncell}, "
      f"grids {grids}, NEAR {near}")
print("class  nx x ny        cell edge   photons   per cell")
for c in range(ncl):
    n_c = sum(int(cs[q * ncell + G.base[c] + G.nx[c] * G.ny[c]] - cs[q * ncell + G.base[c]]) for q in range(grids))
    print(f"{c:5d}  {G.nx[c]:5d} x {G.ny[c]:<5d}  {G.csize[c]:.3e}  {n_c:9d}  {n_c / (G.nx[c] * G.ny[c]):8.3f}")

# the lanes' windows, as k_bre_grid_traverse computes them
f32 = np.float32
d = rays.view("d").astype(f32)
mint, elen = rays.mint.astype(f32), rays.edge_len.astype(f32)
px, py = rays.px.astype(np.int64), rays.py.astype(np.int64)
active = elen >= mint
m, u, v = (np.array(list(x), dtype=f32) for x in (G.m, G.u, G.v))
z = d @ m
iz = f32(1) / z
x = (d @ u) * iz
y = (d @ v) * iz
parity = (px + py) % 2
# pathSet prefilter with a parity-split grid: a ray scans the grid of its own parity only
only_mine = bool(G.parity_split) and bool(cfg.path_set)
passes = [None] if only_mine else list(range(grids))
n = rays.n
n_tiles = (n + 31) // 32
pad = n_tiles * 32 - n


def tiles(vals, fill=0):
    return np.concatenate([vals, np.full(pad, fill, dtype=vals.dtype)]).reshape(n_tiles, 32)


rounds_now = np.zeros(n_tiles, dtype=np.int64)     # batches of the per-class loop
visited_now = 0                                    # classes the per-class loop visits (globally non-empty)
cand_total = np.zeros(n, dtype=np.int64)           # candidates per lane over every class and grid
classes_hit = np.zeros(n_tiles, dtype=np.int64)    # classes with a candidate in some lane's 3x3 window
for c in range(ncl):
    nx, ny, base = int(G.nx[c]), int(G.ny[c]), int(G.base[c])
    if all(cs[q * ncell + base] == cs[q * ncell + base + nx * ny] for q in range(grids)):
        continue
    visited_now += 1
    ic = f32(1) / f32(G.csize[c])
    cx = np.clip(np.floor((x - f32(G.gx0)) * ic).astype(np.int64), 0, nx - 1)
    cy = np.clip(np.floor((y - f32(G.gy0)) * ic).astype(np.int64), 0, ny - 1)
    x0, x1 = np.maximum(cx - 1, 0), np.minimum(cx + 1, nx - 1)
    y0, y1 = np.maximum(cy - 1, 0), np.minimum(cy + 1, ny - 1)
    tot_c = np.zeros(n, dtype=np.int64)
    for q in passes:
        gb = (parity if q is None else q) * ncell + base
        tot = np.zeros(n, dtype=np.int64)
        for dy in range(3):
            yy = y0 + dy
            ok = active & (yy <= y1)
            rb = gb + yy * nx
            tot += np.where(ok, cs[np.where(ok, rb + x1 + 1, 0)] - cs[np.where(ok, rb + x0, 0)], 0)
        rounds_now += (tiles(tot).max(axis=1) + B - 1) // B
        tot_c += tot
    cand_total += tot_c
    classes_hit += tiles(tot_c).max(axis=1) > 0
if near:
    visited_now += 1
    cand_total += np.where(active, near, 0)
    rounds_now += (tiles(np.where(active, near, 0)).max(axis=1) + B - 1) // B
    classes_hit += tiles(active.astype(np.int64)).max(axis=1) > 0
ct = tiles(cand_total)
rounds_stream = (ct.max(axis=1) + B - 1) // B
tested = ct.sum(axis=1)
print(f"\nper tile ({n_tiles} tiles of 32 rays; NEAR counts as a class):")
print(f"  classes the per-class loop visits: {visited_now} (every tile)")
q = np.percentile(classes_hit, [0, 50, 90, 100])
print(f"  classes with a candidate for the tile: mean {classes_hit.mean():.2f}  min/median/p90/max {q[0]:.0f}/{q[1]:.0f}/{q[2]:.0f}/{q[3]:.0f}")
q = np.percentile(cand_total[active], [0, 50, 90, 99, 100])
print(f"  candidates per active lane: mean {cand_total[active].mean():.1f}  min/median/p90/p99/max "
      f"{q[0]:.0f}/{q[1]:.0f}/{q[2]:.0f}/{q[3]:.0f}/{q[4]:.0f}")
for name, r in (("per-class rounds", rounds_now), ("one stream", rounds_stream)):
    slots = r * B * 32
    print(f"  {name:17s}: batches per tile mean {r.mean():6.2f}; lane slots {slots.sum():.4e} for {tested.sum():.4e} "
          f"candidates tested ({tested.sum() / max(slots.sum(), 1) * 100:.1f} % of the slots)")
