"""Time the G-VPM camera distance samples drawn on the device against the host path they replace, at the cfg2 size
(512 x 512 camera rays from gvpm_generate_rays, 1 M photons from gvpm_trace_photons_direct, 40 samples per ray, one
radius for every ray).

  draw:      gvpm_generate_vpm_samples (CUDA events on the context's stream; the call ends in its one small
             read-back) against synth_vpm_samples + upload_vpm_samples of the same ray set (host clock, ending in a
             synchronise);
  iteration: one whole G-VPM iteration on the device - build_points_for_rays, the samples, gather_vpm_device,
             accum_add, accum_fold - against the same iteration with the host samples (host clock, ending in a
             synchronise).

Every loop is warmed up, the two variants alternate, and each number is reported as the median with min and max.
Prints one JSON line, with the GPU's name and power limit; --out also writes it to a file.  Needs a CUDA device."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": q[0], "power_limit": q[1] if len(q) > 1 else None}
    except (OSError, subprocess.SubprocessError):
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": None}


def summary(xs):
    return {"median": round(statistics.median(xs), 4), "min": round(min(xs), 4), "max": round(max(xs), 4)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--w", type=int, default=512)
    ap.add_argument("--h", type=int, default=512)
    ap.add_argument("--photons", type=int, default=1_000_000)
    ap.add_argument("--nb", type=int, default=40)
    ap.add_argument("--reps", type=int, default=7, help="timed repetitions of each variant (alternating)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import numpy as np
    import torch
    import gvpm_b200 as g
    from gvpm_b200.api import Context
    if not torch.cuda.is_available():
        raise SystemExit("time_vpm_device.py measures on a CUDA device; none is available")

    w, h, nb, seed = args.w, args.h, args.nb, 0xC0FFEE + 2
    scene, cam, medium = g.box_scene_default(), g.pinhole_camera(w, h), g.make_medium()
    radius = g.bre_radius(1.0)   # cfg2's scale
    ctx = Context(0)
    ctx.set_medium(medium)
    ctx.set_config(g.make_config(w, h))
    ctx.set_occluders(g.synth_occluders())
    ctx.generate_rays(scene, cam, seed + 1, block=-32)
    n_paths = ctx.trace_photons(scene, args.photons, seed, direct=True)
    rays = ctx.download_rays()
    rad = np.full(rays.n, radius, dtype=np.float32)
    ctx.accum_reset(w, h, apa=False)
    stream = torch.cuda.ExternalStream(ctx.stream())
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def draw_device(k):
        ev[0].record(stream)
        n = ctx.generate_vpm_samples(nb, seed=seed + 2 + k, radius=radius)
        ev[1].record(stream)
        ev[1].synchronize()
        return ev[0].elapsed_time(ev[1]), n

    def draw_host(k):
        ctx.sync()
        t0 = time.perf_counter()
        smp = g.synth_vpm_samples(rays, medium, rad, nb_camera_samples=nb, seed=seed + 2 + k)
        ctx.upload_vpm_samples(smp)
        ctx.sync()
        return (time.perf_counter() - t0) * 1e3, smp.n

    it = [0]

    def iteration(samples):
        def run(k):
            ctx.sync()
            t0 = time.perf_counter()
            ctx.build_points_for_rays(radius, want_kept=False)
            n = samples(k)[1]
            ctx.gather_vpm_device(nb)
            ctx.accum_add()
            it[0] += 1
            ctx.accum_fold(it[0], n_paths)
            ctx.sync()
            return (time.perf_counter() - t0) * 1e3, n
        return run

    variants = {"draw_device": draw_device, "draw_host": draw_host,
                "iteration_device": iteration(draw_device), "iteration_host": iteration(draw_host)}
    pairs = [("draw_device", "draw_host"), ("iteration_device", "iteration_host")]
    times = {k: [] for k in variants}
    counts = {k: set() for k in variants}
    for a, b in pairs:
        for k in range(args.warmup):
            variants[a](k)
            variants[b](k)
        for k in range(args.reps):   # alternating; the same seeds on both sides
            for name in (a, b):
                ms, n = variants[name](k)
                times[name].append(ms)
                counts[name].add(n)
    res = {"tool": "time_vpm_device", **gpu_identity(), "rays": rays.n, "photons": args.photons, "nb": nb,
           "reps": args.reps, "warmup": args.warmup,
           "samples_device": sorted(counts["draw_device"]), "samples_host": sorted(counts["draw_host"]),
           "upload_mb": round(min(counts["draw_host"]) * 40 / 1e6, 1)}
    for k, v in times.items():
        res[k + "_ms"] = summary(v)
    res["draw_speedup"] = round(statistics.median(times["draw_host"]) / statistics.median(times["draw_device"]), 1)
    res["iteration_speedup"] = round(statistics.median(times["iteration_host"]) /
                                     statistics.median(times["iteration_device"]), 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
