"""Times the mesh-scene generators on the GPU against the box tracer (profiles/r7_mesh_trace.md):
  10 M photons (gvpm_trace_photons_direct) in the default box vs gvpm_trace_photons_direct_mesh in its triangulation;
  the same in a height field of about 1 M triangles inside the box;
  gvpm_generate_rays_mesh at 1920 x 1080 (camera outside the box) vs gvpm_generate_rays.
Each timed call is followed by a device synchronise (the tracers end in one anyway: they read their batch totals back),
so a host clock around it is the call's time; every shape is run once before the timed repeats.  Prints one JSON line; --out also writes it to a file."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def _timed(ctx, fn, reps):
    fn()
    ctx.sync()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ctx.sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": sorted(ts)[len(ts) // 2], "min_ms": min(ts), "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--photons", type=int, default=10_000_000)
    ap.add_argument("--field-res", type=int, default=707, help="height field of 2 res^2 triangles")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    import gvpm_b200 as g
    import mesh_scenes as MS
    from gvpm_b200.api import Context
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "photons": a.photons}
    med = g.make_medium()
    box = g.box_scene_default()
    ctx = Context(0)
    ctx.set_medium(med)
    ctx.set_config(g.make_config(1920, 1080))
    n = a.photons
    res["box_photons_direct"] = _timed(ctx, lambda: ctx.trace_photons(box, n, 1, direct=True), a.reps)
    cornell = MS.cornell()
    ctx.set_trace_mesh(**cornell.kwargs())
    res["cornell_mesh_photons_direct"] = _timed(ctx, lambda: ctx.trace_photons_mesh(n, 1, direct=True), a.reps)
    cam_box = g.pinhole_camera(1920, 1080)
    cam = g.lookat_camera(1920, 1080, (0.5, 0.5, -1.5), tan_half_fov_x=float(cam_box.tan_half_fov_x))
    res["box_rays_1080p"] = _timed(ctx, lambda: ctx.generate_rays(box, cam_box, 3), a.reps)
    res["cornell_mesh_rays_1080p"] = _timed(ctx, lambda: ctx.generate_rays_mesh(cam, 3), a.reps)
    field = MS.large_field(a.field_res)
    res["field_triangles"] = int(field.tri.shape[0])
    t0 = time.perf_counter()
    ctx.set_trace_mesh(**field.kwargs())
    res["field_set_trace_mesh_ms"] = (time.perf_counter() - t0) * 1e3
    res["field_mesh_photons_direct"] = _timed(ctx, lambda: ctx.trace_photons_mesh(n, 1, direct=True), a.reps)
    res["field_mesh_rays_1080p"] = _timed(ctx, lambda: ctx.generate_rays_mesh(cam, 3), a.reps)
    ctx.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
