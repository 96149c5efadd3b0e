#!/usr/bin/env python
"""bench.py — one G-BRE 3D mixed-shift gather iteration per step (BASELINE.json configs[4]).

    python bench.py --gpus N --steps K --warmup W            (torchrun launches N ranks for N > 1)
    python bench.py --impl reference ...                     CPU arm: the reference's own compiled G-BRE path on host cores
                                                             (oracle/_ref/libgvpm_functor_ref.so: kd-tree / BVH, traversal and
                                                             shift functor, for every workload; the oracle restatement when
                                                             that library or the memory for it is missing)
    python bench.py --workload poisson1080 [--impl reference]   row f-3: one screened-Poisson reconstruction per step; the
                                                             reference arm is the reference's own solver (OpenMP backend),
                                                             the GPU line also times its CUDA backend on the same device
    python bench.py ... --dump-outputs DIR                   also writes what the timed path computed in its last step
                                                             as DIR/<name>.npy (one GPU; the inputs are seeded, so two
                                                             builds can be compared output for output)

The bench writes nothing into the tree it runs from (which may be read-only): no bytecode caches, and the CPU
baseline's -march=native oracle build goes to a temporary directory.

Workload "cfg5": synthetic 1920x1080 homogeneous-medium Cornell scene, 10 M photons per iteration,
G-BRE 3D kernel, mixed shift (useShiftNull), area MIS, pathSet; radius = bsphereR * scale * 0.01.
A step = accel build + gather of every camera-ray medium segment of the image (primal + 4 gradient
contributions = 27 floats per ray).  N > 1: strong scaling - the 32x32 gather blocks are dealt to the ranks in
cost-balanced column bands of the image (gvpm_b200/shard.py, costs from one untimed pilot iteration); every rank holds
1/N of the iteration's photon set and DISPATCHES it (gvpm_dispatch_*): each photon goes, as a packed 128-byte gather
record over peer-mapped NVLink stores, only to the ranks whose rays can reach it; every rank builds its perspective grid
over what it received and gathers its blocks; results go to rank 0's shared image buffer by device-to-device copies
(north_star: "primal and gradient buffers gathered at the end of each iteration").  The dispatch of iteration k+1 is
double-buffered behind the build + gather of iteration k (a renderer traces the next iteration's photons while the
current one is gathered); the K timed steps contain K dispatches and K result collections.  Ray sets that are not
concurrent fall back to the round-1 whole-set exchange (peer copies, or an NCCL all-gather).

value  = rays / s with the rays and each rank's photon slice already resident in HBM.
e2e    = same through the C ABI with HOST (pinned) buffers: H2D of the photon slice (gvpm_upload_photons_slice)
         and of the rays, all-gather, build, gather, D2H of the 27 planes (gvpm_gather_bre_host), every step.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

WORKLOADS = {
    # name: (w, h, photons, default scale)
    "cfg5": (1920, 1080, 10_000_000, 0.1),
    "cfg1": (256, 256, 100_000, 1.0),
}
# The other techniques of BASELINE.json's configs (technique_main): (technique, w, h, primitives, initialScaleVolume)
TECHNIQUES = {
    "cfg2": ("vpm", 512, 512, 1_000_000, 1.0),          # G-VPM, 40 distance samples per pixel, unit = pixel
    "cfg3": ("beams", 1280, 720, 500_000, 0.1),         # G-Beams 3D kernel
    "cfg4": ("planes", 1280, 720, 200_000, 0.1),        # G-Planes 0D, LASER-style sheet, sensor inside the medium
    "beams1080": ("beams", 1920, 1080, 1_000_000, 0.1), # north_star's second target: G-Beams-3D at 1920x1080
}


# row f-3: screened-Poisson reconstruction of one gradient-domain image set (poisson::Solver, gvpm.cpp:610-690)
POISSON = {"poisson1080": (1920, 1080, "L2D"), "poisson720": (1280, 720, "L2D"), "poisson1080_l1": (1920, 1080, "L1D")}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=sorted(WORKLOADS) + sorted(TECHNIQUES) + sorted(POISSON))
    ap.add_argument("--scale", type=float, default=None, help="initialScaleVolume (paper preset 0.1)")
    ap.add_argument("--photons", type=int, default=None)
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="target CPU-baseline sample time")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path computed in its last step as DIR/<name>.npy "
                         "(a fixed, seeded sample of the rays where the whole output exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


# --------------------------------------------------------------------------------------------
DUMP_MAX_BYTES = 64 << 20
DUMP_MAX_RAYS = 1 << 18     # 27 floats per ray: 28 MB of gather output


def dump_rows(n):
    """--dump-outputs: the rays whose results are written, a fixed seeded sample (sorted) when there are too many"""
    if n <= DUMP_MAX_RAYS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0xD0).choice(n, DUMP_MAX_RAYS, replace=False))


def dump_outputs(path, arrays):
    """--dump-outputs: every array as <path>/<name>.npy (float32 / float64 only, 64 MB at most in all)"""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def dump_gather(path, out_dev, rays, mvol_dev=None):
    """--dump-outputs of a gather: the 27 output floats per ray (mediumFlux[3], shiftedMediumFlux[4][3],
    weightedMediumFlux[4][3]) of the sampled rays, with their index in the ray set and their pixel; for G-VPM also MVol
    (int32 view of the uint32 photon count per ray that drives the host's radius update)"""
    import torch
    rows = dump_rows(rays.n)
    idx = torch.from_numpy(rows).to(out_dev.device)
    arrays = {"gather_out": out_dev[:rays.n * 27].view(rays.n, 27)[idx].cpu().numpy(), "ray_index": rows.astype(np.float64),
              "ray_pixel": np.stack([rays.px[rows], rays.py[rows]], axis=1).astype(np.float64)}
    if mvol_dev is not None:
        arrays["gather_mvol"] = mvol_dev[:rays.n][idx].cpu().numpy().view(np.uint32).astype(np.float64)
    dump_outputs(path, arrays)


def pinned(n, dtype):
    import torch
    t = torch.empty(n, dtype=dtype, pin_memory=torch.cuda.is_available())
    return t, t.numpy()


def make_inputs(args, rank, world, pin=True):
    """Synthetic inputs in pinned host memory (untimed set-up)."""
    import torch
    import gvpm_b200 as g
    from gvpm_b200 import records as R
    w, h, n_ph, scale = WORKLOADS[args.workload]
    if args.photons:
        n_ph = args.photons
    if args.scale:
        scale = args.scale
    seed = 0xC0FFEE + 5
    medium = g.make_medium()
    keep = []

    def alloc(fields, n):
        arrs = {}
        for name, dt, wd in fields:
            tdt = {np.float32: torch.float32, np.uint8: torch.uint8, np.uint32: torch.int32,
                   np.int32: torch.int32}[dt]
            if pin:
                t, a = pinned(n * wd, tdt)
                keep.append(t)
                arrs[name] = a.view(dt)
            else:
                arrs[name] = np.zeros(n * wd, dtype=dt)
        return arrs

    threads = max(1, min(32, (os.cpu_count() or 8) // max(1, world)))
    photons = None
    n_paths = 0
    if rank == 0 or args.impl == "reference":
        photons = R.PhotonSet(n_ph, **alloc(R._PHOTON_FIELDS, n_ph))
        s = g._native.load_synth()
        cs = photons.as_c()
        n_paths = s.gvpm_synth_photons(seed, n_ph, C.byref(medium), 12, 1, 0, 100.0, threads, C.byref(cs))
    # 32x32 gather blocks like the reference (gvpm.cpp:271-290), walked in Z-order inside a block so that
    # consecutive rays are 2x2 pixel quads (the traversal kernel packets 4 consecutive rays)
    full = g.synth_rays(w, h, seed=seed + 1, block=-32)
    # 32x32 gather blocks -> ranks.  "band" (default): column bands of the image, dealt cyclically, so that a rank's
    # rays cross only a few wedges of the scene and gvpm_build_points_for_rays can leave the rest of the photon set out
    # of that rank's hierarchy; "tile": round robin over the blocks (every rank sees the whole scene).
    from gvpm_b200 import shard
    if shard_mode(world) == "band":
        mine = shard.band_indices(full.px, full.py, w, h, world, rank, band_cycles())
    else:
        mine = shard.local_indices(full.px, full.py, w, world, rank)
    sub = full.take(mine)
    rays = R.RaySet(sub.n, **alloc(R._RAY_FIELDS, sub.n))
    for name, _, _ in R._RAY_FIELDS:
        getattr(rays, name)[:] = getattr(sub, name)
    cfg = g.make_config(w, h)
    return dict(w=w, h=h, n_ph=n_ph, scale=scale, medium=medium, photons=photons, n_paths=int(n_paths),
                rays=rays, rays_full_n=full.n, cfg=cfg, tri=g.synth_occluders(), radius=g.bre_radius(scale),
                keep=keep, full_rays=full if (rank == 0 or world > 1) else None, alloc=alloc)


def shard_mode(world):
    return os.environ.get("GVPM_SHARD", "band") if world > 1 else "tile"


def default_push_ctas(world):
    """photon exchange: the copy engines keep up with one or two peers; beyond that the many-small-copies pattern
    (13 fields x N-1 peers) tops out near 220 GB/s per GPU and a 12-CTA store kernel takes over (profiles/r1j)"""
    return 12 if world > 2 else 0


def band_cycles():
    return int(os.environ.get("GVPM_BAND_CYCLES", "2"))


def prune_build(world):
    """build the acceleration structure for the uploaded rays (gvpm_build_points_for_rays): the perspective grid for
    the concurrent primary rays of this workload (any N), or the pruned hierarchy under GVPM_ACCEL=bvh (N > 1, band
    sharding).  GVPM_PRUNE=0: plain gvpm_build_points."""
    if os.environ.get("GVPM_PRUNE", "1") == "0":
        return False
    if os.environ.get("GVPM_ACCEL", "") == "bvh":
        return world > 1 and shard_mode(world) == "band"
    return True


class ClockSampler:
    """nvidia-smi clock/throttle sampling DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.proc = None
        self.lines = []
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class DevView:
    """__cuda_array_interface__ wrapper so torch can alias a raw device pointer (no copy)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def measured_traffic(workload, world):
    """DRAM bytes per launch of the dominant kernels from the committed ncu capture (profiles/traffic.json)."""
    if world != 1:
        return None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            e = json.load(f)[workload]
        return float(e["bytes_per_launch"]), e["source"]
    except Exception:
        return None, None


def l2_roofline(workload, world, kernel_ms):
    """BASELINE.json's metric names "% of HBM/L2 peak": L2 bytes of the dominant kernels (lts__t_bytes.sum of the committed
    ncu capture) over their live duration, against the L2 read bandwidth measured on this pool's B200s with the library's
    own 128-bit load sweep over an L2-resident buffer (tools/measure_l2.py -> profiles/r2_l2_peak.json)."""
    if world != 1:
        return None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            e = json.load(f)[workload]
        with open(os.path.join(ROOT, "profiles", "r2_l2_peak.json")) as f:
            pk = json.load(f)
        b = float(e["l2_bytes_per_launch"])
        ach = b / (kernel_ms * 1e-3) / 1e9
        return {"bytes_per_launch": b, "achieved": ach, "peak": float(pk["l2_read_peak_gbs"]), "unit": "GB/s",
                "frac": ach / float(pk["l2_read_peak_gbs"]),
                "peak_source": "measured: gvpm_measure_read_bandwidth over 16-64 MB (profiles/r2_l2_peak.json)",
                "bytes_source": e["source"]}
    except Exception:
        return None


def _native_lib_path():
    from gvpm_b200 import _native as NAT
    return NAT.LIB_PATH


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# --------------------------------------------------------------------------------------------
def cpu_arm(args, inp, seconds):
    """The reference's CPU gather as restated by the oracle (kd layout + AABB hierarchy + stack DFS,
    worker threads pulling ray tiles), on all host cores, on a bounded sample of the same workload."""
    from oracle import binding as ob
    if "oracle_flags" not in inp:      # BASELINE.md §2: -O3 -march=native, built on the box that is timed (untimed here)
        inp["oracle_flags"] = ob.prefer_native() if ob._lib is None else "as loaded"
    lib = ob.load()
    from gvpm_b200 import _native as N
    cores = ob.hw_threads()
    ph, rays = inp["photons"], inp["full_rays"] if inp.get("full_rays") is not None else inp["rays"]
    cph = ph.as_c()
    tree = lib.gvpm_oracle_tree_build(C.byref(cph), ph.n, inp["radius"], 0)
    build_ms = lib.gvpm_oracle_tree_build_ms(tree)
    # sample = whole 1024-ray tiles spread evenly over the ray list (every k-th tile)
    n_tiles = max(1, rays.n // 1024)

    def run(tile_ids, threads=None):
        idx = (np.asarray(tile_ids)[:, None] * 1024 + np.arange(1024)[None, :]).reshape(-1)
        idx = idx[idx < rays.n]
        sub = rays.take(idx)
        cr = sub.as_c()
        out = np.zeros(sub.n * 27, dtype=np.float32)
        ms = C.c_double(0)
        tri = inp["tri"]
        rc = lib.gvpm_oracle_bre(tree, C.byref(cph), ph.n, C.byref(cr), 0, sub.n, C.byref(inp["medium"]),
                                 C.byref(inp["cfg"]), tri.ctypes.data_as(N.f32p), tri.size // 9, inp["radius"], 0,
                                 threads or cores, out.ctypes.data_as(N.f32p), None, None, None, 0, C.byref(ms))
        assert rc >= 0
        return sub.n, ms.value

    pilot_tiles = np.linspace(0, n_tiles - 1, num=min(n_tiles, max(8, cores // 4)), dtype=np.int64)
    n0, ms0 = run(np.unique(pilot_tiles))
    rate = n0 / max(ms0, 1e-3) * 1e3
    want = int(min(n_tiles, max(len(pilot_tiles), rate * seconds / 1024)))
    tiles = np.unique(np.linspace(0, n_tiles - 1, num=want, dtype=np.int64))
    n1, ms1 = run(tiles)
    # single-thread figure (BASELINE.md §2) on a slice of the same sample, once per process
    if "cpu_single" not in inp:
        k1 = max(2, len(tiles) // max(cores, 1))
        ns, mss = run(tiles[::max(1, len(tiles) // k1)][:k1], threads=1)
        inp["cpu_single"] = ns / max(mss, 1e-3) * 1e3
    lib.gvpm_oracle_tree_free(tree)
    rate = n1 / ms1 * 1e3
    r_full = float(inp.get("rays_full_n", rays.n))
    return {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port",
            "flags": inp["oracle_flags"], "build_ms": build_ms, "gather_ms_sample": ms1,
            "single_thread_value": inp["cpu_single"],
            "iteration_value_including_build": r_full / (build_ms * 1e-3 + r_full / rate),
            "sample": f"{n1} rays ({len(tiles)} of {n_tiles} 1024-ray tiles spread over the image) against all "
                      f"{ph.n} photons; gather only ({ms1:.0f} ms); kd+AABB hierarchy build {build_ms:.0f} ms "
                      f"single-threaded, not included in `value` (iteration_value_including_build adds it to a "
                      f"whole-image gather at the measured rate)"}, ms1, n1


def reference_code_available(inp):
    """Can the reference's OWN compiled G-BRE path (oracle/_ref/libgvpm_functor_ref.so: GPhotonMap::build,
    GradientBeamRadianceEstimator, bre->query, VolumeGradientBREQuery; built from /root/reference where that tree exists and
    shipped with the repo snapshot) be timed on this box?  It keeps one light-path record per photon like the reference
    does (~1.3 KB per photon here)."""
    if os.environ.get("GVPM_REFERENCE_ARM", "code") == "port":
        return False, "GVPM_REFERENCE_ARM=port"
    try:
        from oracle import functor_binding as fb
        if not fb.have_ref():
            return False, "oracle/_ref/libgvpm_functor_ref.so absent"
        fb.load()
    except Exception as e:  # noqa: BLE001
        return False, f"reference library does not load: {e}"
    need = 1.6e3 * inp["photons"].n * 1.5
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:  # noqa: BLE001
        avail = None
    if avail is not None and avail < need:
        return False, f"host memory: {avail / 1e9:.0f} GB available, {need / 1e9:.0f} GB wanted"
    return True, ""


def reference_code_arm(args, inp, seconds):
    """The reference's own compiled code on all host cores, on the same bounded sample as cpu_arm (whole 1024-ray tiles
    spread evenly over the image, against ALL photons): kd build and hierarchy once (single-threaded, as compiled here:
    Mitsuba's parallel kd build needs its scheduler), then bre->query + the shift functor per sampled ray on `cores`
    threads (the reference: BlockScheduler over image blocks)."""
    from oracle import binding as ob
    from oracle import functor_binding as fb
    cores = ob.hw_threads()
    ph, rays = inp["photons"], inp["rays"]
    st = inp.setdefault("ref_code", {})
    if "pass" not in st:
        st["pass"] = fb.BrePass(ph, inp["medium"], inp["cfg"], inp["tri"], inp["radius"], threads=cores)
    bp = st["pass"]
    n_tiles = max(1, rays.n // 1024)

    def run(tile_ids, threads=None, want_out=False):
        idx = (np.asarray(tile_ids)[:, None] * 1024 + np.arange(1024)[None, :]).reshape(-1)
        idx = idx[idx < rays.n]
        sub = rays.take(idx)
        out, calls, ms = bp.run(sub, threads=threads or cores, want_out=want_out)
        return sub, out, calls, ms

    pilot_tiles = np.unique(np.linspace(0, n_tiles - 1, num=min(n_tiles, max(8, cores // 4)), dtype=np.int64))
    sub0, _, _, ms0 = run(pilot_tiles)
    rate = sub0.n / max(ms0, 1e-3) * 1e3
    want = int(min(n_tiles, max(len(pilot_tiles), rate * seconds / 1024)))
    tiles = np.unique(np.linspace(0, n_tiles - 1, num=want, dtype=np.int64))
    sub1, _, calls1, ms1 = run(tiles)
    if "single" not in st:     # single-thread figure + agreement with the restated port, once, on a slice of the sample
        k1 = max(2, len(tiles) // max(2 * cores, 1))
        check_tiles = tiles[::max(1, len(tiles) // k1)][:k1]
        subs, outs, _, mss = run(check_tiles, threads=1, want_out=True)
        st["single"] = subs.n / max(mss, 1e-3) * 1e3
        if os.environ.get("GVPM_REFERENCE_CHECK", "1") != "0":
            lib = ob.load() if ob._lib is not None else (ob.prefer_native(), ob.load())[1]
            from gvpm_b200 import _native as N
            cph, cr = ph.as_c(), subs.as_c()
            tree = lib.gvpm_oracle_tree_build(C.byref(cph), ph.n, inp["radius"], 0)
            po = np.zeros(subs.n * 27, dtype=np.float32)
            pms = C.c_double(0)
            tri = inp["tri"]
            for th, key in ((1, "port_single_thread_value"), (cores, "port_value")):
                rc = lib.gvpm_oracle_bre(tree, C.byref(cph), ph.n, C.byref(cr), 0, subs.n, C.byref(inp["medium"]),
                                         C.byref(inp["cfg"]), tri.ctypes.data_as(N.f32p), tri.size // 9, inp["radius"], 0,
                                         th, po.ctypes.data_as(N.f32p), None, None, None, 0, C.byref(pms))
                assert rc >= 0
                st[key] = subs.n / max(pms.value, 1e-3) * 1e3
            st["port_build_ms"] = lib.gvpm_oracle_tree_build_ms(tree)
            lib.gvpm_oracle_tree_free(tree)
            _, _, _, msm = run(check_tiles)
            st["same_rays_value"] = subs.n / max(msm, 1e-3) * 1e3
            po = po.reshape(-1, 27)
            scale = np.abs(outs).max(axis=1, keepdims=True)
            err = np.abs(po - outs) / np.maximum(np.abs(outs), np.where(scale > 0, 1e-3 * scale, 1.0))
            st["port_max_rel_diff"] = float(err.max())
            st["check_rays"] = int(subs.n)
    rate = sub1.n / ms1 * 1e3
    r_full = float(inp.get("rays_full_n", rays.n))
    build_ms = bp.kd_build_ms + bp.hierarchy_ms
    cb = {"value": rate, "unit": "rays/s", "cores": cores, "kind": "reference",
          "flags": "-O2 -ffp-contract=off, SINGLE_PRECISION SPECTRUM_SAMPLES=3 (oracle/Makefile, target functor_ref)",
          "build_ms": build_ms, "kd_build_ms": bp.kd_build_ms, "hierarchy_ms": bp.hierarchy_ms,
          "gather_ms_sample": ms1, "functor_calls_per_ray": float(calls1.mean()), "single_thread_value": st["single"],
          "iteration_value_including_build": r_full / (build_ms * 1e-3 + r_full / rate),
          "sample": f"{sub1.n} rays ({len(tiles)} of {n_tiles} 1024-ray tiles spread over the image) against all {ph.n} "
                    f"photons, on the reference's own compiled code (GPhotonMap::build, GradientBeamRadianceEstimator, "
                    f"bre->query, VolumeGradientBREQuery: oracle/_ref/libgvpm_functor_ref.so); gather only ({ms1:.0f} ms); "
                    f"kd build {bp.kd_build_ms:.0f} ms + hierarchy {bp.hierarchy_ms:.0f} ms single-threaded, not included in "
                    f"`value`"}
    if "port_value" in st:
        cb["restated_port_on_same_rays"] = {
            "rays": st["check_rays"], "reference_value": st["same_rays_value"], "port_value": st["port_value"],
            "reference_single_thread_value": st["single"], "port_single_thread_value": st["port_single_thread_value"],
            "port_build_ms": st["port_build_ms"], "max_rel_diff": st["port_max_rel_diff"]}
    return cb, ms1, sub1.n


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import __graft_entry__ as ge
    ge.build_cpu_libs()
    inp = make_inputs(args, 0, 1, pin=False)
    inp["full_rays"] = inp["rays"]
    per = max(2.0, min(args.cpu_seconds, 120.0 / max(1, args.steps + args.warmup)))
    vals = []
    cb = None
    use_code, why_not = reference_code_available(inp)
    for i in range(args.warmup + args.steps):
        if use_code:
            try:
                cb, ms, n = reference_code_arm(args, inp, per)
            except Exception as e:  # noqa: BLE001 - the arm must still print its line: fall back to the restated port
                use_code, why_not = False, f"reference code failed: {type(e).__name__}: {e}"
                inp.pop("ref_code", None)
                vals = []
        if not use_code:
            cb, ms, n = cpu_arm(args, inp, per)
            cb["reference_code_not_timed"] = why_not
        if i >= args.warmup:
            vals.append((n, ms))
    if not vals:
        vals.append((n, ms))
    n_tot = sum(v[0] for v in vals)
    ms_tot = sum(v[1] for v in vals)
    value = n_tot / ms_tot * 1e3
    cb["value"] = value
    line = {"impl": "reference", "metric": "camera-ray gathers/sec (primal+4 gradients)", "value": value,
            "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_tot / max(1, len(vals)), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, inp, max(1, args.gpus)), "cpu_baseline": cb,
            "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def rebalance_bands(args, inp, ctx, stream, rank, world):
    """Untimed pilot iteration (what a progressive integrator knows from its previous iteration): every rank gathers its
    equal-size bands once with neighbour counts, the per-block costs (contributing pairs + a per-ray term) are summed
    over the ranks and the bands are re-cut into runs of equal COST (shard.band_owner_weighted).  The photon density of
    the scene is centre-weighted: with equal-size bands the busiest rank of 8 carries ~40 % more than the average."""
    import torch
    import torch.distributed as dist
    from gvpm_b200 import records as R, shard
    if shard_mode(world) != "band" or os.environ.get("GVPM_BALANCE", "1") == "0" or not prune_build(world):
        return None
    w, h, n_ph = inp["w"], inp["h"], inp["n_ph"]
    ctx.photon_staging_select(0)
    ptr, nbytes = ctx.photon_staging(n_ph)
    st = torch.as_tensor(DevView(ptr, nbytes), device="cuda")
    with torch.cuda.stream(stream):
        if rank == 0:
            ctx.upload_photons(inp["photons"])
        dist.broadcast(st, src=0)
        ctx.upload_rays(inp["rays"])
        ctx.build_points_for_rays(inp["radius"], want_kept=False)
    out, counts = ctx.gather_bre()
    del out
    rays = inp["rays"]
    n_tiles = ((w + 31) // 32) * ((h + 31) // 32)
    t = shard.block_index(rays.px, rays.py, h)
    lam = float(os.environ.get("GVPM_BALANCE_RAY_COST", "3"))      # a ray costs about as much as three contributing pairs
    cost = np.bincount(t, weights=counts[:, 1].astype(np.float64) + lam, minlength=n_tiles)
    cost_t = torch.from_numpy(cost).cuda()
    dist.all_reduce(cost_t)
    cost = cost_t.cpu().numpy()
    full = inp["full_rays"]
    owner = shard.band_owner_weighted(full.px, full.py, w, h, world, cost, band_cycles())
    per_rank = np.array([cost[np.unique(shard.block_index(full.px[owner == r], full.py[owner == r], h))].sum() for r in range(world)])
    before = shard.band_owner(full.px, full.py, w, h, world, band_cycles())
    per_before = np.array([cost[np.unique(shard.block_index(full.px[before == r], full.py[before == r], h))].sum() for r in range(world)])
    sub = full.take(np.nonzero(owner == rank)[0])
    rays2 = R.RaySet(sub.n, **inp["alloc"](R._RAY_FIELDS, sub.n))
    for name, _, _ in R._RAY_FIELDS:
        getattr(rays2, name)[:] = getattr(sub, name)
    inp["rays"] = rays2
    del st
    return {"cost_model": f"contributing pairs + {lam:g} per ray, per 32x32 block, from one pilot iteration (untimed)",
            "max_over_mean_equal_blocks": float(per_before.max() / per_before.mean()),
            "max_over_mean_equal_cost": float(per_rank.max() / per_rank.mean())}


def workload_config(args, inp, world):
    return {"workload": f"{args.workload}: {inp['w']}x{inp['h']} homogeneous-medium Cornell box, "
                        f"{inp['n_ph']} photons/iteration, gvpm G-BRE 3D kernel, mixed shift, area MIS, pathSet",
            "rays": inp["rays_full_n"], "photons": inp["n_ph"], "initialScaleVolume": inp["scale"],
            "radius": inp["radius"],
            "parallelism": (f"32x32 gather blocks in {band_cycles()} cost-balanced column bands per GPU over {world} GPU(s), "
                            "every GPU holds 1/N of the photon set and sends each photon to the GPUs whose bands can reach "
                            "it, each perspective grid built over what its GPU received, results collected on rank 0"
                            if shard_mode(world) == "band" else
                            f"image tiles (32x32) round-robin over {world} GPU(s), photon set broadcast, results "
                            "gathered to rank 0"),
            "l2": (f"photon records {inp['n_ph'] * 128 / 1e9:.2f} GB + rays {inp['rays_full_n'] * 320 / 1e9:.2f} GB per step "
                   "against a 126 MB L2: " + ("inputs larger than L2, no flush needed"
                                              if inp["n_ph"] * 128 + inp["rays_full_n"] * 320 > 4 * 126e6
                                              else "SMALLER than 4x L2 - parity-sized workload, not a bench configuration"))}


def diag_phases(v):
    """GVPM_BENCH_DIAG=1: isolated timings of the pieces of a step (max over ranks, ms), to stderr."""
    import torch
    import torch.distributed as dist
    world, rank, stream, ctx = v["world"], v["rank"], v["stream"], v["ctx"]
    views, pg, comm = v["views"], v["pg_photons"], v["comm"]
    res = {}

    def run(name, fn, reps=5):
        fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / reps], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        res[name] = round(float(ms.item()), 3)

    if world > 1 and pg is not None:
        def ag13():
            ws = [dist.all_gather_into_tensor(w, m, group=pg, async_op=True) for w, m in views[1]]
            for w in ws:
                w.wait()
        run("allgather_13_calls", ag13)

        def agc():
            with dist._coalescing_manager(group=pg, device=torch.device("cuda", v["local"]), async_ops=True) as cm:
                for w, m in views[1]:
                    dist.all_gather_into_tensor(w, m, group=pg)
            cm.wait()
        try:
            run("allgather_coalesced", agc)
        except Exception as e:  # noqa: BLE001
            res["allgather_coalesced"] = f"failed: {type(e).__name__}: {e}"[:200]
        big = v["stage_t"][1]
        nb = (big.numel() // world // 256) * 256
        run("allgather_1_call_same_bytes", lambda: dist.all_gather_into_tensor(big[:nb * world], big[rank * nb:(rank + 1) * nb], group=pg))
    if world > 1:
        run("result_gather", lambda: dist.gather(v["out_dev"], v["gathered"], dst=0))

    def up():
        ctx.photon_staging_select(1)
        ctx.upload_photons_slice(v["host_slice"], v["n_ph"], v["s_begin"], stream=v["h2d"].cuda_stream)
    run("h2d_photon_slice", up)

    def bld():
        ctx.photon_staging_select(0)
        ctx.photon_staging(v["n_ph"])
        with torch.cuda.stream(stream):
            ctx.build_points(v["inp"]["radius"])
    run("build", bld)

    def gh():
        with torch.cuda.stream(stream):
            ctx.gather_bre_host(v["rays"], v["out_host"][:v["n_local"] * 27])
    run("gather_bre_host", gh)

    def gi():
        with torch.cuda.stream(stream):
            ctx.gather_bre_into(v["out_dev"].data_ptr(), None)
    run("gather_bre_into", gi)
    if rank == 0:
        print("DIAG " + json.dumps(res), file=sys.stderr, flush=True)



# --------------------------------------------------------------------------------------------
# cfg2 / cfg3 / cfg4 / beams1080: the other gathers of the path, same JSON contract.  A step = accel build + gather of
# every camera ray; `value` from device-resident raw arrays, `e2e` through upload_* + build_* + gather_* with pinned
# host arrays in and out.  N > 1: the 32x32 ray blocks are dealt to the ranks in contiguous runs, the primitive set is
# replicated (every rank holds / uploads all of it), results are gathered to rank 0.
def technique_inputs(args, rank, world):
    import gvpm_b200 as g
    from gvpm_b200 import records as R
    tech, w, h, n_prim, scale = TECHNIQUES[args.workload]
    if args.photons:
        n_prim = args.photons
    if args.scale:
        scale = args.scale
    seed = 0xC0FFEE + {"cfg2": 2, "cfg3": 3, "cfg4": 4, "beams1080": 6}[args.workload]
    threads = max(1, min(32, (os.cpu_count() or 8) // max(1, world)))
    medium = g.make_medium()
    d = dict(tech=tech, w=w, h=h, n_prim=n_prim, scale=scale, medium=medium, tri=g.synth_occluders(),
             radius=g.bre_radius(scale), cfg=g.make_config(w, h), nb=40)
    if tech == "planes":
        full = g.synth_rays(w, h, seed=seed + 1, block=-32, cam_dist=-0.05, cover=0.45)   # sensor inside the medium
    else:
        full = g.synth_rays(w, h, seed=seed + 1, block=-32)
    per = ((full.n + world - 1) // world + 1023) // 1024 * 1024
    lo, hi = min(full.n, rank * per), min(full.n, (rank + 1) * per)
    d["rays"] = full.take(np.arange(lo, hi)) if world > 1 else full
    d["rays_full_n"] = full.n
    d["full_rays"] = full if rank == 0 else None
    if tech == "vpm":
        d["photons"], d["n_paths"] = g.synth_photons(n_prim, medium, seed=seed, threads=threads)
        rad = np.full(d["rays"].n, d["radius"], dtype=np.float32)
        d["samples"] = g.synth_vpm_samples(d["rays"], medium, rad, nb_camera_samples=d["nb"], seed=seed + 2)
    elif tech == "beams":
        d["beams"], d["n_paths"] = R.synth_beams(n_prim, medium, seed=seed, threads=threads)
    else:
        beams, d["n_paths"] = R.synth_beams(n_prim, medium, seed=seed, threads=threads)
        planes = R.synth_planes(beams, medium, seed=seed + 7)
        o = planes.view("origin")   # LASER-style: collimated 0.02-wide emitter (SURVEY.md 8d)
        o[:, 0] = 0.5 + (o[:, 0] - 0.5) * 0.02
        planes.length1[:] *= 0.05
        d["planes"] = planes
    return d


def pin_soa(soa):
    """copy of a records SoA in page-locked memory (the e2e leg's source)"""
    import torch
    keep, arrs = [], {}
    for name, dt, wd in soa.FIELDS:
        a = getattr(soa, name)
        t = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=True)
        v = t.numpy().view(dt)
        v[:] = a.reshape(-1)
        keep.append(t)
        arrs[name] = v
    out = type(soa)(soa.n, **arrs)
    out._keep = keep
    return out


TECH_TEXT = {"vpm": "gvpm G-VPM point photons, uniform 3D kernel, 40 camera distance samples per pixel",
             "beams": "gvpm G-Beams 3D kernel (photon beams x camera beams)",
             "planes": "gvpm G-Planes 0D kernel, LASER-style sheet emitter, sensor inside the medium"}
PRIM_BYTES = {"vpm": 112, "beams": 128, "planes": 64}   # SURVEY.md 8(d) record sizes


def technique_config(args, d, world):
    prim = {"vpm": "photons", "beams": "beams", "planes": "planes"}[d["tech"]]
    fits = d["n_prim"] * PRIM_BYTES[d["tech"]] + d["rays_full_n"] * 320
    return {"workload": f"{args.workload}: {d['w']}x{d['h']} homogeneous-medium Cornell box, {d['n_prim']} {prim}/iteration, "
                        f"{TECH_TEXT[d['tech']]}, mixed shift, area MIS, pathSet",
            "rays": d["rays_full_n"], prim: d["n_prim"], "initialScaleVolume": d["scale"], "radius": d["radius"],
            "parallelism": f"32x32 ray blocks in contiguous runs over {world} GPU(s), {prim} replicated, results gathered to rank 0",
            "l2": f"records {d['n_prim'] * PRIM_BYTES[d['tech']] / 1e6:.0f} MB + rays {d['rays_full_n'] * 320 / 1e6:.0f} MB per step "
                  "against a 126 MB L2: " + ("larger than L2, no flush" if fits > 2 * 126e6 else
                                             "comparable to L2: a 256 MB buffer is written between timed steps (L2 flush)")}


def technique_cpu_arm(args, d, seconds):
    """the oracle restatement of the same gather on all host cores, on a bounded sample of whole 1024-ray tiles"""
    from oracle import binding as ob
    if "oracle_flags" not in d:      # BASELINE.md §2: -O3 -march=native, built on the box that is timed (untimed here)
        d["oracle_flags"] = ob.prefer_native() if ob._lib is None else "as loaded"
    cores = ob.hw_threads()
    rays = d["full_rays"] if d.get("full_rays") is not None else d["rays"]
    n_tiles = max(1, rays.n // 1024)
    tech = d["tech"]

    def run(n_t):
        tiles = np.unique(np.linspace(0, n_tiles - 1, num=max(1, n_t), dtype=np.int64))
        idx = (tiles[:, None] * 1024 + np.arange(1024)[None, :]).reshape(-1)
        idx = idx[idx < rays.n]
        sub = rays.take(idx)
        t0 = time.perf_counter()
        if tech == "vpm":
            import gvpm_b200 as g
            rad = np.full(sub.n, d["radius"], dtype=np.float32)
            smp = g.synth_vpm_samples(sub, d["medium"], rad, nb_camera_samples=d["nb"], seed=11)
            t0 = time.perf_counter()
            r = ob.vpm_gather(d["photons"], sub, smp, d["medium"], d["cfg"], d["tri"], d["nb"], mode="kdtree", threads=cores)
            how = "kd-tree range queries (reference structure), kd build included"
        elif tech == "beams":
            r = ob.beams_gather(d["beams"], sub, d["medium"], d["cfg"], d["tri"], d["radius"], threads=cores)
            how = "BRUTE FORCE over all beams (the oracle has no sub-beam BVH: slower than the reference's traversal)"
        else:
            r = ob.planes_gather(d["planes"], sub, d["medium"], d["cfg"], mode="brute", threads=cores)
            how = "brute force over all planes"
        wall = (time.perf_counter() - t0) * 1e3
        ms = max(r.gather_ms, 1e-3)
        return sub.n, ms, wall, len(tiles), how

    n0, ms0, wall0, _, _ = run(1)
    want = int(min(n_tiles, max(1, seconds * 1e3 / max(wall0, 1e-3))))
    n1, ms1, wall1, nt, how = run(want)
    return {"value": n1 / ms1 * 1e3, "unit": "rays/s", "cores": cores, "kind": "port",
            "sample": f"{n1} rays ({nt} of {n_tiles} 1024-ray tiles spread over the image) against all {d['n_prim']} "
                      f"primitives; {how}; gather {ms1:.0f} ms (wall {wall1:.0f} ms)"}, ms1, n1


def technique_reference_code_arm(args, d, seconds):
    """The reference's own compiled code for this technique on all host cores (oracle/_ref/libgvpm_functor_ref.so): its
    acceleration structure (SubBeamBVH / PhotonPlaneBVH / PointKDTree range query) built once, then its traversal + shift
    functor on a bounded sample of whole 1024-ray tiles spread over the image."""
    from oracle import binding as ob
    from oracle import functor_binding as fb
    cores = ob.hw_threads()
    rays = d["full_rays"] if d.get("full_rays") is not None else d["rays"]
    n_tiles = max(1, rays.n // 1024)
    tech = d["tech"]
    st = d.setdefault("ref_code", {})
    if "pass" not in st:
        if tech == "vpm":
            st["pass"] = fb.TechniquePass("vpm", d["photons"], d["medium"], d["cfg"], tri=d["tri"], threads=cores)
            st["what"] = "GPhotonMap::build + evaluate (PointKDTree range query) + VolumeGradientDistanceQuery"
        elif tech == "beams":
            st["pass"] = fb.TechniquePass("beams", d["beams"], d["medium"], d["cfg"], tri=d["tri"], radius=d["radius"])
            st["what"] = "SubBeamBVH<LTPhotonBeam> + BeamGradRadianceQuery"
        else:
            st["pass"] = fb.TechniquePass("planes", d["planes"], d["medium"], d["cfg"])
            st["what"] = "PhotonPlaneBVH<LTPhotonPlane> + PlaneGradRadianceQuery"
    tp = st["pass"]

    def run(n_t):
        tiles = np.unique(np.linspace(0, n_tiles - 1, num=max(1, n_t), dtype=np.int64))
        idx = (tiles[:, None] * 1024 + np.arange(1024)[None, :]).reshape(-1)
        idx = idx[idx < rays.n]
        sub = rays.take(idx)
        smp = None
        if tech == "vpm":
            import gvpm_b200 as g
            rad = np.full(sub.n, d["radius"], dtype=np.float32)
            smp = g.synth_vpm_samples(sub, d["medium"], rad, nb_camera_samples=d["nb"], seed=11)
        t0 = time.perf_counter()
        _, ms = tp.run(sub, threads=cores, samples=smp, nb_camera_samples=d.get("nb", 0), want_out=False)
        return sub.n, max(ms, 1e-3), (time.perf_counter() - t0) * 1e3, len(tiles)

    # pilot on tiles spread over the image (the cost per ray follows the primitive density: a corner tile says nothing)
    n_pilot = min(n_tiles, 8)
    _, _, wall0, _ = run(n_pilot)
    want = int(min(n_tiles, max(n_pilot, seconds * 1e3 / max(wall0 / n_pilot, 1e-3))))
    n1, ms1, wall1, nt = run(want) if want > n_pilot else run(n_pilot)
    return {"value": n1 / ms1 * 1e3, "unit": "rays/s", "cores": cores, "kind": "reference",
            "flags": "-O2 -ffp-contract=off, SINGLE_PRECISION SPECTRUM_SAMPLES=3 (oracle/Makefile, target functor_ref)",
            "build_ms": tp.build_ms,
            "sample": f"{n1} rays ({nt} of {n_tiles} 1024-ray tiles spread over the image) against all {d['n_prim']} "
                      f"primitives, on the reference's own compiled code ({st['what']}: "
                      f"oracle/_ref/libgvpm_functor_ref.so); gather {ms1:.0f} ms (wall {wall1:.0f} ms); structure build "
                      f"{tp.build_ms:.0f} ms single-threaded, not included in `value`"}, ms1, n1


def technique_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import __graft_entry__ as ge
    ge.build_cpu_libs()
    d = technique_inputs(args, 0, 1)
    per = max(2.0, min(args.cpu_seconds, 120.0 / max(1, args.steps + args.warmup)))
    vals, cb = [], None
    use_code, why_not = False, "GVPM_REFERENCE_ARM=port"
    if os.environ.get("GVPM_REFERENCE_ARM", "code") != "port":
        try:
            from oracle import functor_binding as fb
            use_code = fb.have_ref() and fb.load() is not None
            why_not = "" if use_code else "oracle/_ref/libgvpm_functor_ref.so absent"
        except Exception as e:  # noqa: BLE001
            use_code, why_not = False, f"reference library does not load: {e}"
    for i in range(args.warmup + args.steps):
        if use_code:
            try:
                cb, ms, n = technique_reference_code_arm(args, d, per)
            except Exception as e:  # noqa: BLE001 - fall back to the restated port
                use_code, why_not = False, f"reference code failed: {type(e).__name__}: {e}"
                d.pop("ref_code", None)
                vals = []
        if not use_code:
            cb, ms, n = technique_cpu_arm(args, d, per)
            cb["reference_code_not_timed"] = why_not
        if i >= args.warmup:
            vals.append((n, ms))
    if not vals:
        vals.append((n, ms))
    n_tot, ms_tot = sum(v[0] for v in vals), sum(v[1] for v in vals)
    value = n_tot / ms_tot * 1e3
    cb["value"] = value
    print(json.dumps({"impl": "reference", "metric": "camera-ray gathers/sec (primal+4 gradients)", "value": value,
                      "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": ms_tot / max(1, len(vals)), "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": technique_config(args, d, args.gpus), "cpu_baseline": cb,
                      "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def technique_main(args):
    if args.impl == "reference":
        return technique_reference(args)
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    from gvpm_b200.api import Context
    from gvpm_b200 import _native as NAT
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: gvpm_b200 has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of a one-GPU run")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        ge.build_cpu_libs()
    if world > 1:
        dist.barrier()
    d = technique_inputs(args, rank, world)
    tech = d["tech"]
    ctx = Context(local)
    ctx.set_medium(d["medium"])
    ctx.set_config(d["cfg"])
    ctx.set_occluders(d["tri"])
    stream = torch.cuda.ExternalStream(ctx.stream(), device=local)
    rays = pin_soa(d["rays"])
    n_local = rays.n
    prim = pin_soa(d["photons"] if tech == "vpm" else d["beams"] if tech == "beams" else d["planes"])
    samples = pin_soa(d["samples"]) if tech == "vpm" else None
    out_t, out_host = pinned(max(1, n_local) * 27, torch.float32)
    mvol_t, mvol_host = pinned(max(1, n_local), torch.int32)
    n_pad = torch.tensor([n_local], device="cuda", dtype=torch.int64)
    if world > 1:
        dist.all_reduce(n_pad, op=dist.ReduceOp.MAX)
    n_pad = int(n_pad.item())
    gathered = [torch.empty(n_pad * 27, device="cuda", dtype=torch.float32) for _ in range(world)] \
        if (world > 1 and rank == 0) else None
    send = torch.zeros(n_pad * 27, device="cuda", dtype=torch.float32) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def upload_prims():
        if tech == "vpm":
            ctx.upload_photons(prim)
        elif tech == "beams":
            ctx.upload_beams(prim)
        else:
            ctx.upload_planes(prim)

    def build():
        if tech == "vpm":
            ctx.build_points(d["radius"])
        elif tech == "beams":
            ctx.build_beams(d["radius"])
        else:
            ctx.build_planes()

    def gather_device():
        """-> device pointers (out [n_rays*27] float32, G-VPM: mvol [n_rays] uint32, else None)"""
        if tech == "vpm":
            return ctx.gather_vpm_device(d["nb"])
        if tech == "beams":
            return ctx.gather_beams_device(False)[0], None
        return ctx.gather_planes_device(False)[0], None

    def collect(ptr):
        if world == 1:
            return
        with torch.cuda.stream(stream):
            view = torch.as_tensor(DevView(ptr, n_local * 27 * 4), device="cuda").view(torch.float32)
            send[:n_local * 27].copy_(view)
            dist.gather(send, gathered, dst=0)

    last_out = [None]     # device pointers of the last resident gather's outputs

    def step_resident(k):
        with torch.cuda.stream(stream):
            flush.fill_(k & 255)          # L2 flush between timed steps (untimed work would be nicer; it is 256 MB at HBM speed: ~40 us)
        build()
        last_out[0] = gather_device()
        collect(last_out[0][0])

    def step_e2e(k):
        upload_prims()
        build()
        ctx.upload_rays(rays)
        if tech == "vpm":
            ctx.upload_vpm_samples(samples)
            ctx.gather_vpm(d["nb"], out=out_host[:n_local * 27], mvol=mvol_host[:n_local].view(np.uint32), sample_counts=False)
        elif tech == "beams":
            ctx.gather_beams(counts=False, out=out_host[:n_local * 27])
        else:
            ctx.gather_planes(counts=False, out=out_host[:n_local * 27])

    # untimed set-up: everything resident
    upload_prims()
    build()
    ctx.upload_rays(rays)
    if tech == "vpm":
        ctx.upload_vpm_samples(samples)
    ctx.sync()

    def timed(fn, steps, warmup):
        for k in range(warmup):
            fn(k)
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        e0.record(stream)
        for k in range(warmup, warmup + steps):
            fn(k)
        e1.record(stream)
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), ctx.launch_count() - l0

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    W = max(3, args.warmup)
    ms_total, launches = timed(step_resident, args.steps, W)
    if args.dump_outputs:   # before the untimed gathers below overwrite the output buffers
        out_ptr, mvol_ptr = last_out[0]
        dump_gather(args.dump_outputs, torch.as_tensor(DevView(out_ptr, n_local * 27 * 4), device="cuda").view(torch.float32),
                    rays, None if mvol_ptr is None else
                    torch.as_tensor(DevView(mvol_ptr, n_local * 4), device="cuda").view(torch.int32))
    ms_e2e, _ = timed(step_e2e, args.steps, W)
    clocks = sampler.stop() if rank == 0 else None
    # phases + the roofline numerator H (neighbour pairs) from untimed runs
    kt, kd = [], []
    for _ in range(3):
        build()
        gather_device()
        kt.append(ctx.last_timings())
        kd.append(ctx.last_gather_detail())
    build_ms, gather_ms = float(np.mean([k[0] for k in kt])), float(np.mean([k[1] for k in kt]))
    trav_ms, shade_ms, n_pairs = float(np.mean([k[0] for k in kd])), float(np.mean([k[1] for k in kd])), int(kd[-1][2])
    if tech == "vpm":
        _, mv, sc = ctx.gather_vpm(d["nb"])
        H = int(sc[:, 0].astype(np.int64).sum())
    elif tech == "beams":
        _, cnt = ctx.gather_beams(counts=True)
        H = int(cnt[:, 0].astype(np.int64).sum())
    else:
        _, cnt = ctx.gather_planes(counts=True)
        H = int(cnt[:, 0].astype(np.int64).sum())
    stats = torch.tensor([float(H), 0.0], device="cuda", dtype=torch.float64)
    mx = torch.tensor([build_ms, gather_ms, trav_ms, shade_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(stats)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    if rank == 0:
        R_ = d["rays_full_n"]
        H = int(stats[0].item())
        build_ms, gather_ms, trav_ms, shade_ms = [float(x) for x in mx.tolist()]
        peak, src = peaks()
        rec = PRIM_BYTES[tech]
        per_ray = 428.0 + (d["nb"] * 32.0 if tech == "vpm" else 0.0)
        alg = (R_ / world) * per_ray + (H / world) * rec
        achieved = alg / (gather_ms * 1e-3) / 1e9
        kern = {"vpm": "k_vpm_traverse + k_vpm_shade", "beams": "k_beam_traverse + k_beam_shade", "planes": "k_plane_gather"}[tech]
        h2d = prim.nbytes() + rays.nbytes() * world + (samples.nbytes() * world if samples is not None else 0)
        line = {"metric": "camera-ray gathers/sec (primal+4 gradients)", "value": R_ * args.steps / (ms_total * 1e-3),
                "unit": "rays/s" if tech != "vpm" else "pixels/s", "n_gpus": world, "steps": args.steps, "warmup": W,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": technique_config(args, d, world), "clocks": clocks,
                "e2e": {"value": R_ * args.steps / (ms_e2e * 1e-3), "unit": "rays/s" if tech != "vpm" else "pixels/s",
                        "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(R_ * 27 * 4),
                        "note": "upload_* + build_* + upload_rays + gather_* with pinned host arrays, serial (no overlap of the copies with the kernels yet)"},
                "gpu_launches": int(launches), "native_lib": NAT.LIB_PATH,
                "roofline": {"bound": "hbm", "kernel": kern, "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": None, "peak_source": src,
                             "algorithmic_bytes_per_launch": alg, "kernel_ms": gather_ms, "traverse_ms": trav_ms,
                             "shade_ms": shade_ms, "neighbours_H": H, "pairs_shaded": n_pairs,
                             "note": f"SURVEY 8(d): R*{per_ray:.0f} + H*{rec} bytes over the gather kernels; H = accepted (ray, primitive) pairs"},
                "phases_ms": {"build": build_ms, "gather": gather_ms, "traverse": trav_ms, "shade": shade_ms},
                "light_paths": d["n_paths"]}
        if world == 1 and not args.no_cpu_baseline:
            # the reference's own compiled structures + functors where that library is present (its sub-beam / plane BVHs,
            # not the port's brute force), else the restated port
            cb = None
            if os.environ.get("GVPM_REFERENCE_ARM", "code") != "port":
                try:
                    from oracle import functor_binding as fb
                    if fb.have_ref():
                        cb, _, _ = technique_reference_code_arm(args, d, args.cpu_seconds)
                except Exception as e:  # noqa: BLE001
                    cb = None
                    d.pop("ref_code", None)
                    line["cpu_baseline_reference_code_failed"] = f"{type(e).__name__}: {e}"
            if cb is None:
                cb, _, _ = technique_cpu_arm(args, d, args.cpu_seconds)
            line["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    del out_t, mvol_t, gathered, send, flush, stream, n_pad, stats, mx
    prim._keep = rays._keep = None
    if samples is not None:
        samples._keep = None
    import gc
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    try:
        torch._C._host_emptyCache()
    except Exception:  # noqa: BLE001
        pass
    ctx.close()

# --------------------------------------------------------------------------------------------
def poisson_main(args):
    """`--workload poisson1080 | poisson720 | poisson1080_l1`: one screened-Poisson reconstruction per step (host arrays in
    and out through gvpm_poisson_solve, as the plugin calls it).  The reference arm is the reference's OWN solver compiled
    from /root/reference (oracle/_ref/libgvpm_poisson_ref.so, OpenMP backend on the host cores): cpu_baseline.kind
    "reference"; where its CUDA backend was built too (libgvpm_poisson_ref_cuda.so) the GPU run times it on the same
    device (`reference_cuda_ms`).  Same calls as tools/time_poisson.py."""
    import importlib.util
    if int(os.environ.get("RANK", "0")) != 0:
        return
    w, h, preset = POISSON[args.workload]
    spec = importlib.util.spec_from_file_location("mpg", os.path.join(ROOT, "tests", "golden", "make_poisson_golden.py"))
    G = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(G)
    from oracle import poisson_ref as pr     # checker / reference arm, never the product path
    _, tp, dx, dy, direct = G.images(h, w, 11)
    config = {"workload": f"{args.workload}: screened-Poisson reconstruction ({preset}) of a synthetic {w}x{h} gradient-domain "
                          f"image set (throughput, dx, dy, direct), host arrays in and out", "pixels": w * h, "preset": preset}
    base = {"metric": "reconstructed pixels/sec (screened Poisson)", "unit": "pixels/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config}

    def reference_cpu(reps):
        ts, out = [], None
        for _ in range(reps):
            t0 = time.perf_counter()
            out = pr.solve(tp, dx, dy, direct, backend="OpenMP", **pr.preset(preset))
            ts.append((time.perf_counter() - t0) * 1e3)
        return float(np.mean(ts)), out

    if args.impl == "reference":
        if not pr.available():
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libgvpm_poisson_ref.so absent"}))
            return
        if args.warmup:
            reference_cpu(args.warmup)
        ms, _ = reference_cpu(args.steps)
        value = w * h / (ms * 1e-3)
        cb = {"value": value, "unit": "pixels/s", "cores": os.cpu_count(), "kind": "reference",
              "sample": f"whole {w}x{h} reconstruction, the reference's own poisson::Solver (OpenMP backend), {ms:.0f} ms"}
        print(json.dumps(dict(base, impl="reference", value=value, ms_per_step=ms, cpu_baseline=cb,
                              e2e={"value": value, "unit": "pixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})))
        return
    from gvpm_b200.api import Context
    ctx = Context(0)
    W = max(3, args.warmup)
    for _ in range(W):
        rec = ctx.poisson_solve(tp, dx, dy, direct, preset=preset)
    clocks = ClockSampler(0)
    clocks.start()
    dev_ms, wall = [], []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        rec = ctx.poisson_solve(tp, dx, dy, direct, preset=preset)
        wall.append((time.perf_counter() - t0) * 1e3)
        dev_ms.append(ctx.last_poisson_ms())
    ck = clocks.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"reconstruction": rec})
    ms, wall_ms = float(np.mean(dev_ms)), float(np.mean(wall))
    nbytes = int(tp.nbytes + dx.nbytes + dy.nbytes + direct.nbytes)
    line = dict(base, value=w * h / (ms * 1e-3), ms_per_step=ms, warmup=W, clocks=ck,
                e2e={"value": w * h / (wall_ms * 1e-3), "unit": "pixels/s", "h2d_bytes_per_step": nbytes,
                     "d2h_bytes_per_step": int(rec.nbytes), "ms_per_step": wall_ms},
                timing="value: CUDA events inside gvpm_poisson_solve (copies included); e2e: wall clock around the call")
    if not args.no_cpu_baseline and pr.available():
        rms, want = reference_cpu(1)
        line["cpu_baseline"] = {"value": w * h / (rms * 1e-3), "unit": "pixels/s", "cores": os.cpu_count(), "kind": "reference",
                                "sample": f"one whole {w}x{h} reconstruction, the reference's own poisson::Solver "
                                          f"(OpenMP backend), {rms:.0f} ms"}
        line["max_rel_err_vs_reference"] = float(np.abs(rec.astype(np.float64) - want).max() / np.abs(want).max())
    if pr.cuda_available():
        pr.solve(tp, dx, dy, direct, backend="CUDA", **pr.preset(preset))       # warm-up (context, allocations)
        ts = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            got = pr.solve(tp, dx, dy, direct, backend="CUDA", **pr.preset(preset))
            ts.append((time.perf_counter() - t0) * 1e3)
        line["reference_cuda_ms"] = float(np.mean(ts))
        line["vs_reference_cuda"] = line["reference_cuda_ms"] / wall_ms
        line["max_rel_err_vs_reference_cuda"] = float(np.abs(rec.astype(np.float64) - got).max() / np.abs(got).max())
    try:
        line["gpu_launches"] = int(ctx.launch_count())     # kernels this context launched (warm-up included)
    except Exception:  # noqa: BLE001
        pass
    print(json.dumps(line), flush=True)
    ctx.close()


def main():
    args = parse()
    if args.workload in POISSON:
        return poisson_main(args)
    if args.workload in TECHNIQUES:
        return technique_main(args)
    if args.impl == "reference":
        return reference_main(args)
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    from gvpm_b200.api import Context

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: gvpm_b200 has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of a one-GPU run")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        ge.build_cpu_libs()
    if world > 1:
        dist.barrier()

    inp = make_inputs(args, rank, world)
    ctx = Context(local)
    ctx.set_medium(inp["medium"])
    ctx.set_config(inp["cfg"])
    ctx.set_occluders(inp["tri"])
    if world > 1:
        ctx.set_view_direction((0.0, 0.0, 1.0))   # the synthetic sensor looks down +z: one projection plane for all ranks
    stream = torch.cuda.ExternalStream(ctx.stream(), device=local)
    n_ph = inp["n_ph"]
    balance = rebalance_bands(args, inp, ctx, stream, rank, world) if world > 1 else None
    rays = inp["rays"]
    n_local = rays.n
    # result buffers (device): own shard; rank 0 also the gathered image
    counts_max = torch.tensor([n_local], device="cuda", dtype=torch.int64)
    if world > 1:
        dist.all_reduce(counts_max, op=dist.ReduceOp.MAX)
    n_pad = int(counts_max.item())
    with torch.cuda.stream(stream):
        out_dev = torch.zeros(n_pad * 27, device="cuda", dtype=torch.float32)
        cnt_dev = torch.zeros(n_pad * 2, device="cuda", dtype=torch.int32)
        gathered = [torch.empty_like(out_dev) for _ in range(world)] if (world > 1 and rank == 0) else None
    out_host_t, out_host = pinned((n_pad * 27) * (world if rank == 0 else 1), torch.float32)

    # ---- photon staging: two buffers (double buffering), torch views for NCCL ----------------------------------
    assert n_ph % world == 0, "the photon set is split evenly over the ranks"
    n_slice, s_begin = n_ph // world, rank * (n_ph // world)
    stage_t = []
    for b in (0, 1):
        ctx.photon_staging_select(b)
        ptr, nbytes = ctx.photon_staging(n_ph)
        stage_t.append(torch.as_tensor(DevView(ptr, nbytes), device="cuda"))
    f_off, f_elt = ctx.photon_staging_layout(n_ph)

    def field_views(b):
        """per field: (whole array, this rank's slice) as byte views of staging buffer b"""
        out = []
        for off, elt in zip(f_off, f_elt):
            whole = stage_t[b][off:off + n_ph * elt]
            out.append((whole, whole[s_begin * elt:(s_begin + n_slice) * elt]))
        return out
    views = [field_views(0), field_views(1)]

    # untimed set-up: rank 0 uploads the set, broadcast, every rank keeps its slice in pinned host memory (the e2e
    # leg's source) and both staging buffers hold the rank's slice (the value leg's resident input)
    ctx.photon_staging_select(0)
    ctx.photon_staging(n_ph)
    with torch.cuda.stream(stream):
        if rank == 0:
            ctx.upload_photons(inp["photons"])
        if world > 1:
            dist.broadcast(stage_t[0], src=0)
        stage_t[1].copy_(stage_t[0])
        ctx.upload_rays(rays)
    ctx.sync()
    torch.cuda.synchronize()
    from gvpm_b200 import records as REC
    host_fields, keep_host = {}, []
    for (name, dt, wd), (whole, mine) in zip(REC._PHOTON_FIELDS, views[0]):
        t = torch.empty(mine.numel(), dtype=torch.uint8, pin_memory=True)
        t.copy_(mine)
        keep_host.append(t)
        host_fields[name] = t.numpy().view(dt)
    torch.cuda.synchronize()
    host_slice = REC.PhotonSet(n_slice, **host_fields)

    comm = torch.cuda.Stream(device=local)      # issues the photon all-gathers (NCCL fallback)
    h2d = torch.cuda.Stream(device=local)       # uploads the next iteration's photon slice (e2e leg)
    # Photon exchange between the ranks.  "peer" (default): every rank pushes its slice into the peers' staging
    # buffers with cudaMemcpyAsync over NVLink (copy engines, CUDA IPC mappings: gvpm_peer_*), which overlaps the
    # persistent gather kernels; "nccl": in-place all-gather of the 13 field arrays (SM-based, starved by them).
    exchange = os.environ.get("GVPM_EXCHANGE", "peer") if world > 1 else "none"
    pg_photons = host_pg = None
    inplace_ok = True
    slice_dev = None
    if exchange == "peer":
        blob = torch.frombuffer(bytearray(ctx.peer_export()), dtype=torch.uint8).cuda()
        blobs = [torch.empty_like(blob) for _ in range(world)]
        dist.all_gather(blobs, blob)
        ok = torch.ones(1, device="cuda", dtype=torch.int32)
        try:
            ctx.peer_connect([bytes(b.cpu().numpy().tobytes()) for b in blobs], rank)
        except Exception as e:  # noqa: BLE001 - e.g. no P2P between two devices: every rank falls back together
            print(f"[rank {rank}] peer exchange unavailable ({e}); falling back to NCCL", file=sys.stderr)
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        host_pg = dist.new_group(backend="gloo")   # host-side ordering of the interprocess event records / waits
        push_ctas = int(os.environ.get("GVPM_PUSH_CTAS", str(default_push_ctas(world))))
        ctx.peer_push_mode(push_ctas)
        if int(ok.item()) == 0:
            exchange, host_pg = "nccl", None
    if exchange == "nccl":
        pg_photons = dist.new_group(backend="nccl")
        try:   # NCCL all-gathers in place when the input is the rank's segment of the output; probe torch's checks
            probe = torch.zeros(world * 256, device="cuda", dtype=torch.uint8)
            dist.all_gather_into_tensor(probe, probe[rank * 256:(rank + 1) * 256], group=pg_photons)
            torch.cuda.synchronize()
        except Exception:
            inplace_ok = False
        if not inplace_ok:
            slice_dev = [mine.clone() for _, mine in views[0]]
    ready = [None, None]   # per staging buffer: what the compute stream must wait for before building from it
    # Value leg, N > 1: photon DISPATCH (gvpm_dispatch_*): every rank classifies its resident slice against every
    # receiver's perspective grid and writes the records a receiver can reach into that receiver's inbox (one fused
    # pack + exchange kernel over the peer mappings); a rank builds over what it was sent.  GVPM_VALUE_EXCHANGE=allgather
    # keeps the whole-set exchange above for the value leg too.
    dispatching = world > 1 and os.environ.get("GVPM_VALUE_EXCHANGE", "dispatch") == "dispatch" and prune_build(world) \
        and os.environ.get("GVPM_ACCEL", "") != "bvh"
    if dispatching:
        okd = torch.ones(1, device="cuda", dtype=torch.int32)
        dblob = None
        try:
            dblob = ctx.dispatch_export(world, n_slice)
        except Exception as e:  # noqa: BLE001 - e.g. rays that are not concurrent: every rank falls back together
            print(f"[rank {rank}] photon dispatch unavailable ({e}); the value leg all-gathers the set", file=sys.stderr)
            okd.zero_()
        dist.all_reduce(okd, op=dist.ReduceOp.MIN)
        dispatching = int(okd.item()) == 1
        if dispatching:
            from gvpm_b200 import _native as NAT
            mine = torch.frombuffer(bytearray(dblob), dtype=torch.uint8).cuda()
            allb = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allb, mine)
            try:
                ctx.dispatch_connect([bytes(b.cpu().numpy().tobytes()) for b in allb], rank)
            except Exception as e:  # noqa: BLE001
                print(f"[rank {rank}] photon dispatch unavailable ({e}); the value leg all-gathers the set", file=sys.stderr)
                okd.zero_()
            dist.all_reduce(okd, op=dist.ReduceOp.MIN)
            dispatching = int(okd.item()) == 1
    disp_primed = [False]

    def host_barrier():
        if host_pg is not None:
            dist.barrier(group=host_pg)

    def prefetch(b, from_host):
        """start filling staging buffer b with the NEXT iteration's photon set: (H2D of this rank's slice) + exchange"""
        waits = []
        if from_host:
            ev = torch.cuda.Event()
            ev.record(stream)                   # buffer b was last read by this rank's build two steps ago
            h2d.wait_event(ev)
            ctx.photon_staging_select(b)
            ctx.upload_photons_slice(host_slice, n_ph, s_begin, stream=h2d.cuda_stream)
            up = torch.cuda.Event()
            up.record(h2d)
            waits.append(up)
        if exchange == "peer":
            ctx.peer_push_photon_slice(b, n_ph, s_begin, n_slice, after_stream=h2d.cuda_stream)
            waits.append("peer")
        elif exchange == "nccl":
            if from_host:
                comm.wait_event(waits[0])
            else:
                ev = torch.cuda.Event()
                ev.record(stream)
                comm.wait_event(ev)
            with torch.cuda.stream(comm):
                for i, (whole, mine) in enumerate(views[b]):
                    src = mine if inplace_ok else slice_dev[i]
                    if from_host and not inplace_ok:
                        src.copy_(mine, non_blocking=True)
                    waits.append(dist.all_gather_into_tensor(whole, src, group=pg_photons, async_op=True))
        ready[b] = (b, waits)

    def wait_ready(b):
        if ready[b] is None:
            return
        for w in ready[b][1]:
            if isinstance(w, torch.cuda.Event):
                stream.wait_event(w)
            elif w == "peer":
                ctx.peer_wait_photons(b)
            else:
                with torch.cuda.stream(stream):
                    w.wait()
        ready[b] = None

    # Result gather to rank 0 (north_star): issued from a side stream so that it overlaps the next step's hierarchy
    # build; the gather kernels therefore alternate between two result buffers.  GVPM_COLLECT=inline keeps it on the
    # compute stream.
    coll = torch.cuda.Stream(device=local)
    overlap_collect = world > 1 and os.environ.get("GVPM_COLLECT", "overlap") == "overlap"
    with torch.cuda.stream(stream):
        out_bufs = [out_dev, torch.zeros_like(out_dev) if overlap_collect else out_dev]
    coll_done = [None, None]
    # With the dispatch connected, the results go to rank 0 by plain device-to-device copies into an image buffer rank 0
    # shares over CUDA IPC (gvpm_shared_buffer_*): copy engines over NVLink instead of NCCL's send / receive kernels, which
    # take SMs from the gather kernels, and exactly n_rays rows per rank instead of rows padded to the largest shard.
    peer_collect = dispatching and overlap_collect and os.environ.get("GVPM_COLLECT_VIA", "copy") == "copy"
    img_views = image_bufs = None
    if peer_collect:
        from gvpm_b200 import _native as NAT2
        HB = NAT2.GVPM_SHARED_HANDLE_BYTES
        n_all = [torch.zeros(1, device="cuda", dtype=torch.int64) for _ in range(world)]
        dist.all_gather(n_all, torch.tensor([n_local], device="cuda", dtype=torch.int64))
        rows = [int(t.item()) for t in n_all]
        my_off, rows_total = sum(rows[:rank]), sum(rows)
        hb = torch.zeros(2 * HB, dtype=torch.uint8, device="cuda")
        img_ptrs = []
        if rank == 0:
            hs = []
            for _ in (0, 1):
                p, h_ = ctx.shared_buffer_create(rows_total * 27 * 4)
                img_ptrs.append(p)
                hs.append(h_)
            hb.copy_(torch.frombuffer(bytearray(b"".join(hs)), dtype=torch.uint8))
        dist.broadcast(hb, src=0)
        raw = bytes(hb.cpu().numpy().tobytes())
        if rank != 0:
            img_ptrs = [ctx.shared_buffer_open(raw[i * HB:(i + 1) * HB]) for i in (0, 1)]
        img_views = [torch.as_tensor(DevView(p + my_off * 27 * 4, max(n_local, 1) * 27 * 4), device="cuda").view(torch.float32)
                     for p in img_ptrs]
        if rank == 0:
            image_bufs = [torch.as_tensor(DevView(p, rows_total * 27 * 4), device="cuda").view(torch.float32) for p in img_ptrs]

    def collect(k):
        if world == 1 or os.environ.get("GVPM_COLLECT") == "none":   # "none": diagnostic only (what the result gather costs)
            return
        if peer_collect:
            b = k & 1
            ev = torch.cuda.Event()
            ev.record(stream)
            coll.wait_event(ev)
            with torch.cuda.stream(coll):
                if n_local:
                    img_views[b][:n_local * 27].copy_(out_bufs[b][:n_local * 27], non_blocking=True)
                ctx.collect_signal(b, 0, coll.cuda_stream)
            coll_done[b] = torch.cuda.Event()
            coll_done[b].record(coll)
            return
        if not overlap_collect:
            dist.gather(out_bufs[0], gathered, dst=0)
            return
        ev = torch.cuda.Event()
        ev.record(stream)
        coll.wait_event(ev)
        with torch.cuda.stream(coll):
            dist.gather(out_bufs[k & 1], gathered, dst=0)
        coll_done[k & 1] = torch.cuda.Event()
        coll_done[k & 1].record(coll)

    def wait_collects():
        for i in (0, 1):
            if coll_done[i] is not None:
                stream.wait_event(coll_done[i])
                coll_done[i] = None

    kept = [n_ph]

    def build_resident():
        if prune_build(world):
            ctx.build_points_for_rays(inp["radius"], want_kept=False)
        else:
            ctx.build_points(inp["radius"])

    disp_next = [0]     # inbox generations run on across the timed loop and the diagnostics below
    trace = [] if os.environ.get("GVPM_BENCH_TRACE") else None   # per-step CUDA events (stderr, every rank)

    def mark(what, on=None):
        if trace is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record(on if on is not None else stream)
            trace.append((what, e))

    def step_dispatch(k=None, gather_results=True):
        """value leg, N > 1: (dispatch of step k+1's photons in flight) + build over the inbox + gather + result gather"""
        k = disp_next[0]
        disp_next[0] += 1
        b = k & 1
        if coll_done[b] is not None:            # the result buffer of step k - 2 has been gathered
            stream.wait_event(coll_done[b])
            coll_done[b] = None
        # side stream (overlapped, small persistent grids) from 4 ranks on; with 2 ranks a slice is half the set and the
        # dispatch is better off with the whole machine for a moment (N = 2: 2.85 ms inline, 2.95 on the side stream)
        side = os.environ.get("GVPM_DISPATCH_STREAM", "side" if world > 2 else "inline") == "side"
        if side:   # on the library's priority stream, concurrently with this step (starved by the persistent gather kernels)
            ctx.dispatch_photons(1 - b, n_ph, s_begin, n_slice, inp["radius"], after_stream=h2d.cuda_stream)
        with torch.cuda.stream(stream):
            mark(f"s{k}.begin")
            ctx.build_dispatched(b, inp["radius"])
            mark(f"s{k}.built")
            # step k+1's photons go out between this step's build and its gather, in the compute stream: ~0.1 ms of
            # the step, but every rank's records are in place long before any rank starts its next build (the senders
            # wait for the receivers' release of that inbox on the device)
            if not side:
                ctx.dispatch_photons(1 - b, n_ph, s_begin, n_slice, inp["radius"], after_stream=ctx.stream())
                mark(f"s{k}.dispatched")
            ctx.gather_bre_into(out_bufs[b].data_ptr(), None)
            ctx.dispatch_release(b)
            mark(f"s{k}.gathered")
            if gather_results:
                collect(k)
                if overlap_collect:
                    mark(f"s{k}.collected", coll)

    def step_resident(k):
        """value leg: (photon all-gather of step k+1 in flight) + build + gather (+ result gather)"""
        if dispatching:
            return step_dispatch(k)
        b = k & 1
        wait_ready(b)
        if world > 1:
            prefetch(1 - b, from_host=False)
        ctx.photon_staging_select(b)
        ctx.photon_staging(n_ph)
        if coll_done[b] is not None:            # the result buffer of step k - 2 has been gathered
            stream.wait_event(coll_done[b])
            coll_done[b] = None
        with torch.cuda.stream(stream):
            build_resident()
            ctx.gather_bre_into(out_bufs[b].data_ptr(), None)
            collect(k)
        host_barrier()

    def step_e2e(k):
        """host buffers in, host buffers out, through the C ABI: the photon slice of step k+1 goes up (and is
        all-gathered) while step k is built from the other staging buffer and gathered by the pipelined
        gvpm_gather_bre_host (ray chunks go up while earlier chunks are gathered and their results come down).
        Every rank lands its own tiles in (pinned) host memory of the box, which is where a one-process host
        integrator with one context per GPU reads them; the NCCL gather to rank 0 belongs to the `value` leg."""
        b = k & 1
        wait_ready(b)
        prefetch(1 - b, from_host=True)
        ctx.photon_staging_select(b)
        ctx.photon_staging(n_ph)
        with torch.cuda.stream(stream):
            ctx.build_points(inp["radius"])
            ctx.gather_bre_host(rays, out_host[:n_local * 27])
        host_barrier()

    def timed(fn, steps, warmup, from_host):
        disp = dispatching and fn is step_resident
        if disp:
            assert not disp_primed[0], "one dispatched run per process (inbox generations)"
            disp_primed[0] = True
            ctx.dispatch_photons(0, n_ph, s_begin, n_slice, inp["radius"], after_stream=h2d.cuda_stream)   # step 0 (untimed priming)
        elif world > 1 or from_host:
            prefetch(0, from_host)              # step 0's photon set (untimed priming)
            host_barrier()
        for k in range(warmup):
            fn(k)
        wait_collects()
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        e0.record(stream)
        for k in range(warmup, warmup + steps):
            fn(k)
        if disp:
            ctx.dispatch_join()                 # the K-th dispatch issued inside the timed region ends inside it
        else:
            wait_ready((warmup + steps) & 1)    # the K-th exchange issued inside the timed region ends inside it
        wait_collects()                         # ... and so do the result gathers
        if disp and peer_collect and rank == 0:
            ctx.collect_wait(0)                 # rank 0 has every rank's rows of both image buffers
            ctx.collect_wait(1)
        e1.record(stream)
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if trace:
            t0 = trace[0][1]
            print(f"[trace rank {rank}] " + " ".join(f"{w}={t0.elapsed_time(e):.3f}" for w, e in trace) +
                  f" | timed region {e0.elapsed_time(e1):.3f} ms, starts at {t0.elapsed_time(e0):.3f}", file=sys.stderr, flush=True)
            trace.clear()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        b, g = ctx.last_timings()
        return float(ms.item()), ctx.launch_count() - l0, b, g

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    W = max(3, args.warmup)
    ms_total, launches, build_ms, gather_ms = timed(step_resident, args.steps, W, False)
    if args.dump_outputs:   # the last timed step's result buffer, before the legs below reuse it
        dump_gather(args.dump_outputs, out_bufs[(W + args.steps - 1) & 1], rays)
    collect_ok = None
    if peer_collect:   # what rank 0 holds after the run = what the ranks gathered in their last two steps
        sums = torch.stack([out_bufs[b][:n_local * 27].double().sum() for b in (0, 1)])
        dist.all_reduce(sums)
        if rank == 0:
            got = torch.stack([image_bufs[b].double().sum() for b in (0, 1)])
            collect_ok = bool(torch.allclose(got, sums, rtol=1e-9, atol=0.0)) and bool((got > 0).all())
    ms_e2e, _, _, _ = timed(step_e2e, args.steps, W, True)
    # ---- rows f-1 / f-2: the whole iteration on the device (photons traced, rays generated: nothing uploaded), results
    # to pinned host memory.  N = 1 only; reported next to the host-buffer e2e, never instead of it.
    traced = None
    if world == 1 and os.environ.get("GVPM_BENCH_TRACED", "1") != "0":
        import gvpm_b200 as g
        scene, cam = g.box_scene_default(), g.pinhole_camera(inp["w"], inp["h"])
        tr_paths = [0]

        def step_traced(k):
            tr_paths[0] = ctx.trace_photons(scene, n_ph, 0xC0FFEE + 100 + k, direct=True)
            ctx.generate_rays(scene, cam, 0xC0FFEE + 200 + k, block=-32)
            ctx.build_points_for_rays(inp["radius"], want_kept=False)
            ctx.gather_bre(out=out_host[:n_local * 27], counts=False)
        ms_tr, launches_tr, _, _ = timed(step_traced, args.steps, W, False)
        # phases of one traced step (CUDA events around each call)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        evs[0].record(stream)
        ctx.trace_photons(scene, n_ph, 0xC0FFEE + 99, direct=True); evs[1].record(stream)
        ctx.generate_rays(scene, cam, 0xC0FFEE + 98, block=-32); evs[2].record(stream)
        ctx.build_points_for_rays(inp["radius"], want_kept=False); evs[3].record(stream)
        ctx.gather_bre_into(out_dev.data_ptr(), None); evs[4].record(stream)
        ctx.sync()
        torch.cuda.synchronize()
        traced = {"ms_per_step": ms_tr / args.steps, "value": inp["rays_full_n"] * args.steps / (ms_tr * 1e-3), "unit": "rays/s",
                  "h2d_bytes_per_step": 0, "d2h_bytes_per_step": int(inp["rays_full_n"] * 27 * 4),
                  "phases_ms": {"trace_photons": evs[0].elapsed_time(evs[1]), "generate_rays": evs[1].elapsed_time(evs[2]),
                                "build": evs[2].elapsed_time(evs[3]), "gather": evs[3].elapsed_time(evs[4])},
                  "light_paths": tr_paths[0], "gpu_launches": int(launches_tr),
                  "note": "gvpm_trace_photons_direct + gvpm_generate_rays + gvpm_build_points_for_rays + gvpm_gather_bre "
                          "(27 planes to pinned host memory) per step: inputs are a scene / camera description, created "
                          "on the device - by the contract's definition NOT the end-to-end number, which stays `e2e`"}
        # back to the uploaded set for the remaining diagnostics
        ctx.photon_staging_select(0)
        ctx.photon_staging(n_ph)
        with torch.cuda.stream(stream):
            ctx.upload_rays(rays)
    clocks = sampler.stop() if rank == 0 else None
    # every exchange must have rebuilt the full photon set in both staging buffers
    staging_ok = bool(torch.equal(stage_t[0], stage_t[1]))
    ctx.photon_staging_select(0)
    ctx.photon_staging(n_ph)

    def step_plain():
        if dispatching:
            wait_collects()
            step_dispatch(gather_results=False)
            return
        with torch.cuda.stream(stream):
            build_resident()
            ctx.gather_bre_into(out_dev.data_ptr(), None)
    if os.environ.get("GVPM_BENCH_DIAG"):
        diag_phases(locals())
    # gather-kernel duration averaged over a few launches on the launching stream (CUDA events)
    kt, kd = [], []
    for _ in range(3):
        step_plain()
        kt.append(ctx.last_timings())
        kd.append(ctx.last_gather_detail())
    gather_ms = float(np.mean([k[1] for k in kt]))
    build_ms = float(np.mean([k[0] for k in kt]))
    accel = ctx.accel_kind()
    if dispatching:
        kept[0] = sum(ctx.dispatch_status((disp_next[0] - 1) & 1))   # records received for the last build (synchronises)
    elif prune_build(world):
        with torch.cuda.stream(stream):
            kept[0] = ctx.build_points_for_rays(inp["radius"], want_kept=True)
    trav_ms, shade_ms, n_pairs = float(np.mean([k[0] for k in kd])), float(np.mean([k[1] for k in kd])), kd[-1][2]
    # geometric neighbour counts H (the roofline's numerator) come from one extra, untimed gather: the reference's
    # gather produces no counts, so the timed steps do not either
    with torch.cuda.stream(stream):
        ctx.gather_bre_into(out_dev.data_ptr(), cnt_dev.data_ptr())
    ctx.sync()
    h_geom = torch.tensor([int(cnt_dev.view(-1, 2)[:n_local, 0].to(torch.int64).sum().item())], device="cuda")
    gk = torch.tensor([gather_ms], device="cuda", dtype=torch.float64)
    bk = torch.tensor([build_ms], device="cuda", dtype=torch.float64)
    kept_t = torch.tensor([kept[0], n_local], device="cuda", dtype=torch.int64)
    kept_all = [torch.empty_like(kept_t) for _ in range(world)]
    if world > 1:
        dist.all_reduce(h_geom)
        dist.all_reduce(gk, op=dist.ReduceOp.MAX)
        dist.all_reduce(bk, op=dist.ReduceOp.MAX)
        dist.all_gather(kept_all, kept_t)
    else:
        kept_all = [kept_t]
    build_ms = float(bk.item())

    if rank == 0:
        R = inp["rays_full_n"]
        H = int(h_geom.item())
        value = R * args.steps / (ms_total * 1e-3)
        e2e = R * args.steps / (ms_e2e * 1e-3)
        peak, src = peaks()
        # algorithmic bytes of the dominant kernel (k_gather_bre) per launch, SURVEY.md §8(d):
        # R*(320+108) + H*112 over this rank's rays (the N*112 term belongs to the build kernels)
        alg = (R / world) * 428.0 + (H / world) * 112.0
        achieved = alg / (float(gk.item()) * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic(args.workload if not (args.photons or args.scale) else "", world)
        h2d_bytes = (inp["photons"].nbytes() if inp["photons"] is not None else 0) + rays.nbytes() * world
        line = {"metric": "camera-ray gathers/sec (primal+4 gradients)", "value": value, "unit": "rays/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(args, inp, world),
                "clocks": clocks,
                "e2e": {"value": e2e, "unit": "rays/s", "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(R * 27 * 4),
                        "note": "every rank uploads 1/N of the photon set and its own rays over its own PCIe link; "
                                "the upload + all-gather of step k+1 overlaps the build + gather of step k"},
                "photon_exchange": {"how": {"none": "single GPU", "peer": "slices pushed into the peers' staging buffers over NVLink "
                                            + (f"by a {os.environ.get('GVPM_PUSH_CTAS', str(default_push_ctas(world)))}-CTA store kernel"
                                               if os.environ.get("GVPM_PUSH_CTAS", str(default_push_ctas(world))) != "0"
                                               else "copy engines")
                                            + " (CUDA IPC peer mappings, gvpm_peer_*)",
                                            "nccl": "NCCL all_gather of the 13 field arrays"
                                            + (", in place" if inplace_ok else "")}[exchange],
                                    "double_buffered": True,
                                    "staging_buffers_identical_after_run": staging_ok},
                "gpu_launches": int(launches), "native_lib": _native_lib_path(),
                # the gather is two launches: k_bre_traverse (dominant) + k_bre_shade; SURVEY §8(d)'s
                # per-ray figure covers both, so the roofline is quoted over the pair
                "roofline": {"bound": "hbm", "kernel": ("k_bre_grid_traverse" if accel == "frustum" else "k_bre_traverse") + " + k_bre_shade",
                             "achieved": achieved, "l2": l2_roofline(args.workload if not (args.photons or args.scale) else "", world, float(gk.item())),
                             "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                             "traffic_source": traffic_src, "peak_source": src, "algorithmic_bytes_per_launch": alg,
                             "kernel_ms": float(gk.item()), "traverse_ms": trav_ms, "shade_ms": shade_ms,
                             "neighbours_H": H, "contributing_pairs": n_pairs,
                             "note": "latency- / issue-bound kernels: DRAM traffic is below the algorithmic bytes and L2 traffic "
                                     "at a quarter of its peak (profiles/r2_gather_bre.md); the HBM fraction is reported as "
                                     "the contract asks"},
                "phases_ms": {"build": build_ms, "gather": float(gk.item()), "traverse": trav_ms,
                              "shade": shade_ms},
                "result_collection_verified": collect_ok,
                "result_collection": ("device-to-device copies into rank 0's image buffer (CUDA IPC, copy engines), per-rank generation flags"
                                      if peer_collect else ("NCCL gather to rank 0" if world > 1 else "single GPU")),
                "value_exchange": ("photon dispatch: each rank classifies its resident slice against every receiver's perspective grid and "
                                   "writes the 128-byte records a receiver can reach into that receiver's inbox over NVLink "
                                   "(gvpm_dispatch_*), double-buffered, device-side generation flags" if dispatching else
                                   ("whole-set exchange (see photon_exchange)" if world > 1 else "single GPU")),
                "shards": {"mode": shard_mode(world), "band_cycles": band_cycles() if shard_mode(world) == "band" else None,
                           "pruned_build": prune_build(world), "accel": accel, "balance": balance,
                           "rays_per_rank": [int(k[1].item()) for k in kept_all],
                           "photons_in_hierarchy_per_rank": [int(k[0].item()) for k in kept_all]},
                "light_paths": inp["n_paths"]}
        if traced is not None:
            line["device_traced"] = traced
        if world == 1 and not args.no_cpu_baseline:
            inp["full_rays"] = inp["rays"]
            cb, _, _ = cpu_arm(args, inp, args.cpu_seconds)
            cb["see_also"] = ("`bench.py --impl reference` times the reference's OWN compiled code (cpu_baseline.kind "
                              "\"reference\"); this port is 1.2x - 1.4x faster than the code it restates "
                              "(profiles/r2_cpu_reference_code.md)")
            line["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    # tensors allocated on the context's stream must go before the stream does
    # (device tensors and pinned host buffers that were used on it record events on that stream when
    # they are freed)
    del img_views, image_bufs
    del out_dev, out_bufs, cnt_dev, gathered, stage_t, views, slice_dev, keep_host, host_slice, host_fields, counts_max, h_geom, gk, bk, kept_t, kept_all
    del out_host_t, out_host, rays
    inp.clear()
    import gc
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.stdout.flush()
    # every tensor that lived on the context's stream is gone and torch's caches are empty: destroy the context
    # (gvpm_ctx_destroy) and leave through the interpreter's normal exit, so that exit hooks see libgvpm_b200.so
    del stream
    gc.collect()
    try:
        torch._C._host_emptyCache()
    except Exception:  # noqa: BLE001 - older torch: the pinned cache only queries events, never the stream
        pass
    ctx.close()


if __name__ == "__main__":
    main()
