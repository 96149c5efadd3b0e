"""ctypes binding of the CPU oracle (TEST INFRASTRUCTURE — see oracle/gvpm_oracle.hpp).

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs.  The product package gvpm_b200 never imports this module.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from gvpm_b200 import _native as N

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgvpm_oracle.so")
_lib = None
_native_dir = None


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


def prefer_native():
    """bench.py's CPU legs: build the oracle with -march=native on THIS machine (untimed) into a temporary directory, which
    goes when the process ends, and load that build; falls back to the portable build.  Must be called before the first
    load().  -> the flags in use"""
    global LIB_PATH, _native_dir
    assert _lib is None, "prefer_native() after load()"
    try:
        _native_dir = tempfile.TemporaryDirectory(prefix="gvpm_oracle_native_")
        subprocess.check_call(["make", "-s", "-B", "-C", _HERE, "native", "NATIVE_DIR=" + _native_dir.name])
        LIB_PATH = os.path.join(_native_dir.name, "libgvpm_oracle.so")
        return "-O3 -march=native -ffp-contract=off"
    except Exception:  # noqa: BLE001 - no compiler on the box: the shipped portable build
        return "-O3 -ffp-contract=off (portable build: native rebuild failed)"


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        build()
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.gvpm_oracle_hw_threads.restype = C.c_int
    lib.gvpm_oracle_tree_build.argtypes = [C.POINTER(N.PhotonSoA), C.c_size_t, C.c_float, C.c_int]
    lib.gvpm_oracle_tree_build.restype = vp
    lib.gvpm_oracle_tree_build_ms.argtypes = [vp]
    lib.gvpm_oracle_tree_build_ms.restype = C.c_double
    lib.gvpm_oracle_tree_depth.argtypes = [vp]
    lib.gvpm_oracle_tree_depth.restype = C.c_size_t
    lib.gvpm_oracle_tree_free.argtypes = [vp]
    lib.gvpm_oracle_bre.argtypes = [vp, C.POINTER(N.PhotonSoA), C.c_size_t, C.POINTER(N.RaySoA), C.c_size_t,
                                    C.c_size_t, C.POINTER(N.Medium), C.POINTER(N.Config), N.f32p, C.c_size_t,
                                    C.c_float, C.c_int, C.c_int, N.f32p, N.u32p, N.u64p, N.u32p, C.c_size_t,
                                    C.POINTER(C.c_double)]
    lib.gvpm_oracle_bre.restype = C.c_longlong
    lib.gvpm_oracle_vpm.argtypes = [vp, C.POINTER(N.PhotonSoA), C.c_size_t, C.POINTER(N.RaySoA), C.c_size_t,
                                    C.POINTER(N.VpmSampleSoA), C.c_size_t, C.POINTER(N.Medium), C.POINTER(N.Config),
                                    N.f32p, C.c_size_t, C.c_int, C.c_int, C.c_int, N.f32p, N.f32p, N.u32p, N.u64p,
                                    N.u32p, C.c_size_t, C.POINTER(C.c_double)]
    lib.gvpm_oracle_vpm.restype = C.c_longlong
    lib.gvpm_oracle_beams.argtypes = [C.POINTER(N.BeamSoA), C.c_size_t, C.POINTER(N.RaySoA), C.c_size_t,
                                      C.POINTER(N.Medium), C.POINTER(N.Config), N.f32p, C.c_size_t, C.c_float,
                                      C.c_int, C.c_int, N.f32p, N.u32p, N.u64p, N.u32p, C.c_size_t,
                                      C.POINTER(C.c_double)]
    lib.gvpm_oracle_beams.restype = C.c_longlong
    lib.gvpm_oracle_planes.argtypes = [C.POINTER(N.PlaneSoA), C.c_size_t, C.POINTER(N.RaySoA), C.c_size_t,
                                       C.POINTER(N.Medium), C.POINTER(N.Config), C.c_int, C.c_int, C.c_int, N.f32p,
                                       N.u32p, N.u64p, N.u32p, C.c_size_t, C.POINTER(C.c_double),
                                       C.POINTER(C.c_double)]
    lib.gvpm_oracle_planes.restype = C.c_longlong
    lib.gvpm_oracle_sppm_bre.argtypes = [vp, C.POINTER(N.PhotonSoA), C.c_size_t, C.POINTER(N.RaySoA), C.c_size_t,
                                         C.POINTER(N.Medium), C.POINTER(N.Config), C.c_float, C.c_int, N.f32p, N.u32p,
                                         N.u64p, N.u32p, C.c_size_t, C.POINTER(C.c_double)]
    lib.gvpm_oracle_sppm_bre.restype = C.c_longlong
    lib.gvpm_oracle_sppm_beams.argtypes = [C.POINTER(N.BeamSoA), C.c_size_t, C.POINTER(N.RaySoA), C.c_size_t,
                                           C.POINTER(N.Medium), C.POINTER(N.Config), C.c_float, C.c_int, C.c_int,
                                           C.c_int, N.f32p, N.u32p, N.u64p, N.u32p, C.c_size_t]
    lib.gvpm_oracle_sppm_beams.restype = C.c_longlong
    lib.gvpm_oracle_subbeams.argtypes = [C.POINTER(N.BeamSoA), C.c_size_t, N.f32p, N.u32p, C.c_size_t]
    lib.gvpm_oracle_subbeams.restype = C.c_longlong
    _lib = lib
    return lib


def planes_gather(planes, rays, medium, config, mode="brute", double=False, threads=None, neighbours=False):
    """Restated computeVolumeGradientPlanes gather (gvpm.cpp:782-878), plane0d kernel.  mode "brute": every
    (ray, plane) pair; "kdtree": the reference's balanced kd-tree + AABB hierarchy + DFS (plane_accel.h).
    Returns a BreResult (idx = plane indices with bit 31 set)."""
    lib = load()
    threads = hw_threads() if threads is None else threads
    cp, cr = planes.as_c(), rays.as_c()
    out = np.zeros(rays.n * N.GVPM_OUT_FLOATS, dtype=np.float32)
    counts = np.zeros(rays.n * 2, dtype=np.uint32)
    ms, bms = C.c_double(0), C.c_double(0)
    m = {"brute": 0, "kdtree": 1}[mode]

    def call(offp, idxp, capv):
        r = lib.gvpm_oracle_planes(C.byref(cp), planes.n, C.byref(cr), rays.n, C.byref(medium), C.byref(config), m,
                                   int(double), threads, out.ctypes.data_as(N.f32p), counts.ctypes.data_as(N.u32p),
                                   offp, idxp, capv, C.byref(ms), C.byref(bms))
        if r < 0:
            raise RuntimeError(f"gvpm_oracle_planes failed: {r}")
        return int(r)
    offsets = idx = None
    if neighbours:
        offsets = np.zeros(rays.n + 1, dtype=np.uint64)
        cap = call(offsets.ctypes.data_as(N.u64p), None, 0)
        idx = np.zeros(max(cap, 1), dtype=np.uint32)
        call(offsets.ctypes.data_as(N.u64p), idx.ctypes.data_as(N.u32p), cap)
        idx = idx[:cap]
    else:
        call(None, None, 0)
    return BreResult(out.reshape(rays.n, N.GVPM_OUT_FLOATS), counts.reshape(rays.n, 2), offsets, idx, ms.value,
                     bms.value)


def beams_gather(beams, rays, medium, config, tri, radius, double=False, threads=None, neighbours=False):
    """Restated computeVolumeGradientBeams gather (gvpm.cpp:880-986), beam3d kernel, brute force over all
    (ray, beam) pairs.  Returns a BreResult (idx = beam indices, bit 31 = contributes)."""
    lib = load()
    threads = hw_threads() if threads is None else threads
    cb, cr = beams.as_c(), rays.as_c()
    tri = np.ascontiguousarray(tri, dtype=np.float32)
    out = np.zeros(rays.n * N.GVPM_OUT_FLOATS, dtype=np.float32)
    counts = np.zeros(rays.n * 2, dtype=np.uint32)
    ms = C.c_double(0)

    def call(offp, idxp, capv):
        r = lib.gvpm_oracle_beams(C.byref(cb), beams.n, C.byref(cr), rays.n, C.byref(medium), C.byref(config),
                                  tri.ctypes.data_as(N.f32p), tri.size // 9, radius, int(double), threads,
                                  out.ctypes.data_as(N.f32p), counts.ctypes.data_as(N.u32p), offp, idxp, capv,
                                  C.byref(ms))
        if r < 0:
            raise RuntimeError(f"gvpm_oracle_beams failed: {r}")
        return int(r)
    offsets = idx = None
    if neighbours:
        offsets = np.zeros(rays.n + 1, dtype=np.uint64)
        cap = call(offsets.ctypes.data_as(N.u64p), None, 0)
        idx = np.zeros(max(cap, 1), dtype=np.uint32)
        call(offsets.ctypes.data_as(N.u64p), idx.ctypes.data_as(N.u32p), cap)
        idx = idx[:cap]
    else:
        call(None, None, 0)
    return BreResult(out.reshape(rays.n, N.GVPM_OUT_FLOATS), counts.reshape(rays.n, 2), offsets, idx, ms.value, 0.0)


BEAM_TECHNIQUES = {"beam1d": 0, "beam3d_naive": 1, "beam3d_egsr": 2, "beam3d": 3}


def sppm_beams_gather(beams, rays, medium, config, radius, technique, double=False, threads=None, neighbours=False):
    """Restated sppm primal beam gather (BeamRadianceQuery, beams.h:29-223; sppm.cpp:823-860), brute force over all
    (camera beam, sub-beam) pairs.  technique: key of BEAM_TECHNIQUES.  Returns a BreResult with out [n_rays,3]."""
    lib = load()
    threads = hw_threads() if threads is None else threads
    cb, cr = beams.as_c(), rays.as_c()
    out = np.zeros(rays.n * 3, dtype=np.float32)
    counts = np.zeros(rays.n * 2, dtype=np.uint32)
    tech = BEAM_TECHNIQUES[technique] if isinstance(technique, str) else int(technique)

    def call(offp, idxp, capv):
        r = lib.gvpm_oracle_sppm_beams(C.byref(cb), beams.n, C.byref(cr), rays.n, C.byref(medium), C.byref(config),
                                       radius, tech, int(double), threads, out.ctypes.data_as(N.f32p),
                                       counts.ctypes.data_as(N.u32p), offp, idxp, capv)
        if r < 0:
            raise RuntimeError(f"gvpm_oracle_sppm_beams failed: {r}")
        return int(r)
    offsets = idx = None
    if neighbours:
        offsets = np.zeros(rays.n + 1, dtype=np.uint64)
        cap = call(offsets.ctypes.data_as(N.u64p), None, 0)
        idx = np.zeros(max(cap, 1), dtype=np.uint32)
        call(offsets.ctypes.data_as(N.u64p), idx.ctypes.data_as(N.u32p), cap)
        idx = idx[:cap]
    else:
        call(None, None, 0)
    return BreResult(out.reshape(rays.n, 3), counts.reshape(rays.n, 2), offsets, idx, 0.0, 0.0)


def subbeams(beams):
    """The reference's sub-beam split (beams_accel.h:98-124): (t12 [n,2] float32, beam [n] uint32)."""
    lib = load()
    cb = beams.as_c()
    n = int(lib.gvpm_oracle_subbeams(C.byref(cb), beams.n, None, None, 0))
    t12 = np.zeros(max(n, 1) * 2, dtype=np.float32)
    bi = np.zeros(max(n, 1), dtype=np.uint32)
    lib.gvpm_oracle_subbeams(C.byref(cb), beams.n, t12.ctypes.data_as(N.f32p), bi.ctypes.data_as(N.u32p), n)
    return t12[:2 * n].reshape(n, 2), bi[:n]


def hw_threads():
    return load().gvpm_oracle_hw_threads()


class BreResult:
    def __init__(self, out, counts, offsets, idx, gather_ms, build_ms):
        self.out, self.counts, self.offsets, self.idx = out, counts, offsets, idx
        self.gather_ms, self.build_ms = gather_ms, build_ms

    def neighbours(self, i):
        """(sorted original photon indices of the geometric set, contributes-mask)"""
        a = self.idx[self.offsets[i]:self.offsets[i + 1]]
        return a & np.uint32(0x7FFFFFFF), (a >> np.uint32(31)).astype(bool)


def bre_gather(photons, rays, medium, config, tri, radius, mode="kdtree", double=False, threads=None,
               begin=0, end=None, neighbours=False):
    """Restated computeVolumeGradientPhotonBRE gather (gvpm.cpp:999-1052) over rays [begin,end).

    mode "kdtree": reference-shaped sliding-midpoint kd layout + AABB hierarchy + stack DFS;
    mode "brute":  all photons against the neighbour predicate (tree-independent set)."""
    lib = load()
    end = rays.n if end is None else end
    threads = hw_threads() if threads is None else threads
    cph, cr = photons.as_c(), rays.as_c()
    tri = np.ascontiguousarray(tri, dtype=np.float32)
    tree, build_ms = None, 0.0
    if mode == "kdtree":
        tree = lib.gvpm_oracle_tree_build(C.byref(cph), photons.n, radius, int(double))
        build_ms = lib.gvpm_oracle_tree_build_ms(tree)
    m = end - begin
    out = np.zeros(m * N.GVPM_OUT_FLOATS, dtype=np.float32)
    counts = np.zeros(m * 2, dtype=np.uint32)
    ms = C.c_double(0)
    offsets = idx = None
    try:
        if neighbours:
            offsets = np.zeros(m + 1, dtype=np.uint64)
            need = lib.gvpm_oracle_bre(tree, C.byref(cph), photons.n, C.byref(cr), begin, end, C.byref(medium),
                                       C.byref(config), tri.ctypes.data_as(N.f32p), tri.size // 9, radius,
                                       int(double), threads, out.ctypes.data_as(N.f32p),
                                       counts.ctypes.data_as(N.u32p), offsets.ctypes.data_as(N.u64p), None, 0,
                                       C.byref(ms))
            if need < 0:
                raise RuntimeError(f"gvpm_oracle_bre failed: {need}")
            idx = np.zeros(max(int(need), 1), dtype=np.uint32)
            cap = int(need)
        else:
            cap = 0
        need = lib.gvpm_oracle_bre(tree, C.byref(cph), photons.n, C.byref(cr), begin, end, C.byref(medium),
                                   C.byref(config), tri.ctypes.data_as(N.f32p), tri.size // 9, radius, int(double),
                                   threads, out.ctypes.data_as(N.f32p), counts.ctypes.data_as(N.u32p),
                                   offsets.ctypes.data_as(N.u64p) if neighbours else None,
                                   idx.ctypes.data_as(N.u32p) if neighbours else None, cap, C.byref(ms))
        if need < 0:
            raise RuntimeError(f"gvpm_oracle_bre failed: {need}")
    finally:
        if tree:
            lib.gvpm_oracle_tree_free(tree)
    return BreResult(out.reshape(m, N.GVPM_OUT_FLOATS), counts.reshape(m, 2), offsets,
                     idx[:cap] if neighbours else None, ms.value, build_ms)


def sppm_bre_gather(photons, rays, medium, config, radius, mode="kdtree", threads=None, neighbours=False):
    """Restated sppm primal BRE (sppm.cpp:926-981 + bre.cpp:167-259).  Returns a BreResult with out [n_rays,3]."""
    lib = load()
    threads = hw_threads() if threads is None else threads
    cph, cr = photons.as_c(), rays.as_c()
    tree = lib.gvpm_oracle_tree_build(C.byref(cph), photons.n, radius, 0) if mode == "kdtree" else None
    out = np.zeros(rays.n * 3, dtype=np.float32)
    counts = np.zeros(rays.n * 2, dtype=np.uint32)
    ms = C.c_double(0)

    def call(offp, idxp, capv):
        r = lib.gvpm_oracle_sppm_bre(tree, C.byref(cph), photons.n, C.byref(cr), rays.n, C.byref(medium),
                                     C.byref(config), radius, threads, out.ctypes.data_as(N.f32p),
                                     counts.ctypes.data_as(N.u32p), offp, idxp, capv, C.byref(ms))
        if r < 0:
            raise RuntimeError(f"gvpm_oracle_sppm_bre failed: {r}")
        return int(r)
    offsets = idx = None
    try:
        if neighbours:
            offsets = np.zeros(rays.n + 1, dtype=np.uint64)
            cap = call(offsets.ctypes.data_as(N.u64p), None, 0)
            idx = np.zeros(max(cap, 1), dtype=np.uint32)
            call(offsets.ctypes.data_as(N.u64p), idx.ctypes.data_as(N.u32p), cap)
            idx = idx[:cap]
        else:
            call(None, None, 0)
    finally:
        if tree:
            lib.gvpm_oracle_tree_free(tree)
    return BreResult(out.reshape(rays.n, 3), counts.reshape(rays.n, 2), offsets, idx, ms.value, 0.0)


class VpmResult:
    def __init__(self, out, mvol, sample_counts, offsets, idx, gather_ms):
        self.out, self.mvol, self.sample_counts, self.offsets, self.idx = out, mvol, sample_counts, offsets, idx
        self.gather_ms = gather_ms


def vpm_gather(photons, rays, samples, medium, config, tri, nb_camera_samples, mode="kdtree", double=False,
               threads=None, neighbours=False):
    """Restated computeVolumeGradientPhoton gather (gvpm.cpp:1141-1185) over all distance samples."""
    lib = load()
    threads = hw_threads() if threads is None else threads
    cph, cr, cs = photons.as_c(), rays.as_c(), samples.as_c()
    tri = np.ascontiguousarray(tri, dtype=np.float32)
    tree = lib.gvpm_oracle_tree_build(C.byref(cph), photons.n, 1.0, int(double)) if mode == "kdtree" else None
    out = np.zeros(rays.n * N.GVPM_OUT_FLOATS, dtype=np.float32)
    mvol = np.zeros(rays.n, dtype=np.float32)
    sc = np.zeros(samples.n * 2, dtype=np.uint32)
    ms = C.c_double(0)
    offsets = idx = None
    cap = 0

    def call(offp, idxp, capv):
        r = lib.gvpm_oracle_vpm(tree, C.byref(cph), photons.n, C.byref(cr), rays.n, C.byref(cs), samples.n,
                                C.byref(medium), C.byref(config), tri.ctypes.data_as(N.f32p), tri.size // 9,
                                nb_camera_samples, int(double), threads, out.ctypes.data_as(N.f32p),
                                mvol.ctypes.data_as(N.f32p), sc.ctypes.data_as(N.u32p), offp, idxp, capv,
                                C.byref(ms))
        if r < 0:
            raise RuntimeError(f"gvpm_oracle_vpm failed: {r}")
        return r
    try:
        if neighbours:
            offsets = np.zeros(samples.n + 1, dtype=np.uint64)
            cap = int(call(offsets.ctypes.data_as(N.u64p), None, 0))
            idx = np.zeros(max(cap, 1), dtype=np.uint32)
            call(offsets.ctypes.data_as(N.u64p), idx.ctypes.data_as(N.u32p), cap)
            idx = idx[:cap]
        else:
            call(None, None, 0)
    finally:
        if tree:
            lib.gvpm_oracle_tree_free(tree)
    return VpmResult(out.reshape(rays.n, N.GVPM_OUT_FLOATS), mvol, sc.reshape(samples.n, 2), offsets, idx, ms.value)


def trace_photons(scene, medium, n, seed, max_depth=12, rr_depth=1, min_depth=0):
    """CPU restatement of gvpm_trace_photons (oracle/gvpm_oracle_trace.cpp): -> (PhotonSet, light paths traced)"""
    from gvpm_b200 import records as R
    lib = load()
    lib.gvpm_oracle_trace_photons.argtypes = [C.POINTER(N.BoxScene), C.POINTER(N.Medium), C.c_size_t, C.c_uint64, C.c_int,
                                              C.c_int, C.c_int, C.POINTER(N.PhotonSoA)]
    lib.gvpm_oracle_trace_photons.restype = C.c_longlong
    ps = R.PhotonSet(n)
    cs = ps.as_c()
    paths = lib.gvpm_oracle_trace_photons(C.byref(scene), C.byref(medium), n, seed, max_depth, rr_depth, min_depth, C.byref(cs))
    if paths < 0:
        raise RuntimeError("gvpm_oracle_trace_photons failed")
    return ps, int(paths)


def pm_functions(x):
    """the tracer's polynomial log(x), exp(-x), sin(2 pi frac(x)), cos(2 pi frac(x))"""
    lib = load()
    x = np.ascontiguousarray(x, dtype=np.float32)
    outs = [np.zeros(x.size, np.float32) for _ in range(4)]
    lib.gvpm_oracle_pm_functions.argtypes = [C.c_size_t] + [N.f32p] * 5
    lib.gvpm_oracle_pm_functions.restype = None
    lib.gvpm_oracle_pm_functions(x.size, x.ctypes.data_as(N.f32p), *[o.ctypes.data_as(N.f32p) for o in outs])
    return outs
