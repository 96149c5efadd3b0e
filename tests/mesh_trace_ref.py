"""ctypes binding of tests/mesh_trace_ref.cpp (TEST INFRASTRUCTURE): the CPU restatement of the mesh-scene generators
(gvpm_trace_photons_mesh, gvpm_trace_beams_mesh, gvpm_generate_rays_mesh) and of their closest hit and emitter pick.
The library is compiled on first use into a temporary directory that goes when the process ends, with the flags of the
oracle (no FMA contraction), so nothing is written into the tree."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from gvpm_b200 import _native as N
from gvpm_b200 import records as R

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None
_tmp = None


def load():
    global _lib, _tmp
    if _lib is not None:
        return _lib
    _tmp = tempfile.TemporaryDirectory(prefix="gvpm_mesh_ref_")
    so = os.path.join(_tmp.name, "libmesh_trace_ref.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                           "-o", so, os.path.join(_HERE, "mesh_trace_ref.cpp")])
    lib = C.CDLL(so)
    ms = C.POINTER(N.MeshScene)
    for name, soa in (("mesh_ref_trace_photons", N.PhotonSoA), ("mesh_ref_trace_beams", N.BeamSoA)):
        fn = getattr(lib, name)
        fn.argtypes = [ms, C.POINTER(N.Medium), C.c_size_t, C.c_uint64, C.c_int, C.c_int, C.c_int, C.POINTER(soa)]
        fn.restype = C.c_longlong
    lib.mesh_ref_generate_rays.argtypes = [ms, C.POINTER(N.LookatCamera), C.c_uint64, C.c_int, C.c_int, C.c_int,
                                           C.c_float, C.POINTER(N.RaySoA)]
    lib.mesh_ref_generate_rays.restype = C.c_longlong
    lib.mesh_ref_closest.argtypes = [ms, N.f32p, N.f32p, N.u32p, C.c_size_t, N.f32p, N.u32p, N.f32p]
    lib.mesh_ref_closest.restype = None
    lib.mesh_ref_pick.argtypes = [ms, N.f32p, C.c_size_t, N.u32p]
    lib.mesh_ref_pick.restype = None
    _lib = lib
    return lib


class Scene:
    """the arrays of Context.set_trace_mesh kept alive behind one gvpm_mesh_scene"""

    def __init__(self, tri, albedo, emissive, light_power, lo, hi):
        self.tri = np.ascontiguousarray(tri, dtype=np.float32).reshape(-1, 9)
        n = self.tri.shape[0]
        self.albedo = np.ascontiguousarray(albedo, dtype=np.float32).reshape(n, 3)
        self.emissive = np.ascontiguousarray(emissive, dtype=np.uint8).reshape(n)
        self.light_power, self.lo, self.hi = float(light_power), tuple(lo), tuple(hi)
        self.c = N.MeshScene()
        for a in range(3):
            self.c.lo[a], self.c.hi[a] = float(lo[a]), float(hi[a])
        self.c.n_tri = n
        self.c.tri, self.c.albedo = self.tri.ctypes.data_as(N.f32p), self.albedo.ctypes.data_as(N.f32p)
        self.c.emissive = self.emissive.ctypes.data_as(N.u8p)
        self.c.light_power = self.light_power

    def kwargs(self):
        return dict(tri=self.tri, albedo=self.albedo, emissive=self.emissive, light_power=self.light_power,
                    lo=self.lo, hi=self.hi)


def trace_photons(scene, medium, n, seed, max_depth=12, rr_depth=1, min_depth=0):
    """-> (PhotonSet, light paths traced)"""
    ps = R.PhotonSet(n)
    cs = ps.as_c()
    paths = load().mesh_ref_trace_photons(C.byref(scene.c), C.byref(medium), n, seed, max_depth, rr_depth, min_depth,
                                          C.byref(cs))
    if paths < 0:
        raise RuntimeError("mesh_ref_trace_photons failed")
    return ps, int(paths)


def trace_beams(scene, medium, n, seed, max_depth=12, rr_depth=1, min_depth=0):
    """-> (BeamSet, light paths traced)"""
    bs = R.BeamSet(n)
    cs = bs.as_c()
    paths = load().mesh_ref_trace_beams(C.byref(scene.c), C.byref(medium), n, seed, max_depth, rr_depth, min_depth,
                                        C.byref(cs))
    if paths < 0:
        raise RuntimeError("mesh_ref_trace_beams failed")
    return bs, int(paths)


def generate_rays(scene, camera, seed, block=32, y0=0, y1=None, epsilon=1e-4):
    """-> RaySet in the device's order"""
    y1 = camera.film_h if y1 is None else y1
    rs = R.RaySet(camera.film_w * (y1 - y0))
    cs = rs.as_c()
    got = load().mesh_ref_generate_rays(C.byref(scene.c), C.byref(camera), seed, block, y0, y1, epsilon, C.byref(cs))
    assert got == rs.n, (got, rs.n)
    return rs


def closest(scene, o, d, skip=None):
    """brute-force closest hit -> (t, triangle index or 0xffffffff for the box exit, normal facing the ray)"""
    o = np.ascontiguousarray(o, dtype=np.float32).reshape(-1, 3)
    d = np.ascontiguousarray(d, dtype=np.float32).reshape(-1, 3)
    m = o.shape[0]
    t, tri, n = np.zeros(m, np.float32), np.zeros(m, np.uint32), np.zeros((m, 3), np.float32)
    sk = None if skip is None else np.ascontiguousarray(skip, dtype=np.uint32)
    load().mesh_ref_closest(C.byref(scene.c), o.ctypes.data_as(N.f32p), d.ctypes.data_as(N.f32p),
                            None if sk is None else sk.ctypes.data_as(N.u32p), m, t.ctypes.data_as(N.f32p),
                            tri.ctypes.data_as(N.u32p), n.ctypes.data_as(N.f32p))
    return t, tri, n


def pick(scene, u0):
    """the emitter pick of each u0 -> triangle index"""
    u0 = np.ascontiguousarray(u0, dtype=np.float32)
    out = np.zeros(u0.size, np.uint32)
    load().mesh_ref_pick(C.byref(scene.c), u0.ctypes.data_as(N.f32p), u0.size, out.ctypes.data_as(N.u32p))
    return out
