"""ctypes binding of tests/vpm_samples_ref.cpp (TEST INFRASTRUCTURE): the CPU restatement of gvpm_generate_vpm_samples.
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
    _tmp = tempfile.TemporaryDirectory(prefix="gvpm_vpm_samples_ref_")
    so = os.path.join(_tmp.name, "libvpm_samples_ref.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                           "-o", so, os.path.join(_HERE, "vpm_samples_ref.cpp")])
    lib = C.CDLL(so)
    lib.vpm_samples_ref.argtypes = [C.POINTER(N.RaySoA), C.c_size_t, C.c_int, C.c_int, C.c_uint64,
                                          C.POINTER(N.Medium), C.c_float, C.c_float, N.f32p, C.POINTER(N.VpmSampleSoA)]
    lib.vpm_samples_ref.restype = C.c_longlong
    _lib = lib
    return lib


def vpm_samples(rays, medium, nb_camera_samples=40, seed=0, radius=None, radius_per_ray=None, stratified=False,
                epsilon=1e-4):
    """CPU restatement of gvpm_generate_vpm_samples on a RaySet: -> VpmSampleSet"""
    full = R.VpmSampleSet(rays.n * nb_camera_samples)
    cr, cs = rays.as_c(), full.as_c()
    rad = None
    if radius_per_ray is not None:
        rad = np.ascontiguousarray(radius_per_ray, dtype=np.float32).reshape(-1)
        assert rad.size == rays.n
    n = load().vpm_samples_ref(C.byref(cr), rays.n, nb_camera_samples, int(bool(stratified)), seed,
                                     C.byref(medium), epsilon, 0.0 if radius is None else radius,
                                     None if rad is None else rad.ctypes.data_as(N.f32p), C.byref(cs))
    if n < 0:
        raise RuntimeError("vpm_samples_ref failed")
    return full.take(np.arange(n))
