"""ctypes binding of tests/prims_ref.cpp (TEST INFRASTRUCTURE): the CPU restatement of gvpm_trace_beams and
gvpm_planes_from_beams.  The library is compiled on first use into a temporary directory that goes when the process
ends, with the flags of the oracle (no FMA contraction), so nothing is written into the tree."""
import ctypes as C
import os
import subprocess
import tempfile

from gvpm_b200 import _native as N
from gvpm_b200 import records as R

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None
_tmp = None


def load():
    global _lib, _tmp
    if _lib is not None:
        return _lib
    _tmp = tempfile.TemporaryDirectory(prefix="gvpm_prims_ref_")
    so = os.path.join(_tmp.name, "libprims_ref.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                           "-o", so, os.path.join(_HERE, "prims_ref.cpp")])
    lib = C.CDLL(so)
    lib.prims_ref_trace_beams.argtypes = [C.POINTER(N.BoxScene), C.POINTER(N.Medium), C.c_size_t, C.c_uint64, C.c_int,
                                          C.c_int, C.c_int, C.POINTER(N.BeamSoA)]
    lib.prims_ref_trace_beams.restype = C.c_longlong
    lib.prims_ref_planes_from_beams.argtypes = [C.POINTER(N.BeamSoA), C.c_size_t, C.POINTER(N.Medium), C.c_uint64,
                                                C.POINTER(N.PlaneSoA)]
    lib.prims_ref_planes_from_beams.restype = C.c_longlong
    _lib = lib
    return lib


def trace_beams(scene, medium, n, seed, max_depth=12, rr_depth=1, min_depth=0):
    """CPU restatement of gvpm_trace_beams: -> (BeamSet, light paths traced)"""
    bs = R.BeamSet(n)
    cs = bs.as_c()
    paths = load().prims_ref_trace_beams(C.byref(scene), C.byref(medium), n, seed, max_depth, rr_depth, min_depth,
                                         C.byref(cs))
    if paths < 0:
        raise RuntimeError("prims_ref_trace_beams failed")
    return bs, int(paths)


def planes_from_beams(beams, medium, seed):
    """CPU restatement of gvpm_planes_from_beams: -> PlaneSet (one plane per beam)"""
    ps = R.PlaneSet(beams.n)
    cb, cp = beams.as_c(), ps.as_c()
    if load().prims_ref_planes_from_beams(C.byref(cb), beams.n, C.byref(medium), seed, C.byref(cp)) < 0:
        raise RuntimeError("prims_ref_planes_from_beams failed (sampling_weight must be 1)")
    return ps
