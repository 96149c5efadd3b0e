"""ctypes binding of tests/any_hit_ref.cpp (TEST INFRASTRUCTURE): the oracle's Occluders<float>::anyHit over a whole
triangle list, multithreaded.  The library is compiled on first use into a temporary directory that goes when the process
ends, with the flags of the oracle (no FMA contraction), so nothing is written into the tree."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from gvpm_b200 import _native as N

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None
_tmp = None


def load():
    global _lib, _tmp
    if _lib is not None:
        return _lib
    _tmp = tempfile.TemporaryDirectory(prefix="gvpm_any_hit_ref_")
    so = os.path.join(_tmp.name, "libany_hit_ref.so")
    subprocess.check_call(["g++", "-O3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off",
                           "-fno-fast-math", "-o", so, os.path.join(_HERE, "any_hit_ref.cpp")])
    lib = C.CDLL(so)
    lib.any_hit_ref.argtypes = [N.f32p, C.c_size_t, N.f32p, N.f32p, N.f32p, N.f32p, C.c_size_t, C.c_int, N.u8p]
    lib.any_hit_ref.restype = None
    _lib = lib
    return lib


def any_hit(tri, ro, rd, mint, maxt, threads=None):
    """Occluders::anyHit over the whole triangle list for each ray -> bool[m]."""
    tri = np.ascontiguousarray(tri, dtype=np.float32).reshape(-1)
    ro = np.ascontiguousarray(ro, dtype=np.float32).reshape(-1, 3)
    rd = np.ascontiguousarray(rd, dtype=np.float32).reshape(-1, 3)
    m = ro.shape[0]
    mint = np.ascontiguousarray(np.broadcast_to(np.asarray(mint, dtype=np.float32), (m,)))
    maxt = np.ascontiguousarray(np.broadcast_to(np.asarray(maxt, dtype=np.float32), (m,)))
    hit = np.zeros(m, dtype=np.uint8)
    load().any_hit_ref(tri.ctypes.data_as(N.f32p), tri.size // 9, ro.ctypes.data_as(N.f32p), rd.ctypes.data_as(N.f32p),
                       mint.ctypes.data_as(N.f32p), maxt.ctypes.data_as(N.f32p), m,
                       (os.cpu_count() or 4) if threads is None else threads, hit.ctypes.data_as(N.u8p))
    return hit.astype(bool)
