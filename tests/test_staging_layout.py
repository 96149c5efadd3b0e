"""CPU test: gvpm_photon_staging_layout reports the field arrays of the photon staging buffer as
records._PHOTON_FIELDS describes them, each array starting on a 256-byte boundary.  Callers that fill the
staging buffer themselves (bench.py, device-side producers) place every field from these numbers."""
import ctypes as C

import pytest

from gvpm_b200 import records as R


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from gvpm_b200 import _native
    return _native.load_lib()


@pytest.mark.parametrize("n", [0, 1, 3, 1000, (1 << 20) + 7])
def test_photon_staging_layout(lib, n):
    off = (C.c_size_t * 13)()
    elt = (C.c_size_t * 13)()
    assert lib.gvpm_photon_staging_layout(n, off, elt) == 0
    want_off, want_elt, o = [], [], 0
    for _, dt, width in R._PHOTON_FIELDS:
        e = dt(0).itemsize * width
        want_off.append(o)
        want_elt.append(e)
        o += (e * n + 255) // 256 * 256
    assert list(elt) == want_elt
    assert list(off) == want_off
