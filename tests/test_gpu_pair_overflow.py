"""Pair-list growth.  A gather's traversal writes its (ray or sample, primitive) pairs into a grow-only list; when the
first gather on a fresh context finds more pairs than the list's initial capacity, the gather grows the list and runs
again.  Every entry point that can meet this is checked on inputs dense enough to overflow: counts and neighbour sets
equal the oracle, radiance is within 1e-4 of it, and a second gather on the grown context matches the first.

The range-halving branch of that re-run (taken when the grown list would not fit in half of the free device memory)
is not covered: it needs more pairs than a test can afford."""
import numpy as np
import pytest

import gvpm_b200 as g
from gvpm_b200 import _native as N
import gvpm_testlib as H
from gvpm_b200 import records as R

pytestmark = pytest.mark.gpu


def _bre_cap0(n_rays):    # initial pair-list capacity of the G-BRE gathers
    return max(1 << 20, 16 * n_rays)


def _beam_cap0(n_rays):   # ... of the beam gathers
    return max(1 << 20, 64 * n_rays)


def _vpm_cap0(n_samples):  # ... of the G-VPM gather
    return max(1 << 20, 8 * n_samples)


@pytest.fixture(scope="module")
def bre(built):
    from oracle import binding as ob
    c = H.make_case(n_photons=150000, w=32, h=24, scale=14.0)
    c.ref = ob.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, mode="brute", neighbours=True)
    assert c.ref.counts[:, 1].sum() > _bre_cap0(c.rays.n), "case too sparse to overflow the pair list"
    return c


def _fresh_bre_context(c):
    from gvpm_b200.api import Context
    ctx = Context(0)
    ctx.set_medium(c.medium)
    ctx.set_config(c.config)
    ctx.set_occluders(c.tri)
    ctx.upload_photons(c.photons)
    ctx.build_points(c.radius)
    return ctx


def _check_bre_neighbours(ctx, ref):
    offsets, idx = ctx.dump_neighbours_bre()
    np.testing.assert_array_equal(offsets, ref.offsets)
    np.testing.assert_array_equal(idx, ref.idx)


def test_gather_bre_overflow(bre):
    ctx = _fresh_bre_context(bre)
    ctx.upload_rays(bre.rays)
    out, counts = ctx.gather_bre()
    assert ctx.last_gather_detail()[2] > _bre_cap0(bre.rays.n)
    np.testing.assert_array_equal(counts, bre.ref.counts)
    H.assert_radiance_close(out, bre.ref.out, 1e-4, "gvpm_gather_bre, overflowed")
    _check_bre_neighbours(ctx, bre.ref)
    out2, counts2 = ctx.gather_bre()
    np.testing.assert_array_equal(counts2, counts)
    H.assert_radiance_close(out2, out, 1e-5, "gvpm_gather_bre, second gather")
    ctx.close()


def test_gather_bre_into_overflow_rerun_at_sync(bre):
    import torch
    ctx = _fresh_bre_context(bre)
    ctx.upload_rays(bre.rays)
    n = bre.rays.n

    def gather():
        out = torch.empty(n * N.GVPM_OUT_FLOATS, dtype=torch.float32, device="cuda:0")
        cnt = torch.empty(n * 2, dtype=torch.int32, device="cuda:0")
        torch.cuda.synchronize()
        ctx.gather_bre_into(out.data_ptr(), cnt.data_ptr())
        ctx.sync()   # the overflowed gather is run again here
        return (out.cpu().numpy().reshape(n, N.GVPM_OUT_FLOATS),
                cnt.cpu().numpy().view(np.uint32).reshape(n, 2))

    out, counts = gather()
    assert ctx.last_gather_detail()[2] > _bre_cap0(n)
    np.testing.assert_array_equal(counts, bre.ref.counts)
    H.assert_radiance_close(out, bre.ref.out, 1e-4, "gvpm_gather_bre_into + gvpm_sync, overflowed")
    _check_bre_neighbours(ctx, bre.ref)
    out2, counts2 = gather()
    np.testing.assert_array_equal(counts2, counts)
    H.assert_radiance_close(out2, out, 1e-5, "gvpm_gather_bre_into, second gather")
    ctx.close()


def test_gather_bre_host_overflow(bre):
    ctx = _fresh_bre_context(bre)
    out = ctx.gather_bre_host(bre.rays).copy()
    assert ctx.last_gather_detail()[2] > _bre_cap0(bre.rays.n)
    H.assert_radiance_close(out, bre.ref.out, 1e-4, "gvpm_gather_bre_host, overflowed")
    _, counts = ctx.gather_bre()
    np.testing.assert_array_equal(counts, bre.ref.counts)
    _check_bre_neighbours(ctx, bre.ref)
    out2 = ctx.gather_bre_host(bre.rays)
    H.assert_radiance_close(out2, out, 1e-5, "gvpm_gather_bre_host, second gather")
    ctx.close()


@pytest.fixture(scope="module")
def beams(built):
    c = H.make_case(n_photons=64, w=32, h=24, scale=14.0, rng_seed=1234)
    c.beams, _ = R.synth_beams(50000, c.medium, seed=5, threads=4)
    return c


def _fresh_beam_context(c):
    from gvpm_b200.api import Context
    ctx = Context(0)
    ctx.set_medium(c.medium)
    ctx.set_config(c.config)
    ctx.set_occluders(c.tri)
    ctx.upload_beams(c.beams)
    ctx.build_beams(c.radius)
    ctx.upload_rays(c.rays)
    return ctx


def test_gather_beams_overflow(beams):
    from oracle import binding as ob
    c = beams
    ref = ob.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius, neighbours=True)
    ctx = _fresh_beam_context(c)
    out, counts = ctx.gather_beams()
    assert ctx.last_gather_detail()[2] > _beam_cap0(c.rays.n)
    np.testing.assert_array_equal(counts, ref.counts)
    H.assert_radiance_close(out, ref.out, 1e-4, "gvpm_gather_beams, overflowed")
    offsets, idx = ctx.dump_neighbours_beams()
    np.testing.assert_array_equal(offsets, ref.offsets)
    np.testing.assert_array_equal(idx, ref.idx)
    out2, counts2 = ctx.gather_beams()
    np.testing.assert_array_equal(counts2, counts)
    H.assert_radiance_close(out2, out, 1e-5, "gvpm_gather_beams, second gather")
    ctx.close()


def test_gather_sppm_beams_overflow(beams):
    from oracle import binding as ob
    c = beams
    ref = ob.sppm_beams_gather(c.beams, c.rays, c.medium, c.config, c.radius, "beam3d", neighbours=True)
    ctx = _fresh_beam_context(c)
    out, counts = ctx.gather_sppm_beams("beam3d")
    assert ctx.last_gather_detail()[2] > _beam_cap0(c.rays.n)
    np.testing.assert_array_equal(counts, ref.counts)
    H.assert_radiance_close(out, ref.out, 1e-4, "gvpm_gather_sppm_beams, overflowed")
    offsets, idx = ctx.dump_neighbours_sppm_beams("beam3d")
    np.testing.assert_array_equal(offsets, ref.offsets)
    np.testing.assert_array_equal(idx, ref.idx)
    out2, counts2 = ctx.gather_sppm_beams("beam3d")
    np.testing.assert_array_equal(counts2, counts)
    H.assert_radiance_close(out2, out, 1e-5, "gvpm_gather_sppm_beams, second gather")
    ctx.close()


def test_gather_vpm_overflow(built):
    from oracle import binding as ob
    c = H.make_case(n_photons=150000, w=32, h=24, scale=10.0)
    nb = 8
    rad = np.full(c.rays.n, c.radius, dtype=np.float32)
    samples = g.synth_vpm_samples(c.rays, c.medium, rad, nb_camera_samples=nb, seed=99)
    ref = ob.vpm_gather(c.photons, c.rays, samples, c.medium, c.config, c.tri, nb, mode="brute", neighbours=True)
    ctx = H.gpu_context(c)
    ctx.upload_vpm_samples(samples)
    out, mvol, sc = ctx.gather_vpm(nb)
    assert ctx.last_gather_detail()[2] > _vpm_cap0(samples.n)
    np.testing.assert_array_equal(sc, ref.sample_counts)
    np.testing.assert_array_equal(mvol.astype(np.float32), ref.mvol)
    H.assert_radiance_close(out, ref.out, 1e-4, "gvpm_gather_vpm, overflowed")
    offsets, idx = ctx.dump_neighbours_vpm(nb)
    np.testing.assert_array_equal(offsets, ref.offsets)
    np.testing.assert_array_equal(idx, ref.idx)
    out2, mvol2, sc2 = ctx.gather_vpm(nb)
    np.testing.assert_array_equal(sc2, sc)
    np.testing.assert_array_equal(mvol2, mvol)
    H.assert_radiance_close(out2, out, 1e-5, "gvpm_gather_vpm, second gather")
    ctx.close()
