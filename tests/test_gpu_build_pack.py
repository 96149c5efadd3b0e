"""The staged-photon perspective-grid build packs the kept photons' records in its key pass (k_frustum_pack) and gathers
the sorted position plane from the compact plane_src copy.  Its edges: photon counts that are no multiple of a warp or a
CTA, warps whose photons are all dropped, the unsplit grid of sppm, and a smaller build after a larger one in the same
context (stale records, plane entries or keep words would show).  Every case checks the neighbour dump (bit-exact) and
the radiance against the oracle's brute force, the radiance against the forced box hierarchy (whose build still packs
with k_pack_aos_kept), and the number of kept photons against the key pass of the direct-record path (a rank
dispatching the same photons to itself)."""
import numpy as np
import pytest

import gvpm_testlib as H
from gvpm_b200 import shard

pytestmark = pytest.mark.gpu


def _context(case, monkeypatch=None, bvh=False):
    from gvpm_b200.api import Context
    if bvh:
        monkeypatch.setenv("GVPM_ACCEL", "bvh")
    ctx = Context(0)
    if bvh:
        monkeypatch.delenv("GVPM_ACCEL")
    ctx.set_medium(case.medium)
    ctx.set_config(case.config)
    ctx.set_occluders(case.tri)
    ctx.upload_rays(case.rays)
    return ctx


def _gather(ctx, sppm):
    return ctx.gather_sppm_bre() if sppm else ctx.gather_bre()


def _oracle(case, sppm):
    from oracle import binding as ob
    if sppm:
        return ob.sppm_bre_gather(case.photons, case.rays, case.medium, case.config, case.radius, mode="brute",
                                  neighbours=True)
    return ob.bre_gather(case.photons, case.rays, case.medium, case.config, case.tri, case.radius, mode="brute",
                         neighbours=True)


def _kept_direct(case):
    """photons the direct-record key pass (k_frustum_keys) keeps: one rank dispatching the whole set to itself"""
    ctx = _context(case)
    n = case.photons.n
    ctx.dispatch_connect([ctx.dispatch_export(1, n)], 0)
    ctx.photon_staging(n)
    ctx.upload_photons(case.photons)
    ctx.dispatch_photons(0, n, 0, n, case.radius)
    kept = ctx.build_dispatched(0, case.radius, want_kept=True)
    assert ctx.accel_kind() == "frustum"
    ctx.close()
    return kept


def _check_build(ctx, case, monkeypatch, what, sppm=False):
    """ctx holds case's rays and photons: build the perspective grid, compare with the oracle, the forced hierarchy and
    the direct-record key pass; returns the number of kept photons"""
    kept = ctx.build_points_for_rays(case.radius, want_kept=True)
    assert ctx.accel_kind() == "frustum", what
    assert 0 <= kept <= case.photons.n, what
    out, counts = _gather(ctx, sppm)
    ref = _oracle(case, sppm)
    np.testing.assert_array_equal(counts, ref.counts)
    H.assert_radiance_close(out, ref.out, 1e-4, what)
    if not sppm:
        offsets, idx = ctx.dump_neighbours_bre()
        np.testing.assert_array_equal(offsets, ref.offsets)
        np.testing.assert_array_equal(idx, ref.idx)
    bvh = _context(case, monkeypatch, bvh=True)
    bvh.upload_photons(case.photons)
    bvh.build_points_for_rays(case.radius, want_kept=False)
    assert bvh.accel_kind() == "bvh"
    out_bvh, counts_bvh = _gather(bvh, sppm)
    bvh.close()
    np.testing.assert_array_equal(counts, counts_bvh)
    H.assert_radiance_close(out, out_bvh, 1e-4, what + " (against the hierarchy)")
    assert kept == _kept_direct(case), what
    return kept


@pytest.mark.parametrize("n_photons", [1, 31, 33, 257, 20011])
def test_photon_counts_off_the_warp_and_cta_size(built, monkeypatch, n_photons):
    case = H.make_case(n_photons=n_photons, w=40, h=24, scale=4.0 if n_photons < 300 else 1.5)
    ctx = _context(case)
    ctx.upload_photons(case.photons)
    _check_build(ctx, case, monkeypatch, f"n = {n_photons}")
    ctx.close()


def test_band_shard_drops_whole_warps(built, monkeypatch):
    case = H.make_case(n_photons=40000 + 77, w=64, h=64, scale=0.5)
    case.rays = case.rays.take(shard.band_indices(case.rays.px, case.rays.py, 64, 64, 4, 2, 1))
    ctx = _context(case)
    ctx.upload_photons(case.photons)
    kept = _check_build(ctx, case, monkeypatch, "band shard")
    assert 0 < kept < 0.6 * case.photons.n
    ctx.close()


def test_sppm_grid_without_parity_split(built, monkeypatch):
    case = H.make_case(n_photons=30000 + 5, w=40, h=24, scale=2.0, sppm_primal=True, rng_seed=3)
    ctx = _context(case)
    ctx.upload_photons(case.photons)
    _check_build(ctx, case, monkeypatch, "sppm", sppm=True)
    ctx.close()


def test_smaller_build_after_a_larger_one(built, monkeypatch):
    big = H.make_case(n_photons=60000, w=48, h=32, scale=1.0)
    small = H.make_case(n_photons=20000 + 13, w=48, h=32, scale=1.0, seed=0xBEEF)
    small.rays = big.rays   # one ray set: the second build reuses the occupancy mask of the first
    ctx = _context(big)
    ctx.upload_photons(big.photons)
    _check_build(ctx, big, monkeypatch, "large build")
    ctx.upload_photons(small.photons)
    _check_build(ctx, small, monkeypatch, "smaller build after it")
    ctx.close()
