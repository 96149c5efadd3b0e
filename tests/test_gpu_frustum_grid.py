"""The perspective-grid build of gvpm_build_points_for_rays (concurrent rays: every line passes through the pinhole):
same neighbour sets (bit-exact, against the oracle's brute force) and the same radiance as the box hierarchy; rays that
are not concurrent fall back to the pruned hierarchy."""
import numpy as np
import pytest

import gvpm_b200 as g
import gvpm_testlib as H
from gvpm_b200 import shard

pytestmark = pytest.mark.gpu


def _check(case, what, expect="frustum", sppm=False):
    from oracle import binding as ob
    ctx = H.gpu_context(case)
    out_bvh, counts_bvh = (ctx.gather_sppm_bre() if sppm else ctx.gather_bre())
    kept = ctx.build_points_for_rays(case.radius)
    assert ctx.accel_kind() == expect, (ctx.accel_kind(), what)
    assert 0 <= kept <= case.photons.n
    out, counts = (ctx.gather_sppm_bre() if sppm else ctx.gather_bre())
    np.testing.assert_array_equal(counts, counts_bvh)
    if sppm:
        ref = ob.sppm_bre_gather(case.photons, case.rays, case.medium, case.config, case.radius, mode="brute", neighbours=True)
    else:
        ref = ob.bre_gather(case.photons, case.rays, case.medium, case.config, case.tri, case.radius, mode="brute",
                            neighbours=True)
        offsets, idx = ctx.dump_neighbours_bre()
        np.testing.assert_array_equal(offsets, ref.offsets)
        # per-ray sets (the dump lists a ray's neighbours in traversal order)
        for r in range(0, case.rays.n, max(1, case.rays.n // 400)):
            a, b = int(offsets[r]), int(offsets[r + 1])
            assert sorted(idx[a:b].tolist()) == sorted(ref.idx[a:b].tolist()), f"{what}: ray {r}"
    np.testing.assert_array_equal(counts, ref.counts)
    H.assert_radiance_close(out, ref.out, 1e-4, what)
    if not sppm:
        out_fast, _ = ctx.gather_bre(counts=False)   # filters applied before queueing
        H.assert_radiance_close(out_fast, ref.out, 1e-4, what + " (prefiltered)")
    ctx.close()
    return ref, kept


@pytest.mark.parametrize("kw", [
    {},
    {"scale": 4.0},                              # footprints of several cells: coarser classes
    {"scale": 0.3, "n_photons": 60000},
    {"use_shift_null": False, "path_set": False},
    {"phase": "hg", "hg_g": 0.4, "max_depth": 5},
    {"kernel_3d": False, "use_shift_null": False},
])
def test_frustum_matches_oracle(built, kw):
    case = H.make_case(**kw)
    ref, kept = _check(case, f"frustum {kw}")
    assert ref.counts[:, 0].sum() > 500


def test_frustum_sensor_inside_medium(built):
    """rays start AT the pinhole: photons next to it have unbounded footprints (NEAR bucket)"""
    case = H.make_case(n_photons=40000, w=40, h=24, scale=3.0)
    case.rays = g.synth_rays(40, 24, seed=9, cam_dist=-0.05, cover=0.45)
    ref, kept = _check(case, "frustum inside")
    assert ref.counts[:, 0].sum() > 500


def test_frustum_band_shard_drops_photons(built):
    case = H.make_case(n_photons=60000, w=64, h=64, scale=0.5)
    idx = shard.band_indices(case.rays.px, case.rays.py, 64, 64, 4, 1, 1)
    case.rays = case.rays.take(idx)
    ref, kept = _check(case, "frustum band")
    assert 0 < kept < 0.6 * case.photons.n


def test_frustum_sppm(built):
    case = H.make_case(n_photons=30000, w=40, h=24, scale=2.0, sppm_primal=True, rng_seed=3)
    _check(case, "frustum sppm", sppm=True)


def test_non_concurrent_rays_use_the_hierarchy(built):
    case = H.make_case(n_photons=20000, w=32, h=32, scale=1.5)
    rng = np.random.default_rng(1)
    o = case.rays.view("o")
    o += rng.uniform(-0.02, 0.02, o.shape).astype(np.float32)      # no common point any more
    _check(case, "perturbed origins", expect="bvh")


def test_vpm_after_frustum_build_rebuilds_the_hierarchy(built):
    from oracle import binding as ob
    case = H.make_case(n_photons=30000, w=32, h=24, scale=3.0)
    ctx = H.gpu_context(case)
    ctx.build_points_for_rays(case.radius)
    assert ctx.accel_kind() == "frustum"
    rad = np.full(case.rays.n, case.radius, dtype=np.float32)
    samples = g.synth_vpm_samples(case.rays, case.medium, rad, nb_camera_samples=4, seed=5)
    ref = ob.vpm_gather(case.photons, case.rays, samples, case.medium, case.config, case.tri, 4, mode="brute")
    ctx.upload_vpm_samples(samples)
    out, mvol, sc = ctx.gather_vpm(4)
    assert ctx.accel_kind() == "bvh"
    np.testing.assert_array_equal(sc, ref.sample_counts)
    H.assert_radiance_close(out, ref.out, 1e-4, "vpm after frustum")
    ctx.close()


def test_repeated_sharded_builds_keep_the_same_count(built):
    """Repeated builds of a sharded ray set (each over a new upload of the photons): every build keeps the same number of
    photons, a small part of the set, and gives the oracle's exact neighbour counts and its radiance."""
    from oracle import binding as ob
    case = H.make_case(n_photons=80000, w=64, h=64, scale=0.5)
    idx = shard.band_indices(case.rays.px, case.rays.py, 64, 64, 8, 3, 1)
    case.rays = case.rays.take(idx)
    ref = ob.bre_gather(case.photons, case.rays, case.medium, case.config, case.tri, case.radius, mode="brute")
    ctx = H.gpu_context(case)
    outs = []
    for it in range(3):
        ctx.upload_photons(case.photons)          # a new iteration's photons
        kept = ctx.build_points_for_rays(case.radius)
        assert ctx.accel_kind() == "frustum" and 0 < kept < 0.5 * case.photons.n
        out, counts = ctx.gather_bre()
        np.testing.assert_array_equal(counts, ref.counts)
        H.assert_radiance_close(out, ref.out, 1e-4, f"sharded build {it}")
        outs.append(kept)
    assert outs[0] == outs[1] == outs[2]
    ctx.close()


def test_view_direction_does_not_change_results(built):
    """gvpm_set_view_direction only picks the projection plane of the perspective grid: same neighbour counts, same
    radiance for the default (mean ray direction), the sensor axis and a tilted axis; a zero vector is rejected"""
    from gvpm_b200.api import GvpmError
    case = H.make_case(n_photons=50000, w=64, h=48, scale=2.0)
    res = []
    for d in (None, (0.0, 0.0, 1.0), (0.3, -0.2, 1.0)):
        ctx = H.gpu_context(case)
        if d is not None:
            ctx.set_view_direction(d)
        ctx.build_points_for_rays(case.radius, want_kept=False)
        assert ctx.accel_kind() == "frustum"
        out, counts = ctx.gather_bre()
        res.append((out, counts))
        if d is not None:
            with pytest.raises(GvpmError):
                ctx.set_view_direction((0.0, 0.0, 0.0))
        ctx.close()
    for out, counts in res[1:]:
        np.testing.assert_array_equal(counts, res[0][1])
        H.assert_radiance_close(out, res[0][0], 1e-5, "view direction")
    assert res[0][1][:, 0].sum() > 2000


def test_read_bandwidth_probe(built):
    """gvpm_measure_read_bandwidth (the roofline's L2 / HBM denominators): an L2-resident sweep is faster than an HBM one"""
    from gvpm_b200.api import Context
    ctx = Context(0)
    l2 = max(ctx.measure_read_bandwidth(32 << 20, 50) for _ in range(2))
    hbm = max(ctx.measure_read_bandwidth(2 << 30, 2) for _ in range(2))
    assert l2 > hbm > 1000.0, (l2, hbm)
    ctx.close()
