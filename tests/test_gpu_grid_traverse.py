"""The perspective-grid traversal (k_bre_grid_traverse): a per-tile census of the (class, grid) entries that hold
photons near the tile, then one candidate stream per lane over those entries.  Neighbour counts and index sets equal
the oracle's, radiance is within 1e-4 of it, in every traversal mode (pairs, dump, sppm) and on grids whose photons sit
in a single footprint class or all in the NEAR bucket."""
import numpy as np
import pytest

import gvpm_b200 as g
import gvpm_testlib as H

pytestmark = pytest.mark.gpu


def _check(case, what, sppm=False, oracle_mode="brute"):
    """grid gather against the oracle: counts, per-ray neighbour sets (dump mode), radiance with and without the
    traversal's prefilter; returns the oracle's result and the grid the build made"""
    from oracle import binding as ob
    ctx = H.gpu_context(case)
    ctx.build_points_for_rays(case.radius, want_kept=False)
    assert ctx.accel_kind() == "frustum", what
    grid = ctx.frustum_grid()
    out, counts = (ctx.gather_sppm_bre() if sppm else ctx.gather_bre())
    if sppm:
        ref = ob.sppm_bre_gather(case.photons, case.rays, case.medium, case.config, case.radius, mode=oracle_mode,
                                 neighbours=True)
    else:
        ref = ob.bre_gather(case.photons, case.rays, case.medium, case.config, case.tri, case.radius, mode=oracle_mode,
                            neighbours=True)
        offsets, idx = ctx.dump_neighbours_bre()
        np.testing.assert_array_equal(offsets, ref.offsets)
        # the dump lists a ray's neighbours in traversal order: compare sets, on every ray
        split = np.cumsum(np.diff(offsets.astype(np.int64)))[:-1]
        for r, (a, b) in enumerate(zip(np.split(idx, split), np.split(ref.idx, split))):
            assert np.array_equal(np.sort(a), np.sort(b)), f"{what}: ray {r}"
    np.testing.assert_array_equal(counts, ref.counts)
    H.assert_radiance_close(out, ref.out, 1e-4, what)
    if not sppm:
        out_fast, _ = ctx.gather_bre(counts=False)   # filters applied in the traversal (bench.py's path)
        H.assert_radiance_close(out_fast, ref.out, 1e-4, what + " (prefiltered)")
    ctx.close()
    return ref, grid


def _class_population(grid):
    """photons per footprint class (both parity grids) and in the NEAR bucket"""
    G, cs = grid
    cs = cs.astype(np.int64)
    grids = 2 if G.parity_split else 1
    per = [sum(int(cs[q * G.n_cells + G.base[c] + G.nx[c] * G.ny[c]] - cs[q * G.n_cells + G.base[c]])
               for q in range(grids)) for c in range(G.classes)]
    near = int(cs[grids * G.n_cells + 1] - cs[grids * G.n_cells])
    return per, near


@pytest.mark.parametrize("kw", [
    {"scale": 0.1, "n_photons": 200000, "w": 96, "h": 64},
    {"scale": 1.0, "n_photons": 60000, "w": 64, "h": 48},
    {"scale": 4.0, "n_photons": 40000, "w": 64, "h": 48},   # footprints of several cells: high classes
    {"n_photons": 30000, "w": 37, "h": 23},                 # 851 rays: the last tile holds 19
    {"n_photons": 30000, "w": 11, "h": 7, "scale": 3.0},    # every window clipped by an image border
    {"path_set": False},                                     # one grid (no parity split)
    {"max_depth": 5},
    {"path_set": False, "max_depth": 4, "use_shift_null": False},
])
def test_grid_traverse_matches_oracle(built, kw):
    case = H.make_case(**kw)
    ref, grid = _check(case, f"grid {kw}")
    assert ref.counts[:, 0].sum() > 100
    assert bool(grid[0].parity_split) == case.config.path_set


def test_grid_traverse_cfg1_size(built):
    """bench.py cfg1: 256 x 256 rays, 100 000 photons (oracle: its kd-tree, whose neighbour sets equal brute force's)"""
    case = H.make_case(n_photons=100_000, w=256, h=256, scale=1.0)
    ref, _ = _check(case, "grid cfg1", oracle_mode="kdtree")
    assert ref.counts[:, 0].sum() > 10000


def test_grid_traverse_sensor_inside_medium(built):
    """rays start at the pinhole: photons next to it go to the NEAR bucket, the rest spread over many classes"""
    case = H.make_case(n_photons=40000, w=40, h=24, scale=3.0)
    case.rays = g.synth_rays(40, 24, seed=9, cam_dist=-0.05, cover=0.45)
    ref, grid = _check(case, "grid inside")
    per, near = _class_population(grid)
    assert near > 0 and sum(1 for p in per if p) >= 3, (per, near)
    assert ref.counts[:, 0].sum() > 500


@pytest.mark.parametrize("path_set", [True, False])
def test_grid_traverse_sppm(built, path_set):
    case = H.make_case(n_photons=30000, w=40, h=24, scale=2.0, sppm_primal=True, rng_seed=3, path_set=path_set)
    _check(case, f"grid sppm path_set={path_set}", sppm=True)


def test_grid_traverse_every_photon_near(built):
    """sensor inside the medium, every photon within 2 (r + delta) of the pinhole: the NEAR bucket holds them all"""
    case = H.make_case(n_photons=20000, w=40, h=24, scale=3.0)
    C = np.array([0.5, 0.5, 0.05], dtype=np.float32)
    case.rays = g.synth_rays(40, 24, seed=9, cam_dist=-0.05, cover=0.45)
    rng = np.random.default_rng(5)
    d = rng.normal(size=(case.photons.n, 3))
    d[:, 2] = np.abs(d[:, 2])    # in front of the sensor
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rho = 1.8 * case.radius * rng.uniform(0.05, 1.0, case.photons.n) ** (1 / 3)
    case.photons.view("pos")[:] = (C + d * rho[:, None]).astype(np.float32)
    ref, grid = _check(case, "grid all NEAR")
    per, near = _class_population(grid)
    assert near == case.photons.n and sum(per) == 0, (per, near)
    assert ref.counts[:, 0].sum() > 500


def test_grid_traverse_single_class(built):
    """photons on a shell near the axis, at the distance where their footprint is 3/4 of one class's cell edge: every
    photon falls in that class"""
    from gvpm_b200.api import Context
    case = H.make_case(n_photons=40000, w=64, h=48, scale=1.0)
    ctx = Context(0)
    ctx.set_medium(case.medium)
    ctx.set_config(case.config)
    ctx.upload_photons(case.photons)
    ctx.upload_rays(case.rays)
    ctx.build_points_for_rays(case.radius, want_kept=False)
    G, _ = ctx.frustum_grid()
    ctx.close()
    pr = G.pad_r * 1.001
    # footprint ~ 1.011 pr / rho near the axis (frustum_key): a distance inside the medium whose footprint is 15 % clear
    # of both edges of its class
    cls, rho = None, None
    for r in (2.0, 1.7, 2.3, 1.85, 2.15):
        wf = 1.011 * pr / r
        c = next(c for c in range(G.classes) if G.csize[c] >= wf)
        if G.csize[c] >= 1.15 * wf and (c == 0 or G.csize[c - 1] <= wf / 1.15):
            cls, rho = c, r
            break
    assert cls is not None
    C, m, u, v = (np.array(list(x), dtype=np.float64) for x in (G.C, G.m, G.u, G.v))
    rng = np.random.default_rng(11)
    a, b = rng.uniform(-0.08, 0.08, (2, case.photons.n))
    d = m[None, :] + a[:, None] * u[None, :] + b[:, None] * v[None, :]
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    case.photons.view("pos")[:] = (C + rho * d).astype(np.float32)
    ref, grid = _check(case, "grid single class")
    per, near = _class_population(grid)
    assert near == 0 and per[cls] > 0 and sum(per) == per[cls], (cls, per, near)
    assert ref.counts[:, 0].sum() > 100


def test_grid_traverse_pair_overflow(built):
    """a fresh context whose first grid gather finds more pairs than the pair list's initial capacity (max(2^20, 16 per
    ray)) grows the list and runs again: same counts, neighbour sets and radiance as the oracle"""
    case = H.make_case(n_photons=150000, w=32, h=24, scale=14.0)
    ref, _ = _check(case, "grid overflow")
    assert ref.counts[:, 1].sum() > max(1 << 20, 16 * case.rays.n), "case too sparse to overflow the pair list"
