"""The occluder BVH (occluder_bvh.cu, occluder_device.cuh) against the flat list and the CPU oracle.

1. Any-hit bit for bit: gvpm_occluded through the BVH equals gvpm_occluded through the list on adversarial rays over
   seeded sets from 12 to 10^6 triangles, and both equal the oracle's Occluders::anyHit over the whole list (tests/any_hit_ref.cpp) where the CPU affords it.
2. Whole gathers (G-BRE 3D / 2D, G-VPM, G-Beams 3D / 1D) on a scene of a few thousand occluders, AUTO selecting the
   BVH: neighbour index sets and counts bit-exact against the oracle, radiance within 1e-4 (globally floored and per
   ray); the forced list gives the same counts and radiance within 1e-6.
3. The reference's own functor output (tests/golden/functor_pins*.npz) with the BVH forced.
4. State: switching between large and small sets, n_tri = 0, the AUTO selection, invalid modes."""
import numpy as np
import pytest

import any_hit_ref as AH
import functor_pin_cases as cases
import gvpm_testlib as H
import occluder_sets as S
from oracle import binding as ob

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def _ctx():
    from gvpm_b200.api import Context
    return Context(0)


def _both(ctx, tri, rays):
    ctx.set_occluders(tri)
    ctx.set_occluder_accel("bvh")
    assert ctx.occluder_accel() == ("bvh" if len(tri) else "list")
    bvh = ctx.occluded(*rays)
    ctx.set_occluder_accel("list")
    assert ctx.occluder_accel() == "list"
    lst = ctx.occluded(*rays)
    ctx.set_occluder_accel("auto")
    return bvh, lst


def _report(a, b, rays, what):
    bad = np.flatnonzero(a != b)
    if bad.size:
        i = bad[0]
        o, d, mint, maxt = (np.asarray(x)[i] for x in rays)
        pytest.fail(f"{what}: {bad.size} of {a.size} rays differ; first: o={o.tolist()} d={d.tolist()} "
                    f"mint={float(mint)!r} maxt={float(maxt)!r} ({a[i]} vs {b[i]})")


SETS = {
    "walls": (S.walls, 20000),
    "blocker": (lambda: np.concatenate([S.walls(), S.blocker_sheets()]), 20000),
    "blocker_grid_50k": (lambda: S.blocker_sheets(cells=64), 2000),
    "sphere_20k": (lambda: S.uv_sphere(128, 80), 4000),
    "soup_100k": (lambda: S.soup(100000), 1000),
    "soup_100k_shifted": (lambda: S.soup(100000, shift=1000.0), 1000),
    "oracle_5k": (lambda: np.concatenate([S.walls(), S.blocker_sheets(cells=8), S.uv_sphere(48, 24),
                                          S.soup(2000, seed=9, size=0.03)]), 20000),
}


@pytest.mark.parametrize("name", list(SETS))
def test_bvh_any_hit_equals_list_and_oracle(built, name):
    make, n_oracle = SETS[name]
    tri = make()
    rays = S.adversarial_rays(tri, n=40000, seed=21)
    ctx = _ctx()
    bvh, lst = _both(ctx, tri, rays)
    ctx.close()
    _report(bvh, lst, rays, f"{name}: BVH vs list")
    assert bvh.any() and not bvh.all(), f"{name}: vacuous ray set"
    sub = tuple(np.asarray(x)[:: max(1, len(x) // n_oracle)] for x in rays)
    sel = np.arange(0, len(rays[0]), max(1, len(rays[0]) // n_oracle))
    ref = AH.any_hit(tri, *sub)
    _report(lst[sel], ref, sub, f"{name}: list vs oracle")
    _report(bvh[sel], ref, sub, f"{name}: BVH vs oracle")


def test_bvh_any_hit_height_field_1m(built):
    tri = S.height_field(708)
    assert len(tri) > 990000
    rays = S.adversarial_rays(tri, n=4000, seed=23)
    ctx = _ctx()
    bvh, lst = _both(ctx, tri, rays)
    ctx.close()
    _report(bvh, lst, rays, "height field: BVH vs list")
    assert bvh.any() and not bvh.all()


# ---- whole gathers on a many-occluder scene ------------------------------------------------------------------------
def _scene_tri():
    return np.concatenate([S.walls(), S.blocker_sheets(cells=12), S.uv_sphere(40, 24, r=0.2)]).astype(np.float32)


def _bre(kernel_3d):
    kw = {} if kernel_3d else dict(kernel_3d=False, use_shift_null=False)
    c = H.make_case(n_photons=12000, w=24, h=16, scale=3.0, **kw)
    c.tri = _scene_tri()
    ref = ob.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, mode="brute", neighbours=True)
    ctx = H.gpu_context(c)
    assert ctx.occluder_accel() == "bvh"
    out, counts = ctx.gather_bre()
    offsets, idx = ctx.dump_neighbours_bre()
    np.testing.assert_array_equal(counts, ref.counts)
    np.testing.assert_array_equal(offsets, ref.offsets)
    np.testing.assert_array_equal(idx, ref.idx)
    ctx.set_occluder_accel("list")
    out_l, counts_l = ctx.gather_bre()
    ctx.set_occluders(np.zeros(0, np.float32))
    out_0, _ = ctx.gather_bre()
    ctx.close()
    return out, ref.out, counts, counts_l, out_l, out_0


def _vpm():
    import gvpm_b200 as g
    c = H.make_case(n_photons=20000, w=24, h=16, scale=3.0)
    c.tri = _scene_tri()
    rad = np.full(c.rays.n, c.radius, dtype=np.float32)
    c.samples = g.synth_vpm_samples(c.rays, c.medium, rad, nb_camera_samples=8, seed=99)
    ref = ob.vpm_gather(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, 8, mode="brute", neighbours=True)
    ctx = H.gpu_context(c)
    ctx.upload_vpm_samples(c.samples)
    assert ctx.occluder_accel() == "bvh"
    out, mvol, sc = ctx.gather_vpm(8)
    offsets, idx = ctx.dump_neighbours_vpm(8)
    np.testing.assert_array_equal(sc, ref.sample_counts)
    np.testing.assert_array_equal(offsets, ref.offsets)
    np.testing.assert_array_equal(idx, ref.idx)
    ctx.set_occluder_accel("list")
    out_l, _, sc_l = ctx.gather_vpm(8)
    ctx.set_occluders(np.zeros(0, np.float32))
    out_0, _, _ = ctx.gather_vpm(8)
    ctx.close()
    return out, ref.out, sc, sc_l, out_l, out_0


def _beams(k1d):
    from gvpm_b200 import records as R
    c = H.make_case(n_photons=64, w=24, h=16, scale=3.0, rng_seed=1234, beam_kernel_1d=k1d)
    c.beams, _ = R.synth_beams(3000, c.medium, seed=5, threads=4)
    c.tri = _scene_tri()
    ref = ob.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius, neighbours=True)
    from gvpm_b200.api import Context
    ctx = Context(0)
    ctx.set_medium(c.medium)
    ctx.set_config(c.config)
    ctx.set_occluders(c.tri)
    ctx.upload_beams(c.beams)
    ctx.build_beams(c.radius)
    ctx.upload_rays(c.rays)
    assert ctx.occluder_accel() == "bvh"
    out, counts = ctx.gather_beams()
    offsets, idx = ctx.dump_neighbours_beams()
    np.testing.assert_array_equal(counts, ref.counts)
    np.testing.assert_array_equal(offsets, ref.offsets)
    np.testing.assert_array_equal(idx, ref.idx)
    ctx.set_occluder_accel("list")
    out_l, counts_l = ctx.gather_beams()
    ctx.set_occluders(np.zeros(0, np.float32))
    out_0, _ = ctx.gather_beams()
    ctx.close()
    return out, ref.out, counts, counts_l, out_l, out_0


@pytest.mark.parametrize("what", ["bre3d", "bre2d", "vpm", "beams3d", "beams1d"])
def test_gathers_with_many_occluders(built, what):
    run = {"bre3d": lambda: _bre(True), "bre2d": lambda: _bre(False), "vpm": _vpm,
           "beams3d": lambda: _beams(False), "beams1d": lambda: _beams(True)}[what]
    out, ref, counts, counts_l, out_l, out_0 = run()
    H.assert_radiance_close(out, ref, RTOL, f"{what} BVH vs oracle")
    np.testing.assert_array_equal(counts, counts_l)
    H.assert_radiance_close(out_l, out, 1e-6, f"{what} list vs BVH")
    # the occluders matter: the weighted flux of at least 1 % of the rays changes without them
    w, w0 = np.asarray(out)[:, 15:27], np.asarray(out_0)[:, 15:27]
    changed = (np.abs(w - w0) > 1e-6 * np.abs(w0).max()).any(axis=1).mean()
    assert changed >= 0.01, f"{what}: occluders change only {changed:.2%} of the rays"


# ---- the reference's own output, BVH forced --------------------------------------------------------------------------
@pytest.fixture(scope="module")
def golden():
    return cases.load_golden()


def _close(got, want_bits, what, rows=None):
    want = want_bits.view(np.float32)
    got = np.asarray(got, dtype=np.float32).reshape(want.shape)
    if rows is not None:
        got, want = got[rows], want[rows]
    finite = np.isfinite(want).all(axis=1)
    got, want = got[finite], want[finite]
    assert np.abs(want).max() > 0, f"{what}: empty case"
    assert H.rel_err(got, want).max() <= RTOL, what
    assert H.rel_err_per_ray(got, want)[0].max() <= RTOL, what


@pytest.mark.parametrize("name", list(cases.BRE))
def test_bre_reference_output_bvh_forced(built, golden, name):
    c = cases.bre_case(name)
    ctx = H.gpu_context(c)
    ctx.set_occluder_accel("bvh")
    out, counts = ctx.gather_bre()
    ctx.close()
    calls = golden[f"bre_{name}_calls"]
    rows = None
    if name.startswith("kernel_2d"):   # documented deviation at the segment end (DESIGN.md §6)
        rows = ~cases.past_ray_end(c)
        assert (counts[rows, 0] == calls[rows]).all()
    else:
        assert (counts[:, 0] <= calls).all() and counts[:, 0].sum() >= 0.9 * calls.sum()
    _close(out, golden[f"bre_{name}_bits"], f"G-BRE {name}", rows)


@pytest.mark.parametrize("name", list(cases.VPM))
def test_vpm_reference_output_bvh_forced(built, golden, name):
    c = cases.vpm_case(name)
    ctx = H.gpu_context(c)
    ctx.set_occluder_accel("bvh")
    ctx.upload_vpm_samples(c.samples)
    out, mvol, _ = ctx.gather_vpm(c.nb)
    ctx.close()
    np.testing.assert_array_equal(np.asarray(mvol, dtype=np.float32), golden[f"vpm_{name}_mvol"])
    _close(out, golden[f"vpm_{name}_bits"], f"G-VPM {name}")


@pytest.mark.parametrize("name", list(cases.BEAMS))
def test_beams_reference_output_bvh_forced(built, golden, name):
    from gvpm_b200.api import Context
    c = cases.beams_case(name)
    ctx = Context(0)
    ctx.set_occluder_accel("bvh")
    ctx.set_medium(c.medium)
    ctx.set_config(c.config)
    ctx.set_occluders(c.tri)
    ctx.upload_beams(c.beams)
    ctx.build_beams(c.radius)
    ctx.upload_rays(c.rays)
    out, counts = ctx.gather_beams()
    ctx.close()
    np.testing.assert_array_equal(counts[:, 1], golden[f"beams_{name}_contrib"])
    _close(out, golden[f"beams_{name}_bits"], f"G-Beams {name}")


# ---- state -----------------------------------------------------------------------------------------------------------
def test_occluder_state(built):
    from gvpm_b200.api import GvpmError
    ctx = _ctx()
    assert ctx.occluder_accel() == "list"                     # no occluders
    small, large = S.walls(), S.uv_sphere(24, 12)
    rays = S.adversarial_rays(large, n=4000, seed=3)
    ref_small, ref_large = AH.any_hit(small, *rays), AH.any_hit(large, *rays)
    for _ in range(2):                                          # large -> small -> large ...
        ctx.set_occluders(large)
        assert ctx.occluder_accel() == "bvh"
        np.testing.assert_array_equal(ctx.occluded(*rays), ref_large)
        ctx.set_occluders(small)
        assert ctx.occluder_accel() == "list"
        np.testing.assert_array_equal(ctx.occluded(*rays), ref_small)
    ctx.set_occluder_accel("bvh")                               # forced on a small set
    assert ctx.occluder_accel() == "bvh"
    np.testing.assert_array_equal(ctx.occluded(*rays), ref_small)
    ctx.set_occluders(large[:32])                               # AUTO boundary: 32 -> list, 33 -> BVH
    ctx.set_occluder_accel("auto")
    assert ctx.occluder_accel() == "list"
    ctx.set_occluders(large[:33])
    assert ctx.occluder_accel() == "bvh"
    np.testing.assert_array_equal(ctx.occluded(*rays), AH.any_hit(large[:33], *rays))
    ctx.set_occluders(np.zeros(0, np.float32))                  # n_tri = 0: nothing is hit on either path
    for mode in ("auto", "list", "bvh"):
        ctx.set_occluder_accel(mode)
        assert not ctx.occluded(*rays).any()
    assert ctx.lib.gvpm_set_occluder_accel(ctx.h, 3) == -1      # GVPM_ERR_INVALID
    assert ctx.lib.gvpm_set_occluder_accel(ctx.h, -1) == -1
    with pytest.raises(ValueError):
        ctx.set_occluder_accel("kd")
    one = np.zeros(9, np.float32)                               # above GVPM_MAX_OCCLUDERS: refused before any read
    from gvpm_b200 import _native as N
    assert ctx.lib.gvpm_set_occluders(ctx.h, one.ctypes.data_as(N.f32p), (1 << 24) + 1) == -1
    with pytest.raises(GvpmError):
        ctx._ck(ctx.lib.gvpm_set_occluder_accel(ctx.h, 7), "gvpm_set_occluder_accel")
    ctx.close()
