"""Rows f-1 / f-2 on triangle-mesh scenes: gvpm_trace_photons(_direct)_mesh, gvpm_trace_beams_mesh and
gvpm_generate_rays_mesh against their CPU restatement tests/mesh_trace_ref.cpp (bit-exact, every field, same light-path
count), the errors of gvpm_set_trace_mesh, statistical equivalence with the box tracer on the triangulated box, and the
progressive loop of the README on a mesh scene."""
import numpy as np
import pytest

import gvpm_b200 as g
import gvpm_testlib as H
import mesh_scenes as MS
import mesh_trace_ref as MR

pytestmark = pytest.mark.gpu

SCENES = {"cornell": MS.cornell, "sphere_field": MS.sphere_and_field, "soup": MS.soup}


def _ctx(scene, medium=None, config=None):
    from gvpm_b200.api import Context
    ctx = Context(0)
    ctx.set_medium(medium or g.make_medium())
    ctx.set_config(config or g.make_config(64, 64))
    ctx.set_trace_mesh(**scene.kwargs())
    ctx.set_occluders(scene.tri)
    return ctx


def _same_soa(a, b, what):
    assert a.n == b.n, what
    for name, dt, _ in a.FIELDS:
        x, y = getattr(a, name), getattr(b, name)
        if dt == np.float32:
            x, y = x.view(np.uint32), y.view(np.uint32)
        bad = int(np.count_nonzero(x != y))
        assert bad == 0, f"{what}: {name}: {bad} of {x.size} values differ"


@pytest.mark.parametrize("name", list(SCENES))
@pytest.mark.parametrize("kw", [
    {},
    {"phase": "hg", "hg_g": 0.6, "seed": 9},
    {"max_depth": 5, "min_depth": 2},
    {"rr_depth": 3, "seed": 3},
])
def test_traced_photons_and_beams_equal_the_restatement(built, name, kw):
    scene = SCENES[name]()
    n, seed = 20000, kw.get("seed", 1234)
    med = g.make_medium(phase=kw.get("phase", "isotropic"), g=kw.get("hg_g", 0.0))
    args = dict(max_depth=kw.get("max_depth", 12), rr_depth=kw.get("rr_depth", 1), min_depth=kw.get("min_depth", 0))
    ctx = _ctx(scene, med)
    ref, ref_paths = MR.trace_photons(scene, med, n, seed, **args)
    assert ctx.trace_photons_mesh(n, seed, **args) == ref_paths
    _same_soa(ctx.download_photons(n), ref, f"photons {name} {kw}")
    bref, bpaths = MR.trace_beams(scene, med, n // 2, seed, **args)
    assert ctx.trace_beams_mesh(n // 2, seed, **args) == bpaths
    _same_soa(ctx.download_beams(), bref, f"beams {name} {kw}")
    ctx.close()


@pytest.mark.parametrize("name", list(SCENES))
@pytest.mark.parametrize("cam", ["outside", "inside", "tilted"])
def test_generated_rays_equal_the_restatement(built, name, cam):
    scene = SCENES[name]()
    w, h = 72, 56
    if cam == "outside":
        c = g.lookat_camera(w, h, (0.5, 0.5, -1.5), tan_half_fov_x=0.32)
    elif cam == "inside":
        c = g.lookat_camera(w, h, (0.5, 0.55, 0.05), tan_half_fov_x=0.45)
    else:   # from outside, across a corner: rays enter through several faces
        c = g.lookat_camera(w, h, (-0.6, 1.4, -0.9), forward=(1.0, -0.8, 1.2), up=(0.1, 1.0, 0.0), tan_half_fov_x=0.5)
    ctx = _ctx(scene)
    for block in (32, -16):
        ref = MR.generate_rays(scene, c, 77, block=block)
        assert ctx.generate_rays_mesh(c, 77, block=block) == ref.n
        _same_soa(ctx.download_rays(), ref, f"rays {name} {cam} block {block}")
    ctx.close()


def test_direct_records_give_the_same_gather(built):
    """gvpm_trace_photons_direct_mesh writes the gather's records in place: same neighbour counts as the staged set"""
    scene = MS.sphere_and_field()
    w, h, n = 64, 48, 50000
    med, cfg = g.make_medium(), g.make_config(w, h)
    cam = g.lookat_camera(w, h, (0.5, 0.5, -1.5))
    radius = g.bre_radius(2.0)
    res = []
    for direct in (False, True):
        ctx = _ctx(scene, med, cfg)
        ctx.trace_photons_mesh(n, 77, direct=direct)
        ctx.generate_rays_mesh(cam, 78)
        ctx.build_points(radius)
        out, counts = ctx.gather_bre()
        res.append((out.copy(), counts.copy()))
        ctx.close()
    np.testing.assert_array_equal(res[0][1], res[1][1])
    H.assert_radiance_close(res[1][0], res[0][0], 1e-5, "gather on direct mesh records")
    assert res[0][1][:, 0].sum() > 1000


def test_set_trace_mesh_errors(built):
    from gvpm_b200.api import Context, GvpmError
    base = MS.cornell().kwargs()
    ctx = Context(0)
    with pytest.raises(GvpmError, match="gvpm_set_medium first"):
        ctx.trace_photons_mesh(100, 1)
    ctx.set_medium(g.make_medium())
    with pytest.raises(GvpmError, match="no mesh scene"):
        ctx.trace_photons_mesh(100, 1)
    with pytest.raises(GvpmError, match="no mesh scene"):
        ctx.generate_rays_mesh(g.lookat_camera(8, 8, (0.5, 0.5, -1)), 1)

    def bad(match, **over):
        kw = dict(base, **over)
        with pytest.raises(GvpmError, match=match):
            ctx.set_trace_mesh(**kw)
        with pytest.raises(GvpmError, match="no mesh scene"):   # a failed call leaves none
            ctx.trace_beams_mesh(100, 1)
        ctx.set_trace_mesh(**base)

    bad("empty box", hi=(1.0, 0.0, 1.0))
    bad("not finite", lo=(0.0, -np.inf, 0.0))
    t = base["tri"].copy()
    t[3, 4] = np.nan
    bad("non-finite coordinate", tri=t)
    t = base["tri"].copy()
    t[2, 0] = 1.01
    bad("outside the box", tri=t)
    t = base["tri"].copy()
    t[2, 0] = 1.0 + 5e-7   # inside the 1e-6 tolerance
    ctx.set_trace_mesh(**dict(base, tri=t))
    bad("no emissive triangle", emissive=np.zeros_like(base["emissive"]))
    t = base["tri"].copy()
    em = base["emissive"]
    t[em == 1, 6:9] = t[em == 1, 3:6]   # the light's triangles have no area
    bad("no emissive triangle", tri=t)
    a = base["albedo"].copy()
    a[0, 1] = np.inf
    bad("albedo", albedo=a)
    bad("light_power", light_power=float("nan"))
    one = np.zeros(9, np.float32)
    assert ctx.lib.gvpm_set_trace_mesh(ctx.h, None) == -1
    sc = g._native.MeshScene()
    sc.hi[0] = sc.hi[1] = sc.hi[2] = 1.0
    sc.n_tri = (1 << 24) + 1
    sc.tri = one.ctypes.data_as(g._native.f32p)
    assert ctx.lib.gvpm_set_trace_mesh(ctx.h, sc) == -1
    assert "2^24" in ctx.lib.gvpm_last_error(ctx.h).decode()
    ctx.set_trace_mesh(**base)
    with pytest.raises(GvpmError, match="max_depth must be <= 255"):
        ctx.trace_beams_mesh(100, 1, max_depth=256)
    for cam, match in [(g.lookat_camera(8, 8, (0.5, 0.5, -1), forward=(0, 0, 0)), "forward"),
                       (g.lookat_camera(8, 8, (0.5, 0.5, -1), forward=(0, 1, 0)), "parallel"),
                       (g.lookat_camera(8, 8, (0.5, 0.5, -1), tan_half_fov_x=0.0), "tan_half_fov_x")]:
        with pytest.raises(GvpmError, match=match):
            ctx.generate_rays_mesh(cam, 1)
    with pytest.raises(GvpmError, match="block"):
        ctx.generate_rays_mesh(g.lookat_camera(8, 8, (0.5, 0.5, -1)), 1, block=33)
    ctx.close()


def test_statistically_equal_to_the_box_tracer(built):
    """triangulated default box vs the box tracer: photons per light path, mean flux (4 standard errors) and a 16^3
    histogram of the photon positions, one per light path (chi-square)"""
    from scipy import stats
    n = 2_000_000
    med = g.make_medium()
    scene = MS.cornell()
    ctx = _ctx(scene, med)
    pm = ctx.trace_photons_mesh(n, 5)
    a = ctx.download_photons(n)
    pb = ctx.trace_photons(g.box_scene_default(), n, 6)
    b = ctx.download_photons(n)
    ctx.close()
    # photons per light path: n / paths, a ratio of counts; its standard error from the per-path counts' spread is
    # bounded by that of a Poisson count per path
    ra, rb = n / pm, n / pb
    se = np.sqrt(ra / pm + rb / pb) * 3.0
    assert abs(ra - rb) < 4 * se, (ra, rb, se)
    fa, fb = a.flux.reshape(-1, 3).sum(1) / pm, b.flux.reshape(-1, 3).sum(1) / pb   # flux per emitted path, per photon
    ma, mb = fa.sum(), fb.sum()
    sa, sb = fa.std() * np.sqrt(n), fb.std() * np.sqrt(n)
    assert abs(ma - mb) < 4 * np.hypot(sa, sb), (ma, mb, sa, sb)
    # photons of one light path are correlated (the histogram of all of them is over-dispersed): one per path
    def first(p):
        return p.pos.reshape(-1, 3)[np.unique(p.path_id, return_index=True)[1]]
    ha = np.histogramdd(first(a), bins=16, range=[(0, 1)] * 3)[0].ravel()
    hb = np.histogramdd(first(b), bins=16, range=[(0, 1)] * 3)[0].ravel()
    keep = (ha + hb) > 0
    chi2, p, _, _ = stats.chi2_contingency(np.stack([ha[keep], hb[keep]]))
    assert p > 1e-4, (chi2, p)


def _render(ctx, cam, w, h, iters, n, mesh):
    radius = g.bre_radius(2.0)
    ctx.accum_reset(w, h, apa=True)
    for it in range(1, iters + 1):
        if mesh:
            paths = ctx.trace_photons_mesh(n, 1000 + it, direct=True)
            ctx.generate_rays_mesh(cam, 2000 + it)
        else:
            paths = ctx.trace_photons(g.box_scene_default(), n, 1000 + it, direct=True)
            ctx.generate_rays(g.box_scene_default(), cam, 2000 + it)
        ctx.build_points_for_rays(radius, want_kept=False)
        ctx.gather_bre_device()
        ctx.accum_add()
        ctx.accum_fold(it, paths)
    return ctx.accum_read()[0]


def test_render_matches_the_box_scene_and_the_readme_loop_runs(built):
    """8 device-only G-BRE iterations at 128 x 128 with 1 M photons each, on the triangulated box and on the box: the
    mean radiance of every 16 x 16 tile agrees within the noise; the mesh loop ends in a finite reconstruction"""
    w = h = 128
    med, cfg = g.make_medium(), g.make_config(w, h)
    scene = MS.cornell()
    ctx = _ctx(scene, med, cfg)
    img_m = _render(ctx, g.lookat_camera(w, h, (0.5, 0.5, -1.5), tan_half_fov_x=0.32), w, h, 8, 1_000_000, True)
    rec = ctx.reconstruct_accum()[3]
    assert np.all(np.isfinite(rec))
    ctx.close()
    ctx = _ctx(scene, med, cfg)
    img_b = _render(ctx, g.pinhole_camera(w, h), w, h, 8, 1_000_000, False)
    ctx.close()
    lm = img_m[..., :3].sum(-1)
    lb = img_b[..., :3].sum(-1)
    tm = lm.reshape(8, 16, 8, 16).mean((1, 3))
    tb = lb.reshape(8, 16, 8, 16).mean((1, 3))
    # the noise of a tile mean from the spread of its pixels
    sm = lm.reshape(8, 16, 8, 16).std((1, 3)) / 16
    sb = lb.reshape(8, 16, 8, 16).std((1, 3)) / 16
    z = np.abs(tm - tb) / np.maximum(np.hypot(sm, sb), 1e-12)
    assert np.all(np.isfinite(tm)) and tm.sum() > 0
    assert (z > 5).sum() <= 1, z
