"""Row f-1 for the beam and plane techniques on the device: gvpm_trace_beams and gvpm_planes_from_beams against their
CPU restatement tests/prims_ref.cpp (bit-exact, every field; number of light paths equal), the sub-beam split of
traced beams against the same beams uploaded, and the G-Beams / sppm beam / G-Planes gathers on device-made
primitives against the uploaded copies and the oracle."""
import numpy as np
import pytest

import gvpm_b200 as g
import gvpm_testlib as H
import prims_ref as PR

pytestmark = pytest.mark.gpu


def _ctx(medium=None, config=None):
    from gvpm_b200.api import Context
    ctx = Context(0)
    ctx.set_medium(medium or g.make_medium())
    ctx.set_config(config or g.make_config(64, 64))
    ctx.set_occluders(g.synth_occluders())
    return ctx


def _same_soa(a, b, what):
    assert a.n == b.n, what
    for name, dt, _ in a.FIELDS:
        x, y = getattr(a, name), getattr(b, name)
        if dt == np.float32:
            x, y = x.view(np.uint32), y.view(np.uint32)
        bad = int(np.count_nonzero(x != y))
        assert bad == 0, f"{what}: {name}: {bad} of {x.size} values differ"


def _other_scene():
    scene = g.box_scene_default()
    scene.n_rects = 2
    scene.rect[1].y, scene.rect[1].x0, scene.rect[1].x1, scene.rect[1].z0, scene.rect[1].z1 = 0.25, 0.1, 0.5, 0.1, 0.6
    for c in range(3):
        scene.rect[1].albedo[c] = 0.3 + 0.2 * c
        scene.face_albedo[2][c] = 0.2
    scene.light_x0, scene.light_x1, scene.light_power = 0.2, 0.4, 37.0
    return scene


@pytest.mark.parametrize("kw", [
    {},
    {"seed": 99, "n": 33},
    {"phase": "hg", "hg_g": 0.6, "n": 40000},
    {"max_depth": 5, "min_depth": 2, "n": 20000},
    {"rr_depth": 3, "n": 20000},
    {"n": 300000, "seed": 5},               # several blocks of the path scan, more than one batch is possible
    {"other_scene": True, "n": 30000, "seed": 3},
])
def test_traced_beams_equal_the_restatement(built, kw):
    n, seed = kw.get("n", 60000), kw.get("seed", 1234)
    med = g.make_medium(phase=kw.get("phase", "isotropic"), g=kw.get("hg_g", 0.0))
    if kw.get("other_scene"):
        med = g.make_medium(sigma_t=3.0, albedo=0.6)
    scene = _other_scene() if kw.get("other_scene") else g.box_scene_default()
    args = dict(max_depth=kw.get("max_depth", 12), rr_depth=kw.get("rr_depth", 1), min_depth=kw.get("min_depth", 0))
    ref, ref_paths = PR.trace_beams(scene, med, n, seed, **args)
    ctx = _ctx(med)
    assert ctx.trace_beams(scene, n, seed, **args) == ref_paths
    _same_soa(ctx.download_beams(), ref, f"beams {kw}")
    # a second call (the beams-per-path estimate now sizes one batch) gives the same set
    assert ctx.trace_beams(scene, n, seed, **args) == ref_paths
    _same_soa(ctx.download_beams(), ref, f"beams {kw} (second call)")
    ctx.close()


@pytest.mark.parametrize("n", [1, 33, 50000])
def test_subbeam_split_equals_the_uploaded_copy(built, n):
    """the device-side in-order length sum gives the sub-beam size and count the host sum gives for the same beams"""
    scene, med = g.box_scene_default(), g.make_medium()
    ctx = _ctx(med)
    ctx.trace_beams(scene, n, 17)
    beams = ctx.download_beams()
    traced_subs = ctx.n_subbeams()
    ctx.build_beams(g.bre_radius(3.0))
    ref = _ctx(med)
    ref.upload_beams(beams)
    assert traced_subs == ref.n_subbeams() > 0
    _same_soa(ref.download_beams(), beams, "beam staging after upload")
    # the size itself: the sub-beam cut points of the two builds are the reference's (oracle subbeams)
    from oracle import binding as ob
    t12, _ = ob.subbeams(beams)
    assert t12.shape[0] == traced_subs
    ctx.close()
    ref.close()


def _beam_case(w=40, h=24, scale=3.0, n_beams=6000, seed=5, **cfg):
    cfg.setdefault("rng_seed", 1234)
    c = H.make_case(n_photons=64, w=w, h=h, scale=scale, **cfg)
    c.scene = g.box_scene_default()
    c.seed = seed
    c.n_beams = n_beams
    return c


def _gather_both(c, run):
    """run(ctx) on a context with traced beams and on one with their uploaded copy -> (beams, traced, uploaded)"""
    res = []
    beams = None
    for traced in (True, False):
        ctx = _ctx(c.medium, c.config)
        ctx.set_occluders(c.tri)
        if traced:
            ctx.trace_beams(c.scene, c.n_beams, c.seed)
            beams = ctx.download_beams()
        else:
            ctx.upload_beams(beams)
        ctx.build_beams(c.radius)
        ctx.upload_rays(c.rays)
        res.append(run(ctx))
        ctx.close()
    return beams, res[0], res[1]


@pytest.mark.parametrize("kernel_1d", [False, True])
def test_beam_gather_on_traced_beams(built, kernel_1d):
    from oracle import binding as ob
    c = _beam_case(beam_kernel_1d=kernel_1d)

    def run(ctx):
        out, counts = ctx.gather_beams()
        offsets, idx = ctx.dump_neighbours_beams()
        return out, counts, offsets, idx
    beams, tr, up = _gather_both(c, run)
    for a, b in zip(tr[1:], up[1:]):
        np.testing.assert_array_equal(a, b)
    H.assert_radiance_close(tr[0], up[0], 1e-5, "traced vs uploaded beams")
    ref = ob.beams_gather(beams, c.rays, c.medium, c.config, c.tri, c.radius, neighbours=True)
    np.testing.assert_array_equal(tr[1], ref.counts)
    np.testing.assert_array_equal(tr[2], ref.offsets)
    np.testing.assert_array_equal(tr[3], ref.idx)
    H.assert_radiance_close(tr[0], ref.out, 1e-4, "traced beams vs oracle")
    assert ref.counts[:, 0].sum() > 3000


@pytest.mark.parametrize("tech", ["beam1d", "beam3d_naive", "beam3d_egsr", "beam3d"])
def test_sppm_beams_on_traced_beams(built, tech):
    """the naive technique hashes sub-beam ordinals: equal results pin the device-side sequential length sum"""
    from oracle import binding as ob
    c = _beam_case(max_depth=-1, rng_seed=4321)

    def run(ctx):
        out, counts = ctx.gather_sppm_beams(tech)
        offsets, idx = ctx.dump_neighbours_sppm_beams(tech)
        return out, counts, offsets, idx
    beams, tr, up = _gather_both(c, run)
    for a, b in zip(tr[1:], up[1:]):
        np.testing.assert_array_equal(a, b)
    H.assert_radiance_close(tr[0], up[0], 1e-5, f"sppm {tech}: traced vs uploaded beams")
    ref = ob.sppm_beams_gather(beams, c.rays, c.medium, c.config, c.radius, tech, neighbours=True)
    np.testing.assert_array_equal(tr[1], ref.counts)
    np.testing.assert_array_equal(tr[2], ref.offsets)
    np.testing.assert_array_equal(tr[3], ref.idx)
    H.assert_radiance_close(tr[0], ref.out, 1e-4, f"sppm {tech}: traced beams vs oracle")
    assert ref.counts[:, 0].sum() > 2000


@pytest.mark.parametrize("phase,hg_g", [("isotropic", 0.0), ("hg", 0.6), ("hg", 5e-5)])
@pytest.mark.parametrize("source", ["uploaded", "traced"])
def test_planes_from_beams_equal_the_restatement(built, phase, hg_g, source):
    from gvpm_b200 import records as R
    med = g.make_medium(phase=phase, g=hg_g)
    ctx = _ctx(med)
    if source == "traced":
        ctx.trace_beams(g.box_scene_default(), 50000, 8)
        beams = ctx.download_beams()
    else:
        beams, _ = R.synth_beams(50000, med, seed=8, threads=4)
        ctx.upload_beams(beams)
    ctx.planes_from_beams(42)
    _same_soa(ctx.download_planes(), PR.planes_from_beams(beams, med, 42), f"planes {phase} {hg_g} {source}")
    ctx.build_planes()
    ctx.close()


def test_plane_gather_on_device_made_planes(built):
    """trace beams + planes from beams + build, camera inside the medium: against the oracle on the downloaded planes"""
    from oracle import binding as ob
    w, h = 40, 24
    med, cfg = g.make_medium(), g.make_config(w, h)
    rays = g.synth_rays(w, h, seed=9, cam_dist=-0.05, cover=0.45)
    ctx = _ctx(med, cfg)
    ctx.trace_beams(g.box_scene_default(), 3000, 31)
    ctx.planes_from_beams(32)
    ctx.build_planes()
    ctx.upload_rays(rays)
    out, counts = ctx.gather_planes()
    planes = ctx.download_planes()
    assert planes.n == 3000
    ref = ob.planes_gather(planes, rays, med, cfg)
    np.testing.assert_array_equal(counts, ref.counts)
    H.assert_radiance_close(out, ref.out, 1e-4, "planes from traced beams")
    assert ref.counts[:, 0].sum() > 100
    ctx.close()


def test_error_paths(built):
    from gvpm_b200.api import Context
    scene = g.box_scene_default()
    ctx = Context(0)
    with pytest.raises(RuntimeError, match="gvpm_set_medium"):
        ctx.trace_beams(scene, 100, 1)
    with pytest.raises(RuntimeError, match="no beam set"):
        ctx.planes_from_beams(1)
    ctx.set_medium(g.make_medium())
    with pytest.raises(RuntimeError, match="max_depth"):
        ctx.trace_beams(scene, 100, 1, max_depth=256)
    assert ctx.trace_beams(scene, 0, 1) == 0          # an empty set is fine
    ctx.planes_from_beams(1)
    assert ctx.download_planes().n == 0
    ctx.trace_beams(scene, 100, 1, max_depth=255)
    ctx.set_medium(g.make_medium(sampling_weight=0.5))
    with pytest.raises(RuntimeError, match="mediumSamplingWeight must be 1"):
        ctx.planes_from_beams(1)
    ctx.close()
    fresh = Context(0)
    fresh.upload_beams(g.synth_beams(10, g.make_medium(), threads=1)[0])
    with pytest.raises(RuntimeError, match="gvpm_set_medium"):
        fresh.planes_from_beams(1)
    fresh.close()
