"""CPU checks of the restated mesh-scene generators (tests/mesh_trace_ref.cpp, the checker of gvpm_trace_photons_mesh,
gvpm_trace_beams_mesh and gvpm_generate_rays_mesh): its closest hit against the box scene's analytic surfaces, its
emitter pick against the area fractions, and determinism under the seed."""
import numpy as np
import pytest
from scipy import stats

import gvpm_b200 as g
import mesh_scenes as MS
import mesh_trace_ref as MR

NONE = 0xFFFFFFFF


def _analytic_box(scene, o, d):
    """the box scene's walls, open face and rectangles (intersect_scene's rule) in float64: -> (t, surface id);
    ids 0-4 the walls x=lo, x=hi, y=lo, y=hi, z=hi, 5 the open face, 6 + r rectangle r"""
    lo, hi = np.array(scene.lo[:], np.float64), np.array(scene.hi[:], np.float64)
    m = o.shape[0]
    best, sid = np.full(m, np.inf), np.full(m, -1)
    planes = [(0, lo[0], 0), (0, hi[0], 1), (1, lo[1], 2), (1, hi[1], 3), (2, hi[2], 4), (2, lo[2], 5)]
    with np.errstate(divide="ignore", invalid="ignore"):
        for ax, pos, k in planes:
            t = (pos - o[:, ax]) / d[:, ax]
            upd = (t > 1e-6) & (t < best)
            best[upd], sid[upd] = t[upd], k
        for r in range(scene.n_rects):
            R = scene.rect[r]
            t = (R.y - o[:, 1]) / d[:, 1]
            x, z = o[:, 0] + d[:, 0] * t, o[:, 2] + d[:, 2] * t
            upd = (t > 1e-6) & (t < best) & (x >= R.x0) & (x <= R.x1) & (z >= R.z0) & (z <= R.z1)
            best[upd], sid[upd] = t[upd], 6 + r
    return best, sid


def test_closest_hit_matches_the_box_surfaces():
    box = g.box_scene_default()
    m = g.box_scene_as_mesh(box)
    keep = m["emissive"] == 0   # the box scene's light is no surface
    quad = np.repeat(np.arange(keep.sum() // 2), 2)   # two triangles per wall, then per rectangle
    surf = np.where(quad < 5, quad, quad + 1)          # the analytic ids (5 is the open face)
    scene = MR.Scene(m["tri"][keep], m["albedo"][keep], np.ones(keep.sum(), np.uint8), 1.0, m["lo"], m["hi"])
    rng = np.random.default_rng(3)
    n = 100_000
    o = rng.uniform(0.01, 0.99, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    t, tri, nrm = MR.closest(scene, o, d)
    ta, sid = _analytic_box(box, o.astype(np.float64), d.astype(np.float64))
    got = np.where(tri == NONE, 5, surf[np.minimum(tri, len(surf) - 1)])
    same = got == sid
    # a ray through the diagonal shared by a quad's two triangles may miss both (the strict test is not watertight)
    assert (~same).sum() <= 10, f"{(~same).sum()} of {n} rays hit another surface"
    rel = np.abs(t[same].astype(np.float64) - ta[same]) / ta[same]
    assert rel.max() < 8 * 2.0 ** -23, rel.max()
    hit = same & (tri != NONE)
    assert np.all(np.einsum("ij,ij->i", nrm[hit], d[hit]) <= 0), "normals face the incoming ray"


def test_self_skip_and_ties():
    # two coincident triangles: the smaller index wins; skipping it gives the other
    t0 = [(0.2, 0.5, 0.2), (0.8, 0.5, 0.2), (0.5, 0.5, 0.8)]
    scene = MR.Scene(np.array([t0, t0], np.float32), np.full((2, 3), 0.5), [1, 1], 1.0, (0, 0, 0), (1, 1, 1))
    o, d = np.array([[0.5, 0.1, 0.4]]), np.array([[0.0, 1.0, 0.0]])
    t, tri, _ = MR.closest(scene, o, d)
    assert tri[0] == 0 and abs(t[0] - 0.4) < 1e-6
    t, tri, _ = MR.closest(scene, o, d, skip=[0])
    assert tri[0] == 1
    t, tri, _ = MR.closest(scene, o, -d)   # downwards: nothing but the box exit at y = 0
    assert tri[0] == NONE and abs(t[0] - 0.1) < 1e-6


def test_emitter_pick_follows_the_areas():
    rng = np.random.default_rng(11)
    k = 12
    c = rng.uniform(0.2, 0.8, (k, 1, 3))
    tri = np.clip(c + rng.normal(0, 0.1, (k, 3, 3)) * rng.uniform(0.2, 1.5, (k, 1, 1)), 0, 1).astype(np.float32)
    em = np.ones(k, np.uint8)
    em[3] = 0   # not an emitter
    tri[5, 2] = tri[5, 1]   # zero area: never picked
    scene = MR.Scene(tri, np.full((k, 3), 0.5), em, 1.0, (0, 0, 0), (1, 1, 1))
    n = 1_000_000
    u0 = (rng.integers(0, 1 << 24, n) * (1.0 / (1 << 24))).astype(np.float32)
    got = np.bincount(MR.pick(scene, u0), minlength=k)
    e1, e2 = tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]
    area = 0.5 * np.linalg.norm(np.cross(e1, e2), axis=1) * em
    assert got[3] == 0 and got[5] == 0
    live = area > 0
    expect = area[live] / area.sum() * n
    chi2 = ((got[live] - expect) ** 2 / expect).sum()
    assert stats.chi2.sf(chi2, live.sum() - 1) > 1e-3, (got, expect)
    # u0 close to 1 clamps to the last emitter of non-zero area
    assert MR.pick(scene, np.array([np.float32(1 - 2 ** -24)]))[0] == np.nonzero(live)[0][-1]


@pytest.mark.parametrize("make", [MS.cornell, MS.soup])
def test_deterministic_under_the_seed(make):
    scene = make()
    med = g.make_medium()
    a, pa = MR.trace_photons(scene, med, 3000, 5)
    b, pb = MR.trace_photons(scene, med, 3000, 5)
    c, _ = MR.trace_photons(scene, med, 3000, 6)
    assert pa == pb and np.array_equal(a.pos, b.pos) and np.array_equal(a.flux, b.flux)
    assert not np.array_equal(a.pos, c.pos)
    assert np.all(np.isfinite(a.pos)) and np.all((a.pos >= 0) & (a.pos <= 1))
    bm, _ = MR.trace_beams(scene, med, 2000, 5)
    assert np.all(np.isfinite(bm.end))
