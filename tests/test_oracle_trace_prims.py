"""CPU checks of the restated beam tracer and plane maker (tests/prims_ref.cpp, the checker of gvpm_trace_beams and
gvpm_planes_from_beams): determinism, the beams pinned to the photon walk of oracle/gvpm_oracle_trace.cpp (same walk,
the photons are exactly the beams that end in the medium), and the invariants of the planes."""
import numpy as np
import pytest

import gvpm_b200 as g
import prims_ref as PR
from oracle import binding as ob


def _bits(a):
    return a.view(np.uint32) if a.dtype == np.float32 else a


def _v3(a):
    return a.reshape(-1, 3)


def test_beams_are_deterministic_and_seeded(built):
    scene, med = g.box_scene_default(), g.make_medium()
    a, pa = PR.trace_beams(scene, med, 20000, seed=7)
    b, pb_ = PR.trace_beams(scene, med, 20000, seed=7)
    c, _ = PR.trace_beams(scene, med, 20000, seed=8)
    for name, _, _ in a.FIELDS:
        assert np.array_equal(_bits(getattr(a, name)), _bits(getattr(b, name))), name
    assert pa == pb_ > 0
    assert not np.array_equal(a.origin, c.origin)
    # path ids count the contributing paths: non-decreasing from 0, by steps of at most one
    steps = np.diff(a.path_id.astype(np.int64))
    assert a.path_id[0] == 0 and steps.min() >= 0 and steps.max() <= 1
    assert a.depth.min() >= 1 and a.end_on_surface.any() and not a.end_on_surface.all()
    # end_n is the surface normal of surface ends, zero in the medium
    assert np.all(_v3(a.end_n)[a.end_on_surface == 0] == 0)
    assert np.allclose(np.linalg.norm(_v3(a.end_n)[a.end_on_surface == 1], axis=1), 1.0)


@pytest.mark.parametrize("kw", [{}, {"phase": "hg", "hg_g": 0.6}, {"min_depth": 2, "max_depth": 6}])
def test_beams_pinned_to_the_photon_walk(built, kw):
    """the photons of oracle.trace_photons are the beams that end in the medium, in order, for the same seed"""
    scene = g.box_scene_default()
    med = g.make_medium(phase=kw.get("phase", "isotropic"), g=kw.get("hg_g", 0.0))
    args = dict(max_depth=kw.get("max_depth", 12), min_depth=kw.get("min_depth", 0))
    n = 30000
    beams, _ = PR.trace_beams(scene, med, n, 11, **args)
    photons, _ = ob.trace_photons(scene, med, n, 11, **args)
    inside = np.flatnonzero(beams.end_on_surface == 0)
    m = min(inside.size, n)
    assert m > n // 4
    sel, ph = inside[:m], np.arange(m)
    pairs = [("end", "pos"), ("origin", "parent_pos"), ("depth", "depth"), ("parent_pdf", "parent_pdf"),
             ("prefix_flux", "prefix_flux"), ("rr_weight", "rr_weight"), ("parent_type", "parent_type"),
             ("pred_pos", "pred_pos"), ("parent_n", "parent_n"), ("parent_albedo", "parent_albedo")]
    for bname, pname in pairs:
        x, y = getattr(beams, bname), getattr(photons, pname)
        if x.size == 3 * n:
            x, y = _v3(x), _v3(y)
        x, y = _bits(x[sel]), _bits(y[ph])
        assert np.array_equal(x, y), f"beam {bname} != photon {pname}"
    assert beams.depth.min() >= max(1, args["min_depth"])


@pytest.mark.parametrize("phase,hg_g", [("isotropic", 0.0), ("hg", 0.6), ("hg", -0.4), ("hg", 5e-5)])
def test_planes_from_beams(built, phase, hg_g):
    scene, med = g.box_scene_default(), g.make_medium(phase=phase, g=hg_g)
    beams, _ = PR.trace_beams(scene, med, 40000, 3)
    planes = PR.planes_from_beams(beams, med, 5)
    again = PR.planes_from_beams(beams, med, 5)
    for name, _, _ in planes.FIELDS:
        assert np.array_equal(_bits(getattr(planes, name)), _bits(getattr(again, name))), name
    w0, w1 = _v3(planes.w0).astype(np.float64), _v3(planes.w1).astype(np.float64)
    assert np.allclose(np.linalg.norm(w1, axis=1), 1.0, atol=2e-6)
    assert planes.length1.min() > 1e-4
    assert np.array_equal(planes.origin, beams.origin)
    assert np.array_equal(planes.flux, beams.flux)
    assert np.array_equal(planes.edge_id, beams.depth.astype(np.int32))
    d = _v3(beams.end).astype(np.float64) - _v3(beams.origin)
    length0 = np.linalg.norm(d, axis=1)
    assert np.allclose(planes.length0, length0, rtol=1e-6)
    assert np.allclose(w0, d / length0[:, None], atol=1e-6)
    # the free flights are exponential with rate sigma_t: mean 1 / sigma_t
    sigma_t = float(med.sigma_s[1] + med.sigma_a[1])
    assert abs((planes.length1 - 1e-4).mean() * sigma_t - 1.0) < 0.02
    cos = np.einsum("ij,ij->i", w0, w1)
    if phase == "isotropic" or abs(hg_g) < 1e-4:
        assert np.abs(w1.mean(axis=0)).max() < 0.02
        assert abs(cos.mean()) < 0.02
    else:
        assert abs(cos.mean() - hg_g) < 0.02   # the mean cosine of Henyey-Greenstein is g


def test_planes_need_unit_sampling_weight(built):
    med = g.make_medium(sampling_weight=0.5)
    beams, _ = PR.trace_beams(g.box_scene_default(), g.make_medium(), 100, 1)
    with pytest.raises(RuntimeError):
        PR.planes_from_beams(beams, med, 1)
