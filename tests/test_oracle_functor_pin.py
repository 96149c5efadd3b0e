"""Pins the CONTROL FLOW of the oracle's shift functors against the REFERENCE'S OWN compiled functors (rows a5-a9, a11,
a13-a16 of SURVEY.md §8): VolumeGradientBREQuery::operator() (gvpm/shift/shift_volume_photon.cpp:658-856),
VolumeGradientPositionQuery::operator() (:489-655), BeamGradRadianceQuery::operator() (shift_volume_beams.cpp:139-353) and
PlaneGradRadianceQuery::operator() (shift_volume_planes.h:56-101), plus sppm's primal BeamRadianceQuery::operator()
(photonmapper/beams.h:29-223) and the loop body of BeamRadianceEstimator::query (bre.cpp:167-259; row a20), with
everything they call - the depth / lighting-mode / path-set
filters, the 3-D kernel's random chord position, shiftNull (:119-158), getTypeShift + VertexClassifier, shiftPhotonDiffuse
(:382-486) with its shadow ray and side test, getShiftPos (:858-896), the border rule, the MIS weights (balance and power
heuristic) and the accumulation.

oracle/_ref/libgvpm_functor_ref.so is built from /root/reference (oracle/Makefile, target `functor_ref`) and driven on the
flattened C-ABI inputs by oracle/ref_functor.cpp; tests/golden/functor_pins*.npz hold its outputs on the seeded cases of
tests/functor_pin_cases.py (tests/golden/make_functor_golden.py), so the pin also holds where the reference tree is
absent.  Radiance is compared BIT-EXACTLY (floats as integer bits, sums over the neighbour set in photon order)."""
import os

import numpy as np
import pytest

import functor_pin_cases as cases
import gvpm_testlib as H
from oracle import binding as ob
from oracle import functor_binding as fb



@pytest.fixture(scope="module")
def golden():
    return cases.load_golden()


def _same_rows(got, want, what, rows=None):
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    both_nan = np.isnan(got.view(np.float32)) & np.isnan(want.view(np.float32))   # the reference's own NaNs (planes, HG)
    eq = ((got == want) | both_nan).all(axis=1)
    if rows is not None:
        eq = eq | ~rows
    bad = np.flatnonzero(~eq)
    assert bad.size == 0, f"{what}: {bad.size} of {eq.size} rays differ from the reference functor (first: ray {bad[:5]})"


def test_golden_is_not_trivial(golden):
    f = lambda k: golden[k].view(np.float32)
    d = f("bre_default_bits").reshape(-1, 9, 3)
    assert (d[:, 0] > 0).any(axis=1).mean() > 0.5                          # most rays gather something
    assert not np.array_equal(d[:, 1:5], d[:, 5:9])                        # shifted != weighted base: real gradients
    # every switch the cases flip changes the reference's output
    for a, b in (("default", "no_mis"), ("wide", "wide_no_shift_null"), ("default", "no_path_set"),
                 ("default", "blocker"), ("default", "invalid_offsets"), ("default", "xi_0"),
                 ("default", "kernel_2d"), ("default", "max_depth_4"), ("default", "min_depth_3"),
                 ("default", "surf2media"), ("surf2media", "media2media")):
        assert not np.array_equal(golden[f"bre_{a}_bits"], golden[f"bre_{b}_bits"]), (a, b)
    for a, b in (("default", "no_mis"), ("wide", "wide_no_shift_null"), ("default", "power_heuristic"),
                 ("default", "invalid_offsets"), ("default", "max_depth_4"), ("default", "blocker")):
        assert not np.array_equal(golden[f"vpm_{a}_bits"], golden[f"vpm_{b}_bits"]), (a, b)
    for a, b in (("default", "no_mis"), ("default", "no_shift_null"), ("default", "no_path_set"), ("default", "blocker"),
                 ("default", "power_heuristic"), ("default", "long_beams"), ("default", "beam1d"), ("default", "max_depth_4"),
                 ("default", "invalid_offsets"), ("beam1d", "beam1d_blocker"), ("surf2media", "media2media")):
        assert not np.array_equal(golden[f"beams_{a}_bits"], golden[f"beams_{b}_bits"]), (a, b)
    for a, b in (("default", "no_mis"), ("default", "invalid_offsets"), ("default", "hg_forward_0.3"),
                 ("default", "collimated_sheet"), ("default", "sensor_outside")):
        assert not np.array_equal(golden[f"planes_{a}_bits"], golden[f"planes_{b}_bits"]), (a, b)
    assert not np.isnan(f("planes_default_bits")).any() and not np.isnan(f("planes_hg_forward_0.3_bits")).any()
    # the right and top image borders force weight 1 (no reverse shift): weighted base == primal there, < primal inside
    c = cases.bre_case("default")
    right = c.rays.px == c.w - 1
    prim, wr = d[:, 0], d[:, 6]
    lit = prim.sum(axis=1) > 0
    assert (lit & right).any() and np.array_equal(wr[right], prim[right])
    assert (wr[lit & ~right].sum(axis=1) < prim[lit & ~right].sum(axis=1)).mean() > 0.9


@pytest.mark.parametrize("name", list(cases.BRE))
def test_bre_functor_equals_reference_golden(built, golden, name):
    c = cases.bre_case(name)
    assert cases.input_crc(c) == golden[f"bre_{name}_crc"], "the seeded inputs changed: regenerate the golden vectors"
    res = ob.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, mode="brute", threads=2)
    calls = golden[f"bre_{name}_calls"]
    rows = None
    if name.startswith("kernel_2d"):
        # documented deviation (DESIGN.md §6): the reference's 2-D kernel has no bound at the segment end (an empty
        # block, shift_volume_photon.cpp:726-731; with its hierarchy the result there depends on the tree shape), the
        # oracle applies sppm's explicit bound (bre.cpp:240-242).  Rays with such a photon are left out.
        rows = ~cases.past_ray_end(c)
        assert rows.mean() > 0.9
        assert (res.counts[rows, 0] == calls[rows]).all()
    else:
        # the functor is called on the whole neighbour predicate; the oracle does not count the photons whose random
        # chord position leaves the segment (3-D kernel, :720-724: no contribution)
        assert (res.counts[:, 0] <= calls).all() and res.counts[:, 0].sum() >= 0.9 * calls.sum()
    _same_rows(cases.bits(res.out), golden[f"bre_{name}_bits"], f"G-BRE functor, case {name}", rows)


@pytest.mark.parametrize("name", list(cases.VPM))
def test_vpm_functor_equals_reference_golden(built, golden, name):
    c = cases.vpm_case(name)
    assert cases.input_crc(c) == golden[f"vpm_{name}_crc"], "the seeded inputs changed: regenerate the golden vectors"
    res = ob.vpm_gather(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb, mode="brute", threads=2)
    np.testing.assert_array_equal(res.mvol, golden[f"vpm_{name}_mvol"])     # MVol: photons the range query finds
    _same_rows(cases.bits(res.out), golden[f"vpm_{name}_bits"], f"G-VPM functor, case {name}")


@pytest.mark.parametrize("name", list(cases.BEAMS))
def test_beam_functor_equals_reference_golden(built, golden, name):
    """BeamGradRadianceQuery::operator() (shift_volume_beams.cpp:139-353) with BeamKernelRecord, shiftNull3D,
    getShiftPos / getShiftPos1D, shiftBeamDiffuse and diffuseReconnectionPhotonBeam; beam3d and beam1d kernels.  The two
    sampler draws of the kernel record are fed to the reference as the C ABI derives them."""
    c = cases.beams_case(name)
    assert cases.input_crc(c) == golden[f"beams_{name}_crc"], "the seeded inputs changed: regenerate the golden vectors"
    res = ob.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius, threads=2)
    np.testing.assert_array_equal(res.counts[:, 1], golden[f"beams_{name}_contrib"])   # calls that returned true
    _same_rows(cases.bits(res.out), golden[f"beams_{name}_bits"], f"G-Beams functor, case {name}")


@pytest.mark.parametrize("name", list(cases.PLANES))
def test_plane_functor_equals_reference_golden(built, golden, name):
    """PlaneGradRadianceQuery::operator() (shift_volume_planes.h:56-101) with specularShift (:263-416), its
    re-intersection (:427-453) and PhotonPlane::intersectPlane0D / getContrib0D / invJacobian."""
    c = cases.planes_case(name)
    assert cases.input_crc(c) == golden[f"planes_{name}_crc"], "the seeded inputs changed: regenerate the golden vectors"
    res = ob.planes_gather(c.planes, c.rays, c.medium, c.config, mode="brute", threads=2)
    np.testing.assert_array_equal(res.counts[:, 0], golden[f"planes_{name}_hits"])     # planes the base ray intersects
    _same_rows(cases.bits(res.out), golden[f"planes_{name}_bits"], f"G-Planes functor, case {name}")


@pytest.mark.parametrize("tech", cases.SPPM_BEAM_TECHNIQUES)
@pytest.mark.parametrize("name", list(cases.SPPM_BEAMS))
def test_sppm_beam_functor_equals_reference_golden(built, golden, name, tech):
    """sppm's primal BeamRadianceQuery<PhotonBeam>::operator() (photonmapper/beams.h:29-223), one call per (camera beam,
    sub-beam) of the reference's split, all four sampling techniques."""
    c = cases.sppm_beams_case(name)
    assert cases.input_crc(c) == golden[f"sppmbeams_{name}_crc"], "the seeded inputs changed: regenerate the golden vectors"
    res = ob.sppm_beams_gather(c.beams, c.rays, c.medium, c.config, c.radius, tech, threads=2)
    want, accepted = golden[f"sppmbeams_{name}_{tech}_bits"], golden[f"sppmbeams_{name}_{tech}_true"]
    rows = None
    if tech == "beam3d_naive":
        # documented deviation (DESIGN.md §6): the reference's naive branch has no camera range test (beams.h:77-102; with
        # its BVH the result then depends on which boxes the ray crosses), the oracle applies the [mint, maxt] test of the
        # other 3-D branches (:160-162).  Rays with a sample the oracle drops for that reason are left out.
        rows = res.counts[:, 1] == accepted
        assert rows.mean() > 0.7 and (res.counts[:, 1] <= accepted).all()
    else:
        np.testing.assert_array_equal(res.counts[:, 1], accepted)
    _same_rows(cases.bits(res.out), want, f"sppm beam functor, case {name}, {tech}", rows)
    if tech != "beam3d_naive":
        # with a camera-beam weight the oracle multiplies each term (Li += term * weight), the reference the sum
        # (sppm.cpp:857): equal up to the rounding of the sum
        c = cases.sppm_beams_case(name, unit_weight=False)
        res = ob.sppm_beams_gather(c.beams, c.rays, c.medium, c.config, c.radius, tech, threads=2)
        ref = want.view(np.float32) * c.rays.view("eye_contrib")
        np.testing.assert_allclose(res.out, ref, rtol=2e-6, atol=0)


@pytest.mark.parametrize("name", cases.SPPM_PLANES)
def test_sppm_plane_functor_equals_reference_golden(built, golden, name):
    """sppm's PhotonPlaneQuery::operator() (photonmapper/plane_struct.h:238-256): the plane gather with no valid offset edge
    yields it as its primal, bit for bit; nothing else is accumulated."""
    c = cases.sppm_planes_case(name)
    res = ob.planes_gather(c.planes, c.rays, c.medium, c.config, mode="brute", threads=2)
    np.testing.assert_array_equal(res.counts[:, 0], golden[f"sppmplanes_{name}_hits"])
    _same_rows(cases.bits(res.out[:, :3].copy()), golden[f"sppmplanes_{name}_bits"], f"sppm plane functor, case {name}")
    assert not res.out[:, 3:15].any()                       # no shifted contribution
    assert np.count_nonzero(golden[f"sppmplanes_{name}_bits"]) > 100


def _sppm_bre_case(golden, name):
    flux = golden[f"sppmbre_{name}_flux_bits"].view(np.float32)     # the photons' power after the reference's RGBE round trip
    c = cases.sppm_bre_case(name, quantise=lambda f: flux)
    assert cases.input_crc(c) == golden[f"sppmbre_{name}_crc"], "the seeded inputs changed: regenerate the golden vectors"
    return c


@pytest.mark.parametrize("name", list(cases.SPPM_BRE))
def test_sppm_bre_loop_body_equals_reference_golden(built, golden, name):
    """The loop body of sppm's BeamRadianceEstimator::query (photonmapper/bre.cpp:195-254) per (camera beam, photon) pair.
    Isotropic medium: bit for bit.  Henyey-Greenstein: the reference evaluates the phase function with
    wi = -photon.getDirection(), the flattened form with normalize(parent_pos - pos) where parent_pos = pos - direction
    (include/gvpm_b200.h), equal up to the rounding of that subtraction."""
    c = _sppm_bre_case(golden, name)
    res = ob.sppm_bre_gather(c.photons, c.rays, c.medium, c.config, c.radius, mode="brute", threads=2)
    want = golden[f"sppmbre_{name}_bits"]
    assert np.count_nonzero(want) > 200
    if "hg" in name:
        assert H.rel_err(res.out, want.view(np.float32)).max() < 3e-6
    else:
        _same_rows(cases.bits(res.out), want, f"sppm BRE loop body, case {name}")


@pytest.mark.skipif(not (fb.have_ref() or os.path.isdir(fb.REFERENCE_ROOT)), reason="reference tree / prebuilt library absent")
def test_golden_vectors_are_what_the_reference_computes_now(built, golden):
    """Live: the reference functors, compiled here, reproduce the committed vectors (the fixtures are not stale)."""
    if not fb.have_ref():
        assert fb.build_ref()
    for name in ("default", "hg_forward_0.7", "wide", "power_heuristic_hg", "kernel_2d", "blocker"):
        c = cases.bre_case(name)
        out, calls = fb.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius)
        np.testing.assert_array_equal(cases.bits(out), golden[f"bre_{name}_bits"])
        np.testing.assert_array_equal(calls, golden[f"bre_{name}_calls"])
    for name in ("default", "wide", "power_heuristic"):
        c = cases.vpm_case(name)
        out, mvol = fb.vpm_gather(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb)
        np.testing.assert_array_equal(cases.bits(out), golden[f"vpm_{name}_bits"])
        np.testing.assert_array_equal(mvol, golden[f"vpm_{name}_mvol"])
    for name in ("default", "beam1d", "blocker", "long_beams"):
        c = cases.beams_case(name)
        out, counts = fb.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius)
        np.testing.assert_array_equal(cases.bits(out), golden[f"beams_{name}_bits"])
        np.testing.assert_array_equal(counts[:, 0], golden[f"beams_{name}_contrib"])
    for name in ("default", "hg_forward_0.3", "sensor_outside"):
        c = cases.planes_case(name)
        out, counts = fb.planes_gather(c.planes, c.rays, c.medium, c.config)
        np.testing.assert_array_equal(cases.bits(out), golden[f"planes_{name}_bits"])
        np.testing.assert_array_equal(counts[:, 0], golden[f"planes_{name}_hits"])
    for name in ("default", "big"):
        c = cases.bre_case(name)
        out, calls, _ = fb.bre_pass(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, threads=2)
        np.testing.assert_array_equal(cases.bits(out), golden[f"pass_{name}_bits"])
        np.testing.assert_array_equal(calls, golden[f"pass_{name}_calls"])
    c = cases.vpm_case("wide")
    out, mvol, _ = fb.vpm_pass(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb, threads=2)
    np.testing.assert_array_equal(cases.bits(out), golden["passvpm_wide_bits"])
    c = cases.beams_case("blocker")
    out, acc, _ = fb.beams_pass(c.beams, c.rays, c.medium, c.config, c.tri, c.radius, threads=2)
    np.testing.assert_array_equal(cases.bits(out), golden["passbeams_blocker_bits"])
    c = cases.planes_case("many")
    out, _ = fb.planes_pass(c.planes, c.rays, c.medium, c.config, threads=2)
    np.testing.assert_array_equal(cases.bits(out), golden["passplanes_many_bits"])
    for name in ("kernel_3d", "kernel_2d_hg_backward"):
        c = _sppm_bre_case(golden, name)
        np.testing.assert_array_equal(cases.bits(fb.rgbe_roundtrip(c.photons.flux)), cases.bits(c.photons.flux))
        out = fb.sppm_bre_gather(c.photons, c.direction, c.rays, c.medium, c.config, c.radius)
        np.testing.assert_array_equal(cases.bits(out), golden[f"sppmbre_{name}_bits"])
    c = cases.sppm_beams_case("default")
    for tech in cases.SPPM_BEAM_TECHNIQUES:
        out, counts = fb.sppm_beams_gather(c.beams, c.rays, c.medium, c.config, c.radius, tech)
        np.testing.assert_array_equal(cases.bits(out), golden[f"sppmbeams_default_{tech}_bits"])
        np.testing.assert_array_equal(counts[:, 0], golden[f"sppmbeams_default_{tech}_true"])


@pytest.mark.parametrize("name", cases.PASS)
def test_whole_bre_pass_equals_reference_golden(built, golden, name):
    """The whole gather pass, not only the functor: the reference's GPhotonMap::build (PointKDTree, sliding midpoint),
    GradientBeamRadianceEstimator (hierarchy), bre->query (traversal + neighbour predicate) and VolumeGradientBREQuery per
    camera segment, i.e. the inner loop of computeVolumeGradientPhotonBRE (gvpm.cpp:994-1042), against the oracle's
    reference-shaped mode (its own kd layout + hierarchy + stack DFS): same visiting order, so the sums agree bit for bit."""
    c = cases.bre_case(name)
    res = ob.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, mode="kdtree", threads=2)
    calls = golden[f"pass_{name}_calls"]
    assert (res.counts[:, 0] <= calls).all() and res.counts[:, 0].sum() >= 0.9 * calls.sum()
    _same_rows(cases.bits(res.out), golden[f"pass_{name}_bits"], f"whole G-BRE pass, case {name}")
    # the traversal reaches a few photons in the Epsilon sliver past the ray end that the brute-force set has too, and
    # sums in tree order: the functor-level vectors agree up to that order
    assert H.rel_err(res.out, golden[f"bre_{name}_bits"].view(np.float32)).max() < 1e-5


@pytest.mark.parametrize("name", cases.PASS_VPM)
def test_whole_vpm_pass_equals_reference_golden(built, golden, name):
    """GPhotonMap::build + GPhotonMap::evaluate (PointKDTree range query) + VolumeGradientDistanceQuery per distance sample,
    folded per pixel (gvpm.cpp:1141-1185), against the oracle's reference-shaped mode: bit for bit, MVol included."""
    c = cases.vpm_case(name)
    res = ob.vpm_gather(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb, mode="kdtree", threads=2)
    np.testing.assert_array_equal(res.mvol, golden[f"passvpm_{name}_mvol"])
    _same_rows(cases.bits(res.out), golden[f"passvpm_{name}_bits"], f"whole G-VPM pass, case {name}")


@pytest.mark.parametrize("name", cases.PASS_BEAMS)
def test_whole_beam_pass_matches_reference_golden(built, golden, name):
    """SubBeamBVH<LTPhotonBeam> (sub-beam split, kd-tree, hierarchy, beams_accel.h:90-243) + BeamGradRadianceQuery per camera
    segment (gvpm.cpp:893-941): the reference's traversal hands every accepted (ray, beam) pair of the brute-force gather to
    the functor exactly once; the sums differ by the visiting order only."""
    c = cases.beams_case(name)
    res = ob.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius, threads=2)
    np.testing.assert_array_equal(res.counts[:, 1], golden[f"passbeams_{name}_accepted"])
    want = golden[f"passbeams_{name}_bits"].view(np.float32)
    assert H.rel_err(res.out, want).max() < 2e-6 and H.rel_err_per_ray(res.out, want)[0].max() < 2e-6


@pytest.mark.parametrize("name", cases.PASS_PLANES)
def test_whole_plane_pass_matches_reference_golden(built, golden, name):
    """PhotonPlaneBVH<LTPhotonPlane> (plane_accel.h:93-185) + PlaneGradRadianceQuery per camera segment (gvpm.cpp:837-841):
    same planes as the brute-force gather, sums in the reference's visiting order."""
    c = cases.planes_case(name)
    want = golden[f"passplanes_{name}_bits"].view(np.float32)
    for mode in ("brute", "kdtree"):
        res = ob.planes_gather(c.planes, c.rays, c.medium, c.config, mode=mode, threads=2)
        assert H.rel_err(res.out, want).max() < 3e-6 and H.rel_err_per_ray(res.out, want)[0].max() < 3e-6, mode


def _oracle_out(kind, c):
    if kind == "bre":
        return ob.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, mode="brute", threads=2).out
    if kind == "vpm":
        return ob.vpm_gather(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb, mode="brute", threads=2).out
    if kind == "beams":
        return ob.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius, threads=2).out
    return ob.planes_gather(c.planes, c.rays, c.medium, c.config, mode="brute", threads=2).out


@pytest.mark.parametrize("kind,name", cases.EDGE2)
def test_later_camera_edge_matches_reference_golden(built, golden, kind, name):
    """Camera segment = edge 2 of the camera path (sensor outside the medium).  The reference's sensorMIS then multiplies
    geometry and squared-distance ratios into its two factors, which cancel in their product (gvpm_struct.h:608-631); the
    flattened form carries that product, so only the rounding of the cancelling terms differs: primal bit for bit, the
    gradient terms within 2e-6."""
    c = cases.edge2_case(kind, name)
    got = _oracle_out(kind, c)
    want = golden[f"edge2_{kind}_{name}_bits"].view(np.float32)
    np.testing.assert_array_equal(cases.bits(got[:, :3]), cases.bits(want[:, :3]))
    assert H.rel_err(got, want).max() < 2e-6
    assert H.rel_err_per_ray(got, want)[0].max() < 2e-6
    if kind != "planes":   # the depth filters see the other edge id (the plane functor has none)
        assert not np.array_equal(cases.bits(got), golden[f"{kind}_{name}_bits"])


def test_persistent_passes_equal_the_one_shot_ones(built, golden):
    """bench.py's reference arms keep the reference's structures between gathers; the beam pass then draws the kernel
    record's two numbers from the C ABI's hash inside the harness instead of a table.  Same results as the pinned passes."""
    if not fb.have_ref():
        pytest.skip("prebuilt reference library absent")
    c = cases.beams_case("blocker")
    tp = fb.TechniquePass("beams", c.beams, c.medium, c.config, tri=c.tri, radius=c.radius)
    out, _ = tp.run(c.rays, threads=2)
    tp.close()
    np.testing.assert_array_equal(cases.bits(out), golden["passbeams_blocker_bits"])
    c = cases.planes_case("many")
    tp = fb.TechniquePass("planes", c.planes, c.medium, c.config)
    out, _ = tp.run(c.rays, threads=2)
    tp.close()
    np.testing.assert_array_equal(cases.bits(out), golden["passplanes_many_bits"])
    c = cases.vpm_case("wide")
    tp = fb.TechniquePass("vpm", c.photons, c.medium, c.config, tri=c.tri, threads=2)
    out, _ = tp.run(c.rays, threads=2, samples=c.samples, nb_camera_samples=c.nb)
    tp.close()
    np.testing.assert_array_equal(cases.bits(out), golden["passvpm_wide_bits"])
    c = cases.bre_case("big")
    bp = fb.BrePass(c.photons, c.medium, c.config, c.tri, c.radius, threads=2)
    out, calls, _ = bp.run(c.rays, threads=2)
    bp.close()
    np.testing.assert_array_equal(cases.bits(out), golden["pass_big_bits"])
    np.testing.assert_array_equal(calls, golden["pass_big_calls"])


@pytest.mark.parametrize("kind,name", cases.GLOSSY)
def test_glossy_parents_fail_the_shift_as_the_reference_does(built, golden, kind, name):
    """GVPM_PARENT_OTHER: a surface parent that VertexClassifier calls glossy sends getTypeShift to EManifoldShift, which the
    functors refuse with useManifold = false (shift_volume_photon.cpp:100-110, shift_volume_beams.cpp:398-407): the offset
    keeps weight 1 and no shifted flux unless the null shift applies.  Bit for bit against the reference functors."""
    c = cases.glossy_case(kind, name)
    got = _oracle_out(kind, c) if kind != "bre" else ob.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius,
                                                                   mode="brute", threads=2).out
    _same_rows(cases.bits(got), golden[f"glossy_{kind}_{name}_bits"], f"glossy parents, {kind} {name}")
    assert not np.array_equal(golden[f"glossy_{kind}_{name}_bits"], golden[f"{kind}_{name}_bits"])


def test_harness_refuses_what_it_cannot_rebuild(built):
    """Unknown parent types and camera edge 0 are outside the pin."""
    if not fb.have_ref():
        pytest.skip("prebuilt reference library absent")
    c = cases.bre_case("default")
    c.rays.edge_id[:] = 0
    with pytest.raises(RuntimeError):
        fb.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius)
    c = cases.bre_case("default")
    c.photons.parent_type[:5] = 4
    with pytest.raises(RuntimeError):
        fb.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius)
