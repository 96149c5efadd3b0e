"""CPU: the restatement of gvpm_generate_vpm_samples (tests/vpm_samples_ref.cpp, polynomial log / exp) against
gvpm_synth_vpm_samples (libm), the host draws the device entry replaces.  Both walk the same PCG32 stream per ray in
the same operation order, so they keep the same (ray, sample) set; the values differ in the last bits only.

Bars, settled on these cases (worst seen: t 3.5e-5, pdf_success 1.0e-6, transmittance 6e-7 relative):
  - rays with a different number of samples: at most 1e-4 of the rays (a draw within rounding of the segment end);
  - on rays with sigma_t * edge_len >= 0.02 (shorter segments amplify one ulp of 1 - exp(...)): t within 1e-4,
    pdf_success and transmittance within 1e-5 relative; ray index, pdf_sel and radius exact."""
import numpy as np
import pytest

import gvpm_b200 as g
import vpm_samples_ref as P
from gvpm_b200 import _native as N

T_RTOL, PDF_RTOL, TR_RTOL = 1e-4, 1e-5, 1e-5


def _medium(coloured):
    if not coloured:
        return g.make_medium()
    m = N.Medium()
    for c, (s, a) in enumerate([(1.2, 0.3), (1.6, 0.4), (2.4, 0.2)]):
        m.sigma_s[c], m.sigma_a[c] = s, a
    m.phase_type, m.sampling_weight = N.PHASE_ISOTROPIC, 1.0
    return m


def _rays(seed=5, w=96, h=64):
    """synthetic camera rays, some made empty (0), some very short (around the 4 epsilon threshold) or short"""
    rays = g.synth_rays(w, h, seed=seed)
    rng = np.random.default_rng(seed)
    idx = rng.choice(rays.n, 400, replace=False)
    el = rays.edge_len
    el[idx[:100]] = 0.0
    el[idx[100:150]] = np.float32(4e-4)   # exactly 4 * epsilon: no draws
    el[idx[150:250]] = rng.uniform(2e-4, 1e-3, 100).astype(np.float32)
    el[idx[250:]] = rng.uniform(1e-3, 1e-2, 150).astype(np.float32)
    return rays


def _rel(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    return float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-30))) if got.size else 0.0


def _compare(rays, medium, got, ref):
    n = rays.n
    cg, cr = np.bincount(got.ray, minlength=n), np.bincount(ref.ray, minlength=n)
    same = cg == cr
    assert (~same).sum() <= 1e-4 * n, f"{(~same).sum()} of {n} rays keep a different number of samples"
    sig_min = min(medium.sigma_s[c] + medium.sigma_a[c] for c in range(3))
    keep = same & (np.float32(sig_min) * rays.edge_len >= 0.02)
    mg, mr = np.repeat(keep, cg), np.repeat(keep, cr)
    assert mg.sum() > 0.5 * got.n
    np.testing.assert_array_equal(got.ray[mg], ref.ray[mr])
    np.testing.assert_array_equal(got.pdf_sel[mg], ref.pdf_sel[mr])
    np.testing.assert_array_equal(got.radius[mg], ref.radius[mr])
    errs = (_rel(got.t[mg], ref.t[mr]), _rel(got.pdf_success[mg], ref.pdf_success[mr]),
            _rel(got.view("transmittance")[mg], ref.view("transmittance")[mr]))
    assert errs[0] <= T_RTOL and errs[1] <= PDF_RTOL and errs[2] <= TR_RTOL, errs
    return same


@pytest.mark.parametrize("stratified", [False, True])
@pytest.mark.parametrize("nb", [1, 8, 40])
@pytest.mark.parametrize("per_ray", [False, True])
def test_restatement_draws_the_synth_samples(built, stratified, nb, per_ray):
    rays = _rays()
    med = _medium(coloured=per_ray)   # the per-ray cases also run a medium whose channels differ
    rad = np.random.default_rng(3).uniform(0.01, 0.05, rays.n).astype(np.float32) if per_ray else None
    scalar = np.float32(0.03)
    ref = g.synth_vpm_samples(rays, med, rad if per_ray else scalar, nb_camera_samples=nb, stratified=stratified, seed=7)
    got = P.vpm_samples(rays, med, nb, seed=7, radius=None if per_ray else float(scalar), radius_per_ray=rad,
                        stratified=stratified)
    same = _compare(rays, med, got, ref)
    counts = np.bincount(got.ray, minlength=rays.n)
    el = rays.edge_len
    assert not counts[el <= np.float32(4e-4)].any(), "rays at or below 4 epsilon draw nothing"
    # the draws aim below edge_len - 2 epsilon: a ray past the threshold keeps every draw (or all but a rounding case)
    assert (counts[(el > np.float32(4e-4)) & same] == nb).mean() > 0.999


def test_restatement_depends_on_seed_and_stream(built):
    rays = _rays(w=32, h=16)
    med = _medium(False)
    a = P.vpm_samples(rays, med, 8, seed=1, radius=0.02)
    b = P.vpm_samples(rays, med, 8, seed=2, radius=0.02)
    assert not np.array_equal(a.t[:100], b.t[:100])
    # stratified draw i lies in stratum i of the segment's sampled CDF: t is increasing along each ray
    s = P.vpm_samples(rays, med, 8, seed=1, radius=0.02, stratified=True)
    same_ray = s.ray[1:] == s.ray[:-1]
    assert np.all(s.t[1:][same_ray] >= s.t[:-1][same_ray])
