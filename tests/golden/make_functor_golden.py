"""Regenerates tests/golden/functor_pins*.npz from the REFERENCE'S OWN shift functors (oracle/_ref/libgvpm_functor_ref.so:
VolumeGradientBREQuery::operator() and VolumeGradientPositionQuery::operator(), shift_volume_photon.cpp,
BeamGradRadianceQuery::operator(), shift_volume_beams.cpp, PlaneGradRadianceQuery::operator(), shift_volume_planes.h, sppm's BeamRadianceQuery::operator(), beams.h, and BeamRadianceEstimator::query, bre.cpp,
compiled from
/root/reference by `make -C oracle functor_ref` and driven by oracle/ref_functor.cpp).  Run in the container that holds the
reference tree:
    python tests/golden/make_functor_golden.py
The vectors let tests/test_oracle_functor_pin.py hold the oracle to the reference where the tree is absent."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import __graft_entry__ as ge  # noqa: E402
import functor_pin_cases as cases  # noqa: E402
from oracle import functor_binding as fb  # noqa: E402

if __name__ == "__main__":
    ge.build_cpu_libs()
    assert fb.build_ref(), "the reference tree is needed to regenerate the vectors"
    out = {}
    for name in cases.BRE:
        c = cases.bre_case(name)
        res, calls = fb.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius)
        out[f"bre_{name}_bits"], out[f"bre_{name}_calls"], out[f"bre_{name}_crc"] = cases.bits(res), calls, cases.input_crc(c)
        print(f"bre {name:24s} functor calls {int(calls.sum()):7d}  non-zero outputs {np.count_nonzero(res):6d}")
    for name in cases.VPM:
        c = cases.vpm_case(name)
        res, mvol = fb.vpm_gather(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb)
        out[f"vpm_{name}_bits"], out[f"vpm_{name}_mvol"], out[f"vpm_{name}_crc"] = cases.bits(res), mvol, cases.input_crc(c)
        print(f"vpm {name:24s} photons found {int(mvol.sum()):7d}  non-zero outputs {np.count_nonzero(res):6d}")
    for name in cases.BEAMS:
        c = cases.beams_case(name)
        res, counts = fb.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius)
        out[f"beams_{name}_bits"], out[f"beams_{name}_contrib"] = cases.bits(res), counts[:, 0]
        out[f"beams_{name}_crc"] = cases.input_crc(c)
        print(f"beams {name:22s} contributing pairs {int(counts[:, 0].sum()):6d}  non-zero outputs {np.count_nonzero(res):6d}")
    for name in cases.PLANES:
        c = cases.planes_case(name)
        res, counts = fb.planes_gather(c.planes, c.rays, c.medium, c.config)
        out[f"planes_{name}_bits"], out[f"planes_{name}_hits"] = cases.bits(res), counts[:, 0]
        out[f"planes_{name}_crc"] = cases.input_crc(c)
        print(f"planes {name:21s} intersected pairs {int(counts[:, 0].sum()):7d}  non-zero outputs {np.count_nonzero(res):6d}"
              f"  NaN {int(np.isnan(res).sum())}")
    for name in cases.SPPM_BEAMS:
        c = cases.sppm_beams_case(name)
        for tech in cases.SPPM_BEAM_TECHNIQUES:
            res, counts = fb.sppm_beams_gather(c.beams, c.rays, c.medium, c.config, c.radius, tech)
            out[f"sppmbeams_{name}_{tech}_bits"], out[f"sppmbeams_{name}_{tech}_true"] = cases.bits(res), counts[:, 0]
            print(f"sppm beams {name:22s} {tech:13s} accepted pairs {int(counts[:, 0].sum()):6d}  non-zero {np.count_nonzero(res):5d}")
        out[f"sppmbeams_{name}_crc"] = cases.input_crc(c)
    for kind, name in cases.EDGE2:
        c = cases.edge2_case(kind, name)
        if kind == "bre":
            res = fb.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius)[0]
        elif kind == "vpm":
            res = fb.vpm_gather(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb)[0]
        elif kind == "beams":
            res = fb.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius)[0]
        else:
            res = fb.planes_gather(c.planes, c.rays, c.medium, c.config)[0]
        out[f"edge2_{kind}_{name}_bits"] = cases.bits(res)
        print(f"edge 2 {kind:6s} {name:22s} non-zero outputs {np.count_nonzero(res):6d}")
    for name in cases.SPPM_BRE:
        c = cases.sppm_bre_case(name, quantise=fb.rgbe_roundtrip)
        assert np.array_equal(fb.rgbe_roundtrip(c.photons.flux), c.photons.flux)
        res = fb.sppm_bre_gather(c.photons, c.direction, c.rays, c.medium, c.config, c.radius)
        out[f"sppmbre_{name}_bits"], out[f"sppmbre_{name}_flux_bits"] = cases.bits(res), cases.bits(c.photons.flux)
        out[f"sppmbre_{name}_crc"] = cases.input_crc(c)
        print(f"sppm bre {name:24s} non-zero outputs {np.count_nonzero(res):5d}")
    for name in cases.SPPM_PLANES:
        c = cases.sppm_planes_case(name)
        res, counts = fb.sppm_planes_gather(c.planes, c.rays, c.medium, c.config)
        out[f"sppmplanes_{name}_bits"], out[f"sppmplanes_{name}_hits"] = cases.bits(res), counts[:, 0]
        print(f"sppm planes {name:18s} hits {int(counts[:, 0].sum()):6d}")
    for name in cases.PASS:
        c = cases.bre_case(name)
        res, calls, _ = fb.bre_pass(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, threads=2)
        out[f"pass_{name}_bits"], out[f"pass_{name}_calls"] = cases.bits(res), calls
        print(f"pass {name:22s} functor calls {int(calls.sum()):7d}")
    for kind, name in cases.GLOSSY:
        c = cases.glossy_case(kind, name)
        if kind == "bre":
            res = fb.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius)[0]
        elif kind == "vpm":
            res = fb.vpm_gather(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb)[0]
        else:
            res = fb.beams_gather(c.beams, c.rays, c.medium, c.config, c.tri, c.radius)[0]
        out[f"glossy_{kind}_{name}_bits"] = cases.bits(res)
    for name in cases.PASS_VPM:
        c = cases.vpm_case(name)
        res, mvol, _ = fb.vpm_pass(c.photons, c.rays, c.samples, c.medium, c.config, c.tri, c.nb, threads=2)
        out[f"passvpm_{name}_bits"], out[f"passvpm_{name}_mvol"] = cases.bits(res), mvol
    for name in cases.PASS_BEAMS:
        c = cases.beams_case(name)
        res, acc, _ = fb.beams_pass(c.beams, c.rays, c.medium, c.config, c.tri, c.radius, threads=2)
        out[f"passbeams_{name}_bits"], out[f"passbeams_{name}_accepted"] = cases.bits(res), acc
    for name in cases.PASS_PLANES:
        c = cases.planes_case(name)
        res, _ = fb.planes_pass(c.planes, c.rays, c.medium, c.config, threads=2)
        out[f"passplanes_{name}_bits"] = cases.bits(res)
    print("whole passes of VPM / beams / planes written")
    for part in cases.GOLDEN_PARTS:
        path = os.path.join(cases.GOLDEN_DIR, part)
        np.savez_compressed(path, **{k: v for k, v in out.items() if cases.golden_part(k) == part})
        print("wrote", path, os.path.getsize(path), "bytes")
