#!/usr/bin/env python
"""Generates tests/golden/bre_small.npz: oracle (fp32, brute force) outputs for a small seeded case.

A regression pin of OUR restatement on camera edge 2 (the synthetic camera outside the medium), not reference output: the
reference ships no fixture for the path.  The vectors that ARE reference output - from the reference's own compiled functors -
are tests/golden/functor_pins*.npz (tests/golden/make_functor_golden.py, DESIGN.md §5).
Run from the repo root:  python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import gvpm_testlib as H  # noqa: E402
from oracle import binding as ob  # noqa: E402

P = dict(n_photons=3000, w=24, h=16, scale=4.0, seed=1234)
c = H.make_case(**P)
res = ob.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, mode="brute", neighbours=True,
                    threads=2)
np.savez_compressed(os.path.join(os.path.dirname(__file__), "bre_small.npz"), out=res.out, counts=res.counts,
                    offsets=res.offsets, idx=res.idx, **P)
print("neighbours", int(res.counts[:, 0].sum()), "contributing", int(res.counts[:, 1].sum()))

# G-Planes 0D (tests/test_oracle_planes.py)
PP = dict(n_planes=400, w=20, h=12, seed=4321)
c = H.make_plane_case(**PP)
res = ob.planes_gather(c.planes, c.rays, c.medium, c.config, neighbours=True, threads=2)
np.savez_compressed(os.path.join(os.path.dirname(__file__), "planes_small.npz"), out=res.out, counts=res.counts,
                    offsets=res.offsets, idx=res.idx, **PP)
print("plane hits", int(res.counts[:, 0].sum()))

# sppm primal photon beams, four techniques (tests/test_oracle_sppm_beams.py)
from gvpm_b200 import records as R  # noqa: E402

PB = dict(n_beams=800, w=20, h=12, scale=4.0, seed=77)
c = H.make_case(n_photons=64, w=PB["w"], h=PB["h"], scale=PB["scale"], rng_seed=99, path_set=False, max_depth=7,
                min_depth=2)
c.beams, _ = R.synth_beams(PB["n_beams"], c.medium, seed=PB["seed"], threads=2)
out = {}
for tech in sorted(ob.BEAM_TECHNIQUES):
    r = ob.sppm_beams_gather(c.beams, c.rays, c.medium, c.config, c.radius, tech, threads=2, neighbours=True)
    out["out_" + tech], out["counts_" + tech], out["offsets_" + tech], out["idx_" + tech] = r.out, r.counts, r.offsets, r.idx
    print("sppm beams", tech, "accepted", int(r.counts[:, 0].sum()), "contributing", int(r.counts[:, 1].sum()))
np.savez_compressed(os.path.join(os.path.dirname(__file__), "sppm_beams_small.npz"), **out, **PB)
