"""Seeded cases of the shift-functor pins (tests/test_oracle_functor_pin.py, tests/golden/make_functor_golden.py): the
flattened inputs of the C ABI, evaluated by the reference's own compiled functors (oracle/functor_binding.py) or by the
oracle restatement (oracle/binding.py).  Camera segments are first medium edges (edge_id = 1), the case the reference
harness rebuilds (oracle/ref_functor.cpp)."""
import os
import zlib

import numpy as np

import gvpm_b200 as g
import gvpm_testlib as H
from gvpm_b200 import _native as N


# The reference's outputs on these cases (tests/golden/make_functor_golden.py), stored in parts of under 1 MB each: the point
# functors, the beam / plane functors and the whole passes.
GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_PARTS = ("functor_pins.npz", "functor_pins_beams_planes.npz", "functor_pins_passes.npz")


def golden_part(key):
    """the file of GOLDEN_PARTS that holds a golden key"""
    if key.startswith("pass"):
        return GOLDEN_PARTS[2]
    if key.split("_")[0] in ("beams", "planes", "sppmbeams", "sppmplanes"):
        return GOLDEN_PARTS[1]
    return GOLDEN_PARTS[0]


def load_golden():
    """every golden key of the functor pins, read from its part"""
    out = {}
    for part in GOLDEN_PARTS:
        z = dict(np.load(os.path.join(GOLDEN_DIR, part)))
        assert all(golden_part(k) == part and k not in out for k in z), part
        out.update(z)
    return out


def _invalid_offsets(c):
    c.rays.off_valid[::3] = 0


def _xi(v):
    def f(c):
        c.rays.xi[:] = np.float32(v)
    return f


def _no_tri(c):
    c.tri = np.zeros(0, np.float32)


def _blocker(c):
    """Sheets 2e-4 above every wall of the unit box.  The reference's reconnection shadow ray only spans
    [Epsilon, |parent - offset position| * ShadowEpsilon] (shift_volume_photon.cpp:396-399: 0.1 % of the connection), so
    nothing further from the parent vertex can block it; these sheets cut the connections that leave a wall steeply."""
    e, tris = 2e-4, []
    for axis in range(3):
        for side in (e, 1.0 - e):
            u, v = [k for k in range(3) if k != axis]
            def pt(a, b):
                q = [0.0, 0.0, 0.0]
                q[axis], q[u], q[v] = side, a, b
                return q
            tris += [pt(0, 0), pt(1, 0), pt(1, 1), pt(0, 0), pt(1, 1), pt(0, 1)]
    c.tri = np.concatenate([np.asarray(c.tri, np.float32).reshape(-1), np.asarray(tris, np.float32).reshape(-1)])


# name -> (make_case keywords, post-processing)
BRE = {
    "default": (dict(), None),
    "hg_forward_0.7": (dict(phase="hg", hg_g=0.7), None),     # mean cosine > 0.5: medium vertices classify as glossy
    "hg_backward_0.4": (dict(phase="hg", hg_g=-0.4), None),
    "no_mis": (dict(use_mis=False), None),
    "wide": (dict(scale=10.0), None),                          # kernels overlap the offset rays: null shifts
    "wide_no_shift_null": (dict(scale=10.0, use_shift_null=False), None),
    "no_path_set": (dict(path_set=False), None),
    "power_heuristic_hg": (dict(power_heuristic=True, path_set=False, phase="hg", hg_g=0.3), None),
    # the reference refuses useShiftNull with a 2-D kernel at load time (gvpm_struct.h:305-311), and so does gvpm_set_config
    "kernel_2d": (dict(kernel_3d=False, use_shift_null=False), None),
    "kernel_2d_hg_no_mis": (dict(kernel_3d=False, use_shift_null=False, phase="hg", hg_g=0.4, use_mis=False), None),
    "max_depth_4": (dict(max_depth=4), None),
    "min_depth_3": (dict(min_depth=3), None),
    "surf2media": (dict(lighting_mode=N.SURF2MEDIA), None),
    "media2media": (dict(lighting_mode=N.MEDIA2MEDIA), None),
    "no_occluders": (dict(), _no_tri),
    "blocker": (dict(), _blocker),
    "blocker_wide_hg": (dict(scale=8.0, phase="hg", hg_g=0.6), _blocker),
    "invalid_offsets": (dict(), _invalid_offsets),
    "xi_0": (dict(), _xi(0.0)),
    "xi_1": (dict(), _xi(0.99999994)),
    "big": (dict(n_photons=20000, w=40, h=24, scale=2.0, seed=7, phase="hg", hg_g=0.9), None),
}

VPM = {
    "default": (dict(), None),
    "hg_forward_0.7": (dict(phase="hg", hg_g=0.7), None),
    "no_mis": (dict(use_mis=False), None),
    "wide": (dict(scale=8.0), None),
    "wide_no_shift_null": (dict(scale=8.0, use_shift_null=False), None),
    "max_depth_4": (dict(max_depth=4), None),
    "surf2media": (dict(lighting_mode=N.SURF2MEDIA), None),
    "power_heuristic": (dict(power_heuristic=True), None),
    "invalid_offsets": (dict(), _invalid_offsets),
    "blocker": (dict(), _blocker),
    "one_radius": (dict(vary_radius=False), None),
}
VPM_SAMPLES = 8

BEAMS = {
    "default": (dict(), None),                                  # beam3d (EBeamBeam3D_Optimized)
    "hg_forward_0.7": (dict(phase="hg", hg_g=0.7), None),
    "no_mis": (dict(use_mis=False), None),
    "no_shift_null": (dict(use_shift_null=False), None),
    "no_path_set": (dict(path_set=False), None),
    "power_heuristic": (dict(power_heuristic=True), None),
    "long_beams": (dict(long_beams=True), None),
    "max_depth_4": (dict(max_depth=4), None),
    "surf2media": (dict(lighting_mode=N.SURF2MEDIA), None),
    "media2media": (dict(lighting_mode=N.MEDIA2MEDIA), None),
    "blocker": (dict(), _blocker),
    "invalid_offsets": (dict(), _invalid_offsets),
    "narrow": (dict(scale=1.5, n_beams=4000), None),
    "beam1d": (dict(beam_kernel_1d=True), None),                # EBeamBeam1D with newShiftBeam (gvpm.cpp:95-98)
    "beam1d_hg_backward": (dict(beam_kernel_1d=True, phase="hg", hg_g=-0.3), None),
    "beam1d_no_mis_long": (dict(beam_kernel_1d=True, use_mis=False, long_beams=True), None),
    "beam1d_blocker": (dict(beam_kernel_1d=True), _blocker),
}


def bre_case(name):
    kw, post = BRE[name]
    kw = dict(dict(n_photons=3000, w=16, h=12, scale=3.0), **kw)
    c = H.make_case(**kw)
    c.rays.edge_id[:] = 1
    if post:
        post(c)
    return c


def vpm_case(name):
    kw, post = VPM[name]
    kw = dict(dict(n_photons=6000, w=16, h=12, scale=3.0, vary_radius=True), **kw)
    vary = kw.pop("vary_radius")
    c = H.make_case(**kw)
    c.rays.edge_id[:] = 1
    if post:
        post(c)
    rad = np.full(c.rays.n, c.radius, dtype=np.float32)
    if vary:   # per-pixel SPPM radii (gp.scaleVol, gvpm.cpp:1131,1191-1195)
        rad *= np.random.default_rng(2).uniform(0.4, 1.0, c.rays.n).astype(np.float32)
    c.samples = g.synth_vpm_samples(c.rays, c.medium, rad, nb_camera_samples=VPM_SAMPLES, seed=99)
    c.nb = VPM_SAMPLES
    return c


PLANES = {
    "default": (dict(), None),                                  # sensor inside the medium (gvpm.cpp:785-787)
    "hg_forward_0.3": (dict(phase="hg", hg_g=0.3), None),
    "hg_forward_0.7": (dict(phase="hg", hg_g=0.7), None),       # the reference itself yields NaN for some pairs here
    "hg_backward_0.5": (dict(phase="hg", hg_g=-0.5), None),
    "no_mis": (dict(use_mis=False), None),
    "sensor_outside": (dict(inside=False), None),
    "collimated_sheet": (dict(sheet=True), None),
    "invalid_offsets": (dict(), _invalid_offsets),
    "many": (dict(n_planes=4000, w=24, h=16, seed=11), None),
}


SPPM_PLANES = ("default", "hg_forward_0.3", "sensor_outside", "collimated_sheet")


def sppm_planes_case(name):
    """sppm primal planes: the same records with no valid offset edge (the gather's primal is PhotonPlaneQuery)."""
    c = planes_case(name)
    c.rays.off_valid[:] = 0
    return c


def planes_case(name):
    kw, post = PLANES[name]
    kw = dict(dict(n_planes=1200, w=16, h=12), **kw)
    c = H.make_plane_case(**kw)
    c.rays.edge_id[:] = 1
    if post:
        post(c)
    return c


SPPM_BEAM_TECHNIQUES = ("beam1d", "beam3d_naive", "beam3d_egsr", "beam3d")
SPPM_BEAMS = {
    "default": dict(),
    "hg_forward_long_beams": dict(phase="hg", hg_g=0.6, long_beams=True),
    "depth_window": dict(max_depth=5, min_depth=3),
}


def sppm_beams_case(name, unit_weight=True):
    """sppm primal beams (camera beams at depth 2: edge_id is used as sppm.cpp:853-854 uses beam.depth).  With
    unit_weight the camera beam's weight is 1, so that Li * weight (sppm.cpp:857) is Li bit for bit."""
    from gvpm_b200 import records as R
    kw = dict(dict(w=16, h=12, scale=4.0, rng_seed=99, sppm_primal=True), **SPPM_BEAMS[name])
    c = H.make_case(n_photons=64, **kw)
    c.beams, c.n_beam_paths = R.synth_beams(800, c.medium, seed=5, threads=4)
    if unit_weight:
        c.rays.eye_contrib[:] = 1.0
    return c


SPPM_BRE = {
    "kernel_3d": dict(),
    "kernel_3d_hg_forward": dict(phase="hg", hg_g=0.6),
    "kernel_2d": dict(kernel_3d=False),
    "kernel_2d_hg_backward": dict(kernel_3d=False, phase="hg", hg_g=-0.4),
    "kernel_3d_max_depth_4": dict(max_depth=4),
    "kernel_3d_wide": dict(scale=8.0),
}


def sppm_bre_case(name, quantise=None):
    """sppm primal BRE (camera beams at depth 2).  Returns the case with c.direction = photon.getDirection() and
    parent_pos = pos - direction, the ABI's flattening (include/gvpm_b200.h).  The stock Photon keeps its power in RGBE:
    `quantise` (the reference's Spectrum::toRGBE / fromRGBE round trip) makes the flux representable; without it the flux is
    left as generated (the golden file stores the quantised flux)."""
    kw = dict(dict(n_photons=3000, w=16, h=12, scale=3.0, sppm_primal=True), **SPPM_BRE[name])
    c = H.make_case(**kw)
    c.rays.eye_contrib[:] = 1.0
    pos, par = c.photons.view("pos"), c.photons.view("parent_pos")
    d = pos - par
    c.direction = (d / np.sqrt((d * d).sum(axis=1, keepdims=True))).astype(np.float32)
    par[:] = pos - c.direction
    if quantise is not None:
        c.photons.flux[:] = quantise(c.photons.flux)
    return c


def beams_case(name):
    from gvpm_b200 import records as R
    kw, post = BEAMS[name]
    kw = dict(dict(n_beams=1500, w=16, h=12, scale=4.0, rng_seed=99), **kw)
    n_beams = kw.pop("n_beams")
    c = H.make_case(n_photons=64, **kw)
    c.beams, c.n_beam_paths = R.synth_beams(n_beams, c.medium, seed=5, threads=4)
    c.rays.edge_id[:] = 1
    if post:
        post(c)
    return c


# Later camera edges (edge_id = 2, what the synthetic camera outside the medium produces): sensorMIS multiplies geometry
# and distance terms into its two factors that cancel in their product (gvpm_struct.h:608-631); the flattened form carries
# the product (off_sensor), so the agreement is up to the rounding of those terms, not bit for bit.
EDGE2 = [("bre", "default"), ("bre", "wide"), ("bre", "power_heuristic_hg"), ("bre", "blocker_wide_hg"), ("vpm", "wide"),
         ("beams", "default"), ("beams", "beam1d"), ("beams", "power_heuristic"), ("planes", "default")]


def edge2_case(kind, name):
    c = {"bre": bre_case, "vpm": vpm_case, "beams": beams_case, "planes": planes_case}[kind](name)
    c.rays.edge_id[:] = 2
    return c


# The whole G-BRE pass on the reference's own code (kd build + hierarchy + traversal + functor), sums in traversal order.
PASS = ["default", "wide", "hg_forward_0.7", "blocker_wide_hg", "big"]
# ... and of the other techniques on the reference's own structures (PointKDTree range query, SubBeamBVH, PhotonPlaneBVH)
PASS_VPM = ["default", "wide", "hg_forward_0.7", "one_radius"]
PASS_BEAMS = ["default", "beam1d", "blocker", "long_beams", "narrow"]
PASS_PLANES = ["default", "hg_forward_0.3", "sensor_outside", "many"]


# Parents that need the manifold shift (GVPM_PARENT_OTHER: a glossy surface): the reference refuses them with
# useManifold = false - null shifts still apply, every other offset keeps weight 1 and no shifted flux.  Every third photon /
# beam beyond the first bounce gets such a parent.  (CPU pin only: the synthetic scene has no glossy surface.)
GLOSSY = [("bre", "default"), ("bre", "wide"), ("bre", "no_mis"), ("vpm", "wide"), ("beams", "default"), ("beams", "beam1d")]


def glossy_case(kind, name):
    c = {"bre": bre_case, "vpm": vpm_case, "beams": beams_case}[kind](name)
    rec = c.beams if kind == "beams" else c.photons
    m = (np.arange(rec.n) % 3 == 0) & (rec.parent_type != 0)
    rec.parent_type[m] = N.PARENT_OTHER if hasattr(N, "PARENT_OTHER") else 3
    return c


def input_crc(c):
    """Fingerprint of the generated inputs: the golden outputs only mean something for exactly these arrays."""
    h = 0
    for a in (c.rays.o, c.rays.d, c.rays.off_o, c.rays.off_d, c.rays.off_valid, c.rays.xi, c.rays.eye_contrib,
              c.rays.off_sensor):
        h = zlib.crc32(np.ascontiguousarray(a).tobytes(), h)
    if hasattr(c, "photons"):
        for a in (c.photons.pos, c.photons.flux, c.photons.parent_pos, c.photons.parent_type, c.tri):
            h = zlib.crc32(np.ascontiguousarray(a).tobytes(), h)
    if hasattr(c, "planes"):
        for a in (c.planes.origin, c.planes.w0, c.planes.w1, c.planes.length0, c.planes.length1, c.planes.flux,
                  c.planes.edge_id):
            h = zlib.crc32(np.ascontiguousarray(a).tobytes(), h)
    if hasattr(c, "beams"):
        for a in (c.beams.origin, c.beams.end, c.beams.flux, c.beams.parent_type, c.beams.parent_pdf, c.beams.path_id):
            h = zlib.crc32(np.ascontiguousarray(a).tobytes(), h)
    if hasattr(c, "samples"):
        for a in (c.samples.ray, c.samples.t, c.samples.radius, c.samples.pdf_success):
            h = zlib.crc32(np.ascontiguousarray(a).tobytes(), h)
    return np.uint32(h)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def past_ray_end(c):
    """Rays with a photon of the neighbour predicate whose projection lies beyond the segment end (within a margin):
    where the reference's 2-D kernel leaves `baseProjDist > edgeLen` as an empty block (shift_volume_photon.cpp:726-731)
    and the oracle applies the explicit bound (DESIGN.md §6)."""
    p = c.photons.view("pos").astype(np.float64)
    o, d = c.rays.view("o").astype(np.float64), c.rays.view("d").astype(np.float64)
    dd = np.einsum("rpk,rk->rp", p[None, :, :] - o[:, None, :], d)
    foot = o[:, None, :] + dd[:, :, None] * d[:, None, :]
    dist2 = ((foot - p[None, :, :]) ** 2).sum(axis=2)
    r2 = float(c.radius) ** 2
    hit = (dist2 < 1.01 * r2) & (dd > c.rays.edge_len[:, None].astype(np.float64) - 1e-3)
    return hit.any(axis=1)
