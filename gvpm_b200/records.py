"""Host-side containers for the flattened inputs of the gather (numpy SoA <-> C structs).

PhotonSet mirrors what GPhotonMap holds after tryAppend (gvpm/gvpm_accel.h:119-199) and RaySet the
(gather point, medium edge) list computeVolumeGradientPhotonBRE walks (gvpm.cpp:1008-1042) with
the four ShiftGatherPoint records (gvpm/shift/shift_cameraPath.h).  Layout = include/gvpm_b200.h.
"""
import ctypes as C

import numpy as np

from . import _native as N

_PHOTON_FIELDS = [
    ("pos", np.float32, 3), ("flux", np.float32, 3), ("parent_pos", np.float32, 3),
    ("pred_pos", np.float32, 3), ("parent_n", np.float32, 3), ("prefix_flux", np.float32, 3),
    ("parent_albedo", np.float32, 3), ("parent_pdf", np.float32, 1), ("edge_pdf", np.float32, 1),
    ("rr_weight", np.float32, 1), ("parent_type", np.uint8, 1), ("depth", np.uint8, 1),
    ("path_id", np.uint32, 1),
]
_RAY_FIELDS = [
    ("o", np.float32, 3), ("d", np.float32, 3), ("mint", np.float32, 1), ("maxt", np.float32, 1),
    ("edge_len", np.float32, 1), ("eye_contrib", np.float32, 3), ("xi", np.float32, 1),
    ("px", np.int32, 1), ("py", np.int32, 1), ("edge_id", np.int32, 1), ("off_valid", np.uint8, 4),
    ("off_o", np.float32, 12), ("off_d", np.float32, 12), ("off_len", np.float32, 4),
    ("off_eye", np.float32, 12), ("off_sensor", np.float32, 4),
]
_CT = {np.float32: C.c_float, np.uint8: C.c_uint8, np.uint32: C.c_uint32, np.int32: C.c_int32}


class _SoA:
    FIELDS = []
    CSTRUCT = None

    def __init__(self, n, **arrays):
        self.n = int(n)
        for name, dt, w in self.FIELDS:
            a = arrays.get(name)
            if a is None:
                a = np.zeros(self.n * w, dtype=dt)
            a = np.ascontiguousarray(a, dtype=dt).reshape(-1)
            if a.size != self.n * w:
                raise ValueError(f"{name}: expected {self.n * w} elements, got {a.size}")
            setattr(self, name, a)

    def as_c(self):
        s = self.CSTRUCT()
        for name, dt, _ in self.FIELDS:
            setattr(s, name, getattr(self, name).ctypes.data_as(C.POINTER(_CT[dt])))
        return s

    def take(self, idx):
        """Subset / reorder by element index."""
        idx = np.asarray(idx)
        out = {}
        for name, dt, w in self.FIELDS:
            out[name] = getattr(self, name).reshape(self.n, w)[idx].reshape(-1)
        return type(self)(len(idx), **out)

    def copy(self):
        return self.take(np.arange(self.n))

    def view(self, name):
        for fname, _, w in self.FIELDS:
            if fname == name:
                return getattr(self, name).reshape(self.n, w)
        raise KeyError(name)

    def nbytes(self):
        return sum(getattr(self, name).nbytes for name, _, _ in self.FIELDS)

    def save(self, path):
        np.savez_compressed(path, n=self.n, **{name: getattr(self, name) for name, _, _ in self.FIELDS})

    @classmethod
    def load(cls, path):
        z = np.load(path)
        return cls(int(z["n"]), **{name: z[name] for name, _, _ in cls.FIELDS})


class PhotonSet(_SoA):
    FIELDS = _PHOTON_FIELDS
    CSTRUCT = N.PhotonSoA


class RaySet(_SoA):
    FIELDS = _RAY_FIELDS
    CSTRUCT = N.RaySoA


_VPM_FIELDS = [
    ("ray", np.uint32, 1), ("t", np.float32, 1), ("transmittance", np.float32, 3),
    ("pdf_success", np.float32, 1), ("pdf_sel", np.float32, 1), ("radius", np.float32, 1),
]


_BEAM_FIELDS = [
    ("origin", np.float32, 3), ("end", np.float32, 3), ("flux", np.float32, 3), ("prefix_flux", np.float32, 3),
    ("parent_n", np.float32, 3), ("parent_albedo", np.float32, 3), ("pred_pos", np.float32, 3),
    ("end_n", np.float32, 3), ("parent_pdf", np.float32, 1), ("rr_weight", np.float32, 1),
    ("parent_type", np.uint8, 1), ("end_on_surface", np.uint8, 1), ("depth", np.uint8, 1),
    ("path_id", np.uint32, 1),
]


class BeamSet(_SoA):
    """Photon beams (LTPhotonBeam, gvpm/gvpm_beams.h:18-43) flattened with their parent-vertex data."""
    FIELDS = _BEAM_FIELDS
    CSTRUCT = N.BeamSoA


def synth_beams(n, medium, seed=0xC0FFEE, max_depth=12, rr_depth=1, min_depth=0, power=100.0, threads=8):
    """Seeded light-path random walks -> BeamSet (every medium edge); returns (beams, nbPathBeams)."""
    s = N.load_synth()
    bs = BeamSet(n)
    cs = bs.as_c()
    paths = s.gvpm_synth_beams(seed, n, C.byref(medium), max_depth, rr_depth, min_depth, power, threads,
                               C.byref(cs))
    if paths < 0:
        raise RuntimeError("gvpm_synth_beams failed")
    return bs, int(paths)


_PLANE_FIELDS = [
    ("origin", np.float32, 3), ("w0", np.float32, 3), ("length0", np.float32, 1), ("w1", np.float32, 3),
    ("length1", np.float32, 1), ("flux", np.float32, 3), ("edge_id", np.int32, 1),
]


class PlaneSet(_SoA):
    """Photon planes (LTPhotonPlane, gvpm/gvpm_plane.h:18-46)."""
    FIELDS = _PLANE_FIELDS
    CSTRUCT = N.PlaneSoA


def synth_planes(beams, medium, seed=0xC0FFEE):
    """Beams -> planes through the host mirror of LTPhotonPlane::transformBeam (one sampler, beam order)."""
    s = N.load_synth()
    ps = PlaneSet(beams.n)
    cb, cp = beams.as_c(), ps.as_c()
    got = s.gvpm_synth_planes(seed, C.byref(cb), beams.n, C.byref(medium), C.byref(cp))
    assert got == beams.n
    return ps


class VpmSampleSet(_SoA):
    """Camera distance samples of the G-VPM gather (gvpm.cpp:1141-1175), one per (pixel, sample)."""
    FIELDS = _VPM_FIELDS
    CSTRUCT = N.VpmSampleSoA


def synth_vpm_samples(rays, medium, radius_per_ray, nb_camera_samples=40, stratified=False, seed=0xC0FFEE,
                      epsilon=1e-4):
    """Host-side edge selection + HomogeneousMedium::sampleDistance(EDistanceAlwaysValid) for gather points
    with one medium edge (homogeneous.cpp:293-430)."""
    s = N.load_synth()
    radius_per_ray = np.ascontiguousarray(np.broadcast_to(np.asarray(radius_per_ray, dtype=np.float32), (rays.n,)))
    full = VpmSampleSet(rays.n * nb_camera_samples)
    cs, cr = full.as_c(), rays.as_c()
    n = s.gvpm_synth_vpm_samples(seed, C.byref(cr), rays.n, nb_camera_samples, int(stratified), C.byref(medium),
                                 epsilon, radius_per_ray.ctypes.data_as(N.f32p), C.byref(cs))
    return full.take(np.arange(n))


def make_medium(sigma_t=2.0, albedo=0.8, phase="isotropic", g=0.0, sampling_weight=1.0):
    m = N.Medium()
    ss, sa = np.float32(sigma_t * albedo), np.float32(sigma_t * (1.0 - albedo))
    for i in range(3):
        m.sigma_s[i] = ss
        m.sigma_a[i] = sa
    m.phase_type = N.PHASE_HG if phase == "hg" else N.PHASE_ISOTROPIC
    m.hg_g = g
    m.sampling_weight = sampling_weight
    return m


def make_config(film_w, film_h, max_depth=12, min_depth=0, lighting_mode=N.ALL2MEDIA, use_mis=True,
                use_shift_null=True, path_set=True, power_heuristic=False, kernel_3d=True,
                shadow_maxt_scale=1e-3, epsilon=1e-4, long_beams=False, rng_seed=0, beam_kernel_1d=False, sppm_primal=False):
    """Defaults = the paper presets (scripts/scene/generatorGVPM.py:44-50: useMIS=area, mixed shift,
    maxDepth 12) with pathSet at its plugin default (gvpm_struct.h:328)."""
    c = N.Config()
    c.max_depth, c.min_depth, c.lighting_mode = max_depth, min_depth, lighting_mode
    c.use_mis, c.use_shift_null, c.path_set = int(use_mis), int(use_shift_null), int(path_set)
    c.power_heuristic, c.kernel_3d = int(power_heuristic), int(kernel_3d)
    c.film_w, c.film_h = film_w, film_h
    c.shadow_maxt_scale, c.epsilon = shadow_maxt_scale, epsilon
    c.long_beams, c.rng_seed = int(long_beams), int(rng_seed) & 0xFFFFFFFF
    c.beam_kernel_1d = int(beam_kernel_1d)
    c.sppm_primal = int(sppm_primal)
    return c


# bounding-sphere radius of the medium AABB [0,1]^3 of the synthetic scene (gvpm.cpp:989,
# volume_utils.h:219): radius = bsphereR * globalScaleVolume * POURCENTAGE_BS
SYNTH_BSPHERE_R = float(np.sqrt(np.float32(3.0)) * np.float32(0.5))


def bre_radius(scale_volume, bsphere_r=SYNTH_BSPHERE_R):
    return float(np.float32(bsphere_r) * np.float32(scale_volume) * np.float32(0.01))


def synth_photons(n, medium, seed=0xC0FFEE, max_depth=12, rr_depth=1, min_depth=0, power=100.0, threads=8):
    """Seeded light-path random walks -> PhotonSet; returns (photons, nbPathVolume)."""
    s = N.load_synth()
    ps = PhotonSet(n)
    cs = ps.as_c()
    paths = s.gvpm_synth_photons(seed, n, C.byref(medium), max_depth, rr_depth, min_depth, power, threads,
                                 C.byref(cs))
    if paths < 0:
        raise RuntimeError("gvpm_synth_photons failed")
    return ps, int(paths)


def synth_rays(w, h, seed=0xC0FFEE, block=32, y0=0, y1=None, cam_dist=1.5, cover=0.96, epsilon=1e-4):
    s = N.load_synth()
    y1 = h if y1 is None else y1
    n = w * (y1 - y0)
    rs = RaySet(n)
    cs = rs.as_c()
    got = s.gvpm_synth_rays(seed, w, h, block, y0, y1, cam_dist, cover, epsilon, C.byref(cs))
    assert got == n, (got, n)
    return rs


def synth_occluders():
    s = N.load_synth()
    n = s.gvpm_synth_occluders(None)
    tri = np.zeros(n * 9, dtype=np.float32)
    s.gvpm_synth_occluders(tri.ctypes.data_as(N.f32p))
    return tri


def box_scene_default():
    """The Cornell box of the synthetic workloads as a gvpm_box_scene (rows f-1 / f-2: on-device generators)."""
    sc = N.BoxScene()
    rc = N.load_lib().gvpm_box_scene_default(C.byref(sc))
    assert rc == 0
    return sc


def pinhole_camera(w, h, cam_dist=1.5, cover=0.96):
    """The sensor of synth_rays(): at (0.5, 0.5, -cam_dist) looking down +z; cam_dist < 0: inside the medium at
    z = -cam_dist with tan(fov/2) = cover."""
    cam = N.PinholeCamera()
    cam.pos[0], cam.pos[1], cam.pos[2] = 0.5, 0.5, -cam_dist
    inside = cam_dist < 0
    cam.tan_half_fov_x = np.float32(cover) if inside else np.float32(0.5) * np.float32(cover) / np.float32(cam_dist)
    cam.film_w, cam.film_h, cam.inside_medium = w, h, int(inside)
    return cam


def lookat_camera(w, h, pos, forward=(0.0, 0.0, 1.0), up=(0.0, 1.0, 0.0), tan_half_fov_x=0.32):
    """A pinhole with a look-at frame (gvpm_lookat_camera) for the mesh generators: forward = +z, up = +y is the frame of
    pinhole_camera()."""
    cam = N.LookatCamera()
    for a in range(3):
        cam.pos[a], cam.forward[a], cam.up[a] = float(pos[a]), float(forward[a]), float(up[a])
    cam.tan_half_fov_x = float(np.float32(tan_half_fov_x))
    cam.film_w, cam.film_h = w, h
    return cam


def box_scene_as_mesh(scene):
    """A gvpm_box_scene as mesh-scene arrays: two triangles per wall (the open face z = lo stays open), per rectangle and
    for the light (emissive, wound so that its normal points down, with the ceiling's albedo).  -> dict of the keyword
    arguments of Context.set_trace_mesh."""
    lo = np.array(scene.lo[:], dtype=np.float32)
    hi = np.array(scene.hi[:], dtype=np.float32)
    quads, alb, emit = [], [], []

    def quad(a, b, c, d, albedo, e=0):
        # a b c d in order around the quad: triangles (a, b, c) and (a, c, d) share its winding
        quads.extend([(a, b, c), (a, c, d)])
        alb.extend([albedo, albedo])
        emit.extend([e, e])

    x0, y0, z0 = lo
    x1, y1, z1 = hi
    fa = [tuple(scene.face_albedo[i][:]) for i in range(5)]
    quad((x0, y0, z0), (x0, y1, z0), (x0, y1, z1), (x0, y0, z1), fa[0])   # x = lo
    quad((x1, y0, z0), (x1, y0, z1), (x1, y1, z1), (x1, y1, z0), fa[1])   # x = hi
    quad((x0, y0, z0), (x0, y0, z1), (x1, y0, z1), (x1, y0, z0), fa[2])   # y = lo
    quad((x0, y1, z0), (x1, y1, z0), (x1, y1, z1), (x0, y1, z1), fa[3])   # y = hi
    quad((x0, y0, z1), (x0, y1, z1), (x1, y1, z1), (x1, y0, z1), fa[4])   # z = hi
    for r in range(scene.n_rects):
        R = scene.rect[r]
        quad((R.x0, R.y, R.z0), (R.x1, R.y, R.z0), (R.x1, R.y, R.z1), (R.x0, R.y, R.z1), tuple(R.albedo[:]))
    ly = scene.light_y
    # winding (x0, z0) -> (x1, z0) -> (x1, z1): the normal cross((dx, 0, 0), (dx, 0, dz)) = (0, -dx dz, 0) points down
    quad((scene.light_x0, ly, scene.light_z0), (scene.light_x1, ly, scene.light_z0), (scene.light_x1, ly, scene.light_z1),
         (scene.light_x0, ly, scene.light_z1), fa[3], 1)
    tri = np.array(quads, dtype=np.float32).reshape(-1, 9)
    return dict(tri=tri, albedo=np.array(alb, dtype=np.float32).reshape(-1, 3), emissive=np.array(emit, dtype=np.uint8),
                light_power=float(scene.light_power), lo=lo, hi=hi)
