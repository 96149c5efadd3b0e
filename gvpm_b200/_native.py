"""ctypes declarations for the C ABI in include/gvpm_b200.h and loaders for the in-tree libraries.

The product library (libgvpm_b200.so, built from gvpm_b200/csrc by nvcc for sm_100a) has no CPU
fallback: loading fails loudly when the file is missing, and gvpm_ctx_create fails when there is
no CUDA device.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GVPM_B200_LIB: load another build of the same library (kernel-tuning experiments only)
LIB_PATH = os.environ.get("GVPM_B200_LIB") or os.path.join(_HERE, "libgvpm_b200.so")
SYNTH_LIB_PATH = os.path.join(_HERE, "synth", "libgvpm_synth.so")

GVPM_OUT_FLOATS = 27
GVPM_PEER_BLOB_BYTES = 384
GVPM_DISPATCH_BLOB_BYTES = 512
GVPM_MAX_PEERS = 8
GVPM_SHARED_HANDLE_BYTES = 96
PARENT_EMITTER, PARENT_SURFACE, PARENT_MEDIUM, PARENT_OTHER = 0, 1, 2, 3
PHASE_ISOTROPIC, PHASE_HG = 0, 1
SURF2MEDIA, MEDIA2MEDIA = 1 << 2, 1 << 4
ALL2MEDIA = SURF2MEDIA | MEDIA2MEDIA

f32p = C.POINTER(C.c_float)
u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
u64p = C.POINTER(C.c_uint64)


class Medium(C.Structure):
    _fields_ = [("sigma_s", C.c_float * 3), ("sigma_a", C.c_float * 3), ("phase_type", C.c_int32),
                ("hg_g", C.c_float), ("sampling_weight", C.c_float)]


class Config(C.Structure):
    _fields_ = [("max_depth", C.c_int32), ("min_depth", C.c_int32), ("lighting_mode", C.c_int32),
                ("use_mis", C.c_int32), ("use_shift_null", C.c_int32), ("path_set", C.c_int32),
                ("power_heuristic", C.c_int32), ("kernel_3d", C.c_int32), ("film_w", C.c_int32),
                ("film_h", C.c_int32), ("shadow_maxt_scale", C.c_float), ("epsilon", C.c_float),
                ("long_beams", C.c_int32), ("rng_seed", C.c_uint32), ("beam_kernel_1d", C.c_int32), ("sppm_primal", C.c_int32)]


class PhotonSoA(C.Structure):
    _fields_ = [("pos", f32p), ("flux", f32p), ("parent_pos", f32p), ("pred_pos", f32p),
                ("parent_n", f32p), ("prefix_flux", f32p), ("parent_albedo", f32p),
                ("parent_pdf", f32p), ("edge_pdf", f32p), ("rr_weight", f32p),
                ("parent_type", u8p), ("depth", u8p), ("path_id", u32p)]


class RaySoA(C.Structure):
    _fields_ = [("o", f32p), ("d", f32p), ("mint", f32p), ("maxt", f32p), ("edge_len", f32p),
                ("eye_contrib", f32p), ("xi", f32p), ("px", i32p), ("py", i32p), ("edge_id", i32p),
                ("off_valid", u8p), ("off_o", f32p), ("off_d", f32p), ("off_len", f32p),
                ("off_eye", f32p), ("off_sensor", f32p)]


class BeamSoA(C.Structure):
    _fields_ = [("origin", f32p), ("end", f32p), ("flux", f32p), ("prefix_flux", f32p), ("parent_n", f32p),
                ("parent_albedo", f32p), ("pred_pos", f32p), ("end_n", f32p), ("parent_pdf", f32p),
                ("rr_weight", f32p), ("parent_type", u8p), ("end_on_surface", u8p), ("depth", u8p),
                ("path_id", u32p)]


class PlaneSoA(C.Structure):
    _fields_ = [("origin", f32p), ("w0", f32p), ("length0", f32p), ("w1", f32p), ("length1", f32p),
                ("flux", f32p), ("edge_id", i32p)]


class VpmSampleSoA(C.Structure):
    _fields_ = [("ray", u32p), ("t", f32p), ("transmittance", f32p), ("pdf_success", f32p),
                ("pdf_sel", f32p), ("radius", f32p)]


class BoxRect(C.Structure):
    _fields_ = [("y", C.c_float), ("x0", C.c_float), ("x1", C.c_float), ("z0", C.c_float), ("z1", C.c_float),
                ("albedo", C.c_float * 3)]


class BoxScene(C.Structure):
    _fields_ = [("lo", C.c_float * 3), ("hi", C.c_float * 3), ("face_albedo", (C.c_float * 3) * 5),
                ("n_rects", C.c_int32), ("rect", BoxRect * 4), ("light_y", C.c_float), ("light_x0", C.c_float),
                ("light_x1", C.c_float), ("light_z0", C.c_float), ("light_z1", C.c_float), ("light_power", C.c_float)]


class PinholeCamera(C.Structure):
    _fields_ = [("pos", C.c_float * 3), ("tan_half_fov_x", C.c_float), ("film_w", C.c_int32), ("film_h", C.c_int32),
                ("inside_medium", C.c_int32)]


class MeshScene(C.Structure):
    _fields_ = [("lo", C.c_float * 3), ("hi", C.c_float * 3), ("n_tri", C.c_size_t), ("tri", f32p), ("albedo", f32p),
                ("emissive", u8p), ("light_power", C.c_float)]


class LookatCamera(C.Structure):
    _fields_ = [("pos", C.c_float * 3), ("forward", C.c_float * 3), ("up", C.c_float * 3), ("tan_half_fov_x", C.c_float),
                ("film_w", C.c_int32), ("film_h", C.c_int32)]


class PoissonParams(C.Structure):
    _fields_ = [("alpha", C.c_float), ("irls_iter_max", C.c_int32), ("irls_reg_init", C.c_float),
                ("irls_reg_iter", C.c_float), ("cg_iter_max", C.c_int32), ("cg_iter_check", C.c_int32),
                ("cg_precond", C.c_int32), ("cg_tolerance", C.c_float)]


# gvpm_device.cuh FrustumGrid (gvpm_frustum_grid copies it out as raw bytes)
GVPM_GRID_CLASSES = 16


class FrustumGrid(C.Structure):
    _fields_ = [("C", C.c_float * 3), ("m", C.c_float * 3), ("u", C.c_float * 3), ("v", C.c_float * 3),
                ("gx0", C.c_float), ("gy0", C.c_float), ("csize", C.c_float * GVPM_GRID_CLASSES),
                ("xmin", C.c_float), ("xmax", C.c_float), ("ymin", C.c_float), ("ymax", C.c_float), ("pad_r", C.c_float),
                ("nx", C.c_uint32 * GVPM_GRID_CLASSES), ("ny", C.c_uint32 * GVPM_GRID_CLASSES),
                ("base", C.c_uint32 * GVPM_GRID_CLASSES), ("n_cells", C.c_uint32), ("classes", C.c_int32),
                ("parity_split", C.c_int32)]


# gvpm_beam_technique (volTechnique strings of sppm.cpp:208-209)
BEAM_TECHNIQUES = {"beam1d": 0, "beam3d_naive": 1, "beam3d_egsr": 2, "beam3d": 3}

# every symbol include/gvpm_b200.h declares (tests check the .so exports all of them)
ABI_SYMBOLS = [
    "gvpm_abi_version", "gvpm_ctx_create", "gvpm_ctx_destroy", "gvpm_last_error", "gvpm_sync",
    "gvpm_stream", "gvpm_set_medium", "gvpm_set_config", "gvpm_set_occluders",
    "gvpm_set_occluder_accel", "gvpm_occluder_accel_kind", "gvpm_occluded",
    "gvpm_upload_photons", "gvpm_photon_staging", "gvpm_build_points", "gvpm_build_points_for_rays", "gvpm_accel_kind", "gvpm_frustum_grid", "gvpm_set_view_direction",
    "gvpm_photon_staging_select", "gvpm_photon_staging_layout", "gvpm_upload_photons_slice",
    "gvpm_peer_export", "gvpm_peer_connect", "gvpm_peer_push_photon_slice", "gvpm_peer_wait_photons", "gvpm_peer_push_mode",
    "gvpm_dispatch_export", "gvpm_dispatch_connect", "gvpm_dispatch_photons", "gvpm_build_dispatched", "gvpm_dispatch_release",
    "gvpm_dispatch_status", "gvpm_dispatch_join", "gvpm_shared_buffer_create", "gvpm_shared_buffer_open", "gvpm_collect_signal",
    "gvpm_collect_wait",
    "gvpm_upload_rays", "gvpm_ray_staging", "gvpm_commit_rays", "gvpm_gather_bre", "gvpm_gather_sppm_bre",
    "gvpm_gather_bre_device", "gvpm_gather_bre_into", "gvpm_gather_bre_host", "gvpm_dump_neighbours_bre",
    "gvpm_compute_gradient", "gvpm_compute_gradient_reuse_primal", "gvpm_poisson_preset", "gvpm_poisson_solve", "gvpm_reconstruct", "gvpm_last_poisson_ms", "gvpm_last_timings", "gvpm_last_gather_detail", "gvpm_launch_count",
    "gvpm_upload_vpm_samples", "gvpm_gather_vpm", "gvpm_gather_vpm_device", "gvpm_dump_neighbours_vpm",
    "gvpm_generate_vpm_samples",
    "gvpm_upload_beams", "gvpm_build_beams", "gvpm_gather_beams", "gvpm_gather_beams_device", "gvpm_dump_neighbours_beams", "gvpm_beam_subbeam_count",
    "gvpm_gather_sppm_beams", "gvpm_dump_neighbours_sppm_beams",
    "gvpm_box_scene_default", "gvpm_generate_rays", "gvpm_trace_photons", "gvpm_trace_photons_direct", "gvpm_trace_beams", "gvpm_planes_from_beams",
    "gvpm_set_trace_mesh", "gvpm_trace_photons_mesh", "gvpm_trace_photons_direct_mesh", "gvpm_trace_beams_mesh",
    "gvpm_generate_rays_mesh", "gvpm_read_device", "gvpm_measure_read_bandwidth", "gvpm_staging_peek",
    "gvpm_upload_planes", "gvpm_build_planes", "gvpm_gather_planes", "gvpm_gather_planes_device", "gvpm_dump_neighbours_planes",
    "gvpm_accum_reset", "gvpm_accum_add", "gvpm_accum_fold", "gvpm_accum_read", "gvpm_accum_device",
    "gvpm_compute_gradient_accum", "gvpm_reconstruct_accum",
]

_lib = None
_synth = None


def load_lib():
    """Load the product library.  Raises if it was not built: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  gvpm_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.gvpm_abi_version.restype = C.c_int
    lib.gvpm_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.gvpm_ctx_destroy.argtypes = [vp]
    lib.gvpm_last_error.argtypes = [vp]
    lib.gvpm_last_error.restype = C.c_char_p
    lib.gvpm_sync.argtypes = [vp]
    lib.gvpm_stream.argtypes = [vp]
    lib.gvpm_stream.restype = vp
    lib.gvpm_set_medium.argtypes = [vp, C.POINTER(Medium)]
    lib.gvpm_set_config.argtypes = [vp, C.POINTER(Config)]
    lib.gvpm_set_occluders.argtypes = [vp, f32p, C.c_size_t]
    lib.gvpm_set_occluder_accel.argtypes = [vp, C.c_int]
    lib.gvpm_occluder_accel_kind.argtypes = [vp]
    lib.gvpm_occluded.argtypes = [vp, f32p, f32p, f32p, f32p, C.c_size_t, C.POINTER(C.c_uint8)]
    lib.gvpm_upload_photons.argtypes = [vp, C.POINTER(PhotonSoA), C.c_size_t]
    lib.gvpm_photon_staging.argtypes = [vp, C.c_size_t, C.POINTER(vp), C.POINTER(C.c_size_t)]
    lib.gvpm_build_points.argtypes = [vp, C.c_float]
    lib.gvpm_build_points_for_rays.argtypes = [vp, C.c_float, u32p]
    lib.gvpm_accel_kind.argtypes = [vp]
    lib.gvpm_frustum_grid.argtypes = [vp, vp, C.c_size_t, u32p, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.gvpm_box_scene_default.argtypes = [C.POINTER(BoxScene)]
    lib.gvpm_generate_rays.argtypes = [vp, C.POINTER(BoxScene), C.POINTER(PinholeCamera), C.c_uint64, C.c_int, C.c_int,
                                       C.c_int, C.c_float]
    lib.gvpm_trace_photons.argtypes = [vp, C.POINTER(BoxScene), C.c_size_t, C.c_uint64, C.c_int, C.c_int, C.c_int, u64p]
    lib.gvpm_trace_photons_direct.argtypes = [vp, C.POINTER(BoxScene), C.c_size_t, C.c_uint64, C.c_int, C.c_int, C.c_int, u64p]
    lib.gvpm_trace_beams.argtypes = [vp, C.POINTER(BoxScene), C.c_size_t, C.c_uint64, C.c_int, C.c_int, C.c_int, u64p]
    lib.gvpm_planes_from_beams.argtypes = [vp, C.c_uint64]
    lib.gvpm_set_trace_mesh.argtypes = [vp, C.POINTER(MeshScene)]
    for name in ("gvpm_trace_photons_mesh", "gvpm_trace_photons_direct_mesh", "gvpm_trace_beams_mesh"):
        getattr(lib, name).argtypes = [vp, C.c_size_t, C.c_uint64, C.c_int, C.c_int, C.c_int, u64p]
    lib.gvpm_generate_rays_mesh.argtypes = [vp, C.POINTER(LookatCamera), C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_float]
    lib.gvpm_read_device.argtypes = [vp, vp, vp, C.c_size_t]
    lib.gvpm_measure_read_bandwidth.argtypes = [vp, C.c_size_t, C.c_int, C.POINTER(C.c_double)]
    lib.gvpm_staging_peek.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_size_t)]
    lib.gvpm_photon_staging_select.argtypes = [vp, C.c_int]
    lib.gvpm_photon_staging_layout.argtypes = [C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    lib.gvpm_upload_photons_slice.argtypes = [vp, C.POINTER(PhotonSoA), C.c_size_t, C.c_size_t, C.c_size_t, vp]
    lib.gvpm_peer_export.argtypes = [vp, vp]
    lib.gvpm_peer_connect.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.gvpm_peer_push_photon_slice.argtypes = [vp, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, vp]
    lib.gvpm_peer_wait_photons.argtypes = [vp, C.c_int]
    lib.gvpm_peer_push_mode.argtypes = [vp, C.c_int]
    lib.gvpm_set_view_direction.argtypes = [vp, f32p]
    lib.gvpm_dispatch_export.argtypes = [vp, C.c_int, C.c_size_t, vp]
    lib.gvpm_dispatch_connect.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.gvpm_dispatch_photons.argtypes = [vp, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_float, vp]
    lib.gvpm_build_dispatched.argtypes = [vp, C.c_int, C.c_float, u32p]
    lib.gvpm_dispatch_release.argtypes = [vp, C.c_int]
    lib.gvpm_dispatch_status.argtypes = [vp, u32p, C.c_int]
    lib.gvpm_dispatch_join.argtypes = [vp]
    lib.gvpm_shared_buffer_create.argtypes = [vp, C.c_size_t, C.POINTER(vp), vp]
    lib.gvpm_shared_buffer_open.argtypes = [vp, vp, C.POINTER(vp)]
    lib.gvpm_collect_signal.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.gvpm_collect_wait.argtypes = [vp, C.c_int]
    lib.gvpm_upload_rays.argtypes = [vp, C.POINTER(RaySoA), C.c_size_t]
    lib.gvpm_ray_staging.argtypes = [vp, C.c_size_t, C.POINTER(vp), C.POINTER(C.c_size_t)]
    lib.gvpm_commit_rays.argtypes = [vp]
    lib.gvpm_gather_bre.argtypes = [vp, f32p, u32p]
    lib.gvpm_gather_sppm_bre.argtypes = [vp, f32p, u32p]
    lib.gvpm_gather_bre_device.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    lib.gvpm_gather_bre_into.argtypes = [vp, vp, vp]
    lib.gvpm_gather_bre_host.argtypes = [vp, C.POINTER(RaySoA), C.c_size_t, f32p]
    lib.gvpm_dump_neighbours_bre.argtypes = [vp, u64p, u32p, C.c_size_t]
    lib.gvpm_compute_gradient.argtypes = [vp, f32p, C.c_int, C.c_int, C.c_int, f32p, f32p, f32p]
    lib.gvpm_compute_gradient_reuse_primal.argtypes = [vp, f32p, C.c_int, C.c_int, C.c_int, C.c_float, f32p, f32p, f32p]
    lib.gvpm_poisson_preset.argtypes = [C.c_char_p, C.POINTER(PoissonParams)]
    lib.gvpm_poisson_solve.argtypes = [vp, C.c_int, C.c_int, f32p, f32p, f32p, f32p, C.POINTER(PoissonParams), f32p]
    lib.gvpm_reconstruct.argtypes = [vp, f32p, C.c_int, C.c_int, C.c_int, f32p, C.POINTER(PoissonParams), f32p, f32p, f32p, f32p]
    lib.gvpm_accum_reset.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.gvpm_accum_add.argtypes = [vp]
    lib.gvpm_accum_fold.argtypes = [vp, C.c_int, C.c_uint64]
    lib.gvpm_accum_read.argtypes = [vp, C.c_int, f32p, u8p, u64p]
    lib.gvpm_accum_device.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    lib.gvpm_compute_gradient_accum.argtypes = [vp, C.c_int, C.c_int, C.c_float, f32p, f32p, f32p]
    lib.gvpm_reconstruct_accum.argtypes = [vp, C.c_int, f32p, C.POINTER(PoissonParams), f32p, f32p, f32p, f32p]
    lib.gvpm_last_poisson_ms.argtypes = [vp]
    lib.gvpm_last_poisson_ms.restype = C.c_float
    lib.gvpm_last_timings.argtypes = [vp, f32p, f32p]
    lib.gvpm_last_gather_detail.argtypes = [vp, f32p, f32p, u64p]
    lib.gvpm_upload_beams.argtypes = [vp, C.POINTER(BeamSoA), C.c_size_t]
    lib.gvpm_build_beams.argtypes = [vp, C.c_float]
    lib.gvpm_gather_beams.argtypes = [vp, f32p, u32p]
    lib.gvpm_beam_subbeam_count.argtypes = [vp]
    lib.gvpm_beam_subbeam_count.restype = C.c_uint64
    lib.gvpm_gather_beams_device.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    lib.gvpm_gather_planes_device.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    lib.gvpm_gather_vpm_device.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(vp)]
    lib.gvpm_dump_neighbours_beams.argtypes = [vp, u64p, u32p, C.c_size_t]
    lib.gvpm_gather_sppm_beams.argtypes = [vp, C.c_int, f32p, u32p]
    lib.gvpm_dump_neighbours_sppm_beams.argtypes = [vp, C.c_int, u64p, u32p, C.c_size_t]
    lib.gvpm_upload_planes.argtypes = [vp, C.POINTER(PlaneSoA), C.c_size_t]
    lib.gvpm_build_planes.argtypes = [vp]
    lib.gvpm_gather_planes.argtypes = [vp, f32p, u32p]
    lib.gvpm_dump_neighbours_planes.argtypes = [vp, u64p, u32p, C.c_size_t]
    lib.gvpm_upload_vpm_samples.argtypes = [vp, C.POINTER(VpmSampleSoA), C.c_size_t]
    lib.gvpm_gather_vpm.argtypes = [vp, C.c_int, f32p, u32p, u32p]
    lib.gvpm_dump_neighbours_vpm.argtypes = [vp, C.c_int, u64p, u32p, C.c_size_t]
    lib.gvpm_generate_vpm_samples.argtypes = [vp, C.c_int, C.c_int, C.c_uint64, C.c_float, C.c_float, vp,
                                              C.POINTER(C.c_size_t)]
    lib.gvpm_launch_count.argtypes = [vp]
    lib.gvpm_launch_count.restype = C.c_uint64
    for name in ABI_SYMBOLS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int and name not in ("gvpm_abi_version",):
            fn.restype = C.c_int
    _lib = lib
    return lib


def load_synth():
    global _synth
    if _synth is not None:
        return _synth
    if not os.path.exists(SYNTH_LIB_PATH):
        raise RuntimeError(f"{SYNTH_LIB_PATH} is missing: run __graft_entry__.build()")
    s = C.CDLL(SYNTH_LIB_PATH)
    s.gvpm_synth_photons.argtypes = [C.c_uint64, C.c_size_t, C.POINTER(Medium), C.c_int, C.c_int, C.c_int,
                                     C.c_float, C.c_int, C.POINTER(PhotonSoA)]
    s.gvpm_synth_photons.restype = C.c_longlong
    s.gvpm_synth_occluders.argtypes = [f32p]
    s.gvpm_synth_occluders.restype = C.c_size_t
    s.gvpm_synth_rays.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                  C.c_float, C.c_float, C.POINTER(RaySoA)]
    s.gvpm_synth_rays.restype = C.c_size_t
    s.gvpm_synth_vpm_samples.argtypes = [C.c_uint64, C.POINTER(RaySoA), C.c_size_t, C.c_int, C.c_int,
                                         C.POINTER(Medium), C.c_float, f32p, C.POINTER(VpmSampleSoA)]
    s.gvpm_synth_vpm_samples.restype = C.c_size_t
    s.gvpm_synth_beams.argtypes = [C.c_uint64, C.c_size_t, C.POINTER(Medium), C.c_int, C.c_int, C.c_int,
                                   C.c_float, C.c_int, C.POINTER(BeamSoA)]
    s.gvpm_synth_beams.restype = C.c_longlong
    s.gvpm_synth_planes.argtypes = [C.c_uint64, C.POINTER(BeamSoA), C.c_size_t, C.POINTER(Medium),
                                    C.POINTER(PlaneSoA)]
    s.gvpm_synth_planes.restype = C.c_size_t
    _synth = s
    return s
