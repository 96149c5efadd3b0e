"""Thin Python handle on the C ABI (include/gvpm_b200.h).  Every method is one C call; errors raise.

This is the call a host integrator makes per iteration (INTEGRATION.md):
    ctx.set_medium / set_config / set_occluders           once per scene
    ctx.upload_photons(photons); ctx.build_points(r)      replaces gvpm.cpp:453 + gvpm_accel.cpp:10-55
    ctx.upload_rays(rays)                                 the gather points of the iteration
    out, counts = ctx.gather_bre()                        replaces gvpm.cpp:999-1052
"""
import ctypes as C

import numpy as np

from . import _native as N


class GvpmError(RuntimeError):
    pass


class Context:
    def __init__(self, device=0):
        self.lib = N.load_lib()
        h = C.c_void_p()
        rc = self.lib.gvpm_ctx_create(device, C.byref(h))
        if rc != 0:
            raise GvpmError(f"gvpm_ctx_create({device}) failed ({rc}): "
                            f"{self.lib.gvpm_last_error(None).decode()}")
        self.h = h
        self.n_rays = 0
        self.n_photons = 0
        self.n_samples = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.gvpm_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc != 0:
            raise GvpmError(f"{what} failed ({rc}): {self.lib.gvpm_last_error(self.h).decode()}")

    # ---- scene constants
    def set_medium(self, medium):
        self._ck(self.lib.gvpm_set_medium(self.h, C.byref(medium)), "gvpm_set_medium")

    def set_config(self, config):
        self._ck(self.lib.gvpm_set_config(self.h, C.byref(config)), "gvpm_set_config")

    def set_occluders(self, tri):
        tri = np.ascontiguousarray(tri, dtype=np.float32).reshape(-1)
        self._ck(self.lib.gvpm_set_occluders(self.h, tri.ctypes.data_as(N.f32p), tri.size // 9),
                 "gvpm_set_occluders")

    # ---- photons
    def upload_photons(self, photons):
        cs = photons.as_c()
        self._ck(self.lib.gvpm_upload_photons(self.h, C.byref(cs), photons.n), "gvpm_upload_photons")
        self.n_photons = photons.n

    def photon_staging(self, n):
        dev, nbytes = C.c_void_p(), C.c_size_t()
        self._ck(self.lib.gvpm_photon_staging(self.h, n, C.byref(dev), C.byref(nbytes)), "gvpm_photon_staging")
        self.n_photons = n
        return dev.value, nbytes.value

    def photon_staging_select(self, which):
        self._ck(self.lib.gvpm_photon_staging_select(self.h, int(which)), "gvpm_photon_staging_select")

    def photon_staging_layout(self, n):
        """-> (offsets[13], elem_bytes[13]) of the field arrays inside the staging buffer."""
        off = (C.c_size_t * 13)()
        elt = (C.c_size_t * 13)()
        self._ck(self.lib.gvpm_photon_staging_layout(n, off, elt), "gvpm_photon_staging_layout")
        return list(off), list(elt)

    def upload_photons_slice(self, photons_slice, n_total, begin, stream=None):
        """photons_slice: a PhotonSet holding photons [begin, begin + photons_slice.n) of a set of n_total."""
        cs = photons_slice.as_c()
        self._ck(self.lib.gvpm_upload_photons_slice(self.h, C.byref(cs), n_total, begin, photons_slice.n, stream),
                 "gvpm_upload_photons_slice")

    def peer_export(self):
        """-> bytes: this context's IPC blob (staging buffers + events) for gvpm_peer_connect on the other ranks."""
        buf = (C.c_ubyte * N.GVPM_PEER_BLOB_BYTES)()
        self._ck(self.lib.gvpm_peer_export(self.h, buf), "gvpm_peer_export")
        return bytes(buf)

    def peer_connect(self, blobs, self_index):
        raw = b"".join(blobs)
        buf = (C.c_ubyte * len(raw)).from_buffer_copy(raw)
        self._ck(self.lib.gvpm_peer_connect(self.h, buf, len(blobs), self_index), "gvpm_peer_connect")

    def peer_push_photon_slice(self, which, n_total, begin, count, after_stream=None):
        self._ck(self.lib.gvpm_peer_push_photon_slice(self.h, which, n_total, begin, count, after_stream),
                 "gvpm_peer_push_photon_slice")

    def peer_wait_photons(self, which):
        self._ck(self.lib.gvpm_peer_wait_photons(self.h, which), "gvpm_peer_wait_photons")

    def peer_push_mode(self, sm_ctas):
        """sm_ctas > 0: push kernel of that many CTAs (stores through the peer mappings); 0: copy engines."""
        self._ck(self.lib.gvpm_peer_push_mode(self.h, int(sm_ctas)), "gvpm_peer_push_mode")

    # ---- photon dispatch between ranks (gvpm_dispatch_*) ----
    def dispatch_export(self, n_peers, region_cap):
        """-> bytes: this context's dispatch blob (inboxes, control block, ray fit); needs this rank's rays uploaded."""
        buf = (C.c_ubyte * N.GVPM_DISPATCH_BLOB_BYTES)()
        self._ck(self.lib.gvpm_dispatch_export(self.h, int(n_peers), int(region_cap), buf), "gvpm_dispatch_export")
        return bytes(buf)

    def dispatch_connect(self, blobs, self_index):
        raw = b"".join(blobs)
        buf = (C.c_ubyte * len(raw)).from_buffer_copy(raw)
        self._ck(self.lib.gvpm_dispatch_connect(self.h, buf, len(blobs), self_index), "gvpm_dispatch_connect")

    def dispatch_photons(self, which, n_total, begin, count, radius, after_stream=None):
        self._ck(self.lib.gvpm_dispatch_photons(self.h, which, n_total, begin, count, C.c_float(radius), after_stream),
                 "gvpm_dispatch_photons")

    def build_dispatched(self, which, radius, want_kept=False):
        kept = C.c_uint32(0)
        self._ck(self.lib.gvpm_build_dispatched(self.h, which, C.c_float(radius), C.byref(kept) if want_kept else None),
                 "gvpm_build_dispatched")
        return int(kept.value) if want_kept else None

    def dispatch_release(self, which):
        self._ck(self.lib.gvpm_dispatch_release(self.h, which), "gvpm_dispatch_release")

    def measure_read_bandwidth(self, nbytes, reps):
        """GB/s of `reps` passes of 128-bit loads over an nbytes device buffer (L2 peak when it fits in L2)"""
        v = C.c_double(0.0)
        self._ck(self.lib.gvpm_measure_read_bandwidth(self.h, int(nbytes), int(reps), C.byref(v)), "gvpm_measure_read_bandwidth")
        return float(v.value)

    def shared_buffer_create(self, nbytes):
        """-> (device pointer, handle bytes): a device buffer other ranks can open and write (CUDA IPC)"""
        dev = C.c_void_p()
        h = (C.c_ubyte * N.GVPM_SHARED_HANDLE_BYTES)()
        self._ck(self.lib.gvpm_shared_buffer_create(self.h, int(nbytes), C.byref(dev), h), "gvpm_shared_buffer_create")
        return dev.value, bytes(h)

    def shared_buffer_open(self, handle):
        dev = C.c_void_p()
        h = (C.c_ubyte * N.GVPM_SHARED_HANDLE_BYTES).from_buffer_copy(handle)
        self._ck(self.lib.gvpm_shared_buffer_open(self.h, h, C.byref(dev)), "gvpm_shared_buffer_open")
        return dev.value

    def collect_signal(self, which, root=0, stream=None):
        self._ck(self.lib.gvpm_collect_signal(self.h, which, root, stream), "gvpm_collect_signal")

    def collect_wait(self, which):
        self._ck(self.lib.gvpm_collect_wait(self.h, which), "gvpm_collect_wait")

    def dispatch_join(self):
        self._ck(self.lib.gvpm_dispatch_join(self.h), "gvpm_dispatch_join")

    def dispatch_status(self, which):
        """synchronises; -> records received per sender for inbox `which` (raises on a protocol failure)"""
        counts = (C.c_uint32 * N.GVPM_MAX_PEERS)()
        self._ck(self.lib.gvpm_dispatch_status(self.h, counts, which), "gvpm_dispatch_status")
        return [int(c) for c in counts]

    def build_points(self, radius):
        self._ck(self.lib.gvpm_build_points(self.h, C.c_float(radius)), "gvpm_build_points")

    def build_points_for_rays(self, radius, want_kept=True):
        """Acceleration structure over the photons the uploaded rays can reach only (perspective grid when the rays
        are concurrent, pruned box hierarchy otherwise); -> number of photons kept (want_kept=False: no read-back)."""
        kept = C.c_uint32(0)
        self._ck(self.lib.gvpm_build_points_for_rays(self.h, C.c_float(radius), C.byref(kept) if want_kept else None),
                 "gvpm_build_points_for_rays")
        return int(kept.value) if want_kept else None

    def set_view_direction(self, direction):
        """axis of the perspective grid's projection plane (None: the mean ray direction)"""
        if direction is None:
            self._ck(self.lib.gvpm_set_view_direction(self.h, None), "gvpm_set_view_direction")
            return
        d = (C.c_float * 3)(*[float(v) for v in direction])
        self._ck(self.lib.gvpm_set_view_direction(self.h, d), "gvpm_set_view_direction")

    def accel_kind(self):
        """'bvh' or 'frustum': what the last point build produced"""
        return {0: "bvh", 1: "frustum"}[int(self.lib.gvpm_accel_kind(self.h))]

    # ---- on-device generators (rows f-1, f-2)
    def generate_rays(self, scene, camera, seed, block=32, y0=0, y1=None, epsilon=1e-4):
        """camera-ray medium segments + offsets of a pinhole sensor, generated and committed on the device"""
        y1 = camera.film_h if y1 is None else y1
        self._ck(self.lib.gvpm_generate_rays(self.h, C.byref(scene), C.byref(camera), C.c_uint64(seed), block, y0, y1,
                                             C.c_float(epsilon)), "gvpm_generate_rays")
        self.n_rays = camera.film_w * (y1 - y0)
        return self.n_rays

    def trace_photons(self, scene, n, seed, max_depth=12, rr_depth=1, min_depth=0, direct=False):
        """the iteration's volume photons traced on the device into the selected staging buffer (direct: straight into
        the gather's records); -> light paths traced"""
        paths = C.c_uint64(0)
        fn = self.lib.gvpm_trace_photons_direct if direct else self.lib.gvpm_trace_photons
        self._ck(fn(self.h, C.byref(scene), n, C.c_uint64(seed), max_depth, rr_depth, min_depth, C.byref(paths)),
                 "gvpm_trace_photons")
        self.n_photons = n
        return int(paths.value)

    def trace_beams(self, scene, n, seed, max_depth=12, rr_depth=1, min_depth=0):
        """the iteration's photon beams traced on the device, committed as gvpm_upload_beams commits them (call
        build_beams next); -> light paths traced (nbPathBeams)"""
        paths = C.c_uint64(0)
        self._ck(self.lib.gvpm_trace_beams(self.h, C.byref(scene), n, C.c_uint64(seed), max_depth, rr_depth, min_depth,
                                           C.byref(paths)), "gvpm_trace_beams")
        return int(paths.value)

    def planes_from_beams(self, seed):
        """one photon plane per beam of the current beam set, made on the device (call build_planes next)"""
        self._ck(self.lib.gvpm_planes_from_beams(self.h, C.c_uint64(seed)), "gvpm_planes_from_beams")

    def photon_staging_peek(self, n=None):
        dev, cnt = C.c_void_p(), C.c_size_t()
        self._ck(self.lib.gvpm_staging_peek(self.h, 0, C.byref(dev), C.byref(cnt)), "gvpm_staging_peek")
        return dev.value, cnt.value

    def ray_staging_peek(self):
        dev, cnt = C.c_void_p(), C.c_size_t()
        self._ck(self.lib.gvpm_staging_peek(self.h, 1, C.byref(dev), C.byref(cnt)), "gvpm_staging_peek")
        return dev.value, cnt.value

    def download_photons(self, n):
        """parity aid: the staged photon set as a PhotonSet"""
        from . import records as R
        ptr, _ = self.photon_staging_peek(n)
        off, elt = self.photon_staging_layout(n)
        ps = R.PhotonSet(n)
        for (name, dt, wd), o, e in zip(R._PHOTON_FIELDS, off, elt):
            a = getattr(ps, name)
            self._ck(self.lib.gvpm_read_device(self.h, C.c_void_p(ptr + o), a.ctypes.data_as(C.c_void_p), a.nbytes),
                     "gvpm_read_device")
        return ps

    def download_rays(self):
        """parity aid: the staged (un-packed) ray arrays as a RaySet"""
        from . import records as R
        n = self.n_rays
        ptr, _ = self.ray_staging_peek()
        rs = R.RaySet(n)
        o = 0
        for name, _, _ in R._RAY_FIELDS:   # the field arrays back to back, each starting on a 256-byte boundary
            a = getattr(rs, name)
            self._ck(self.lib.gvpm_read_device(self.h, C.c_void_p(ptr + o), a.ctypes.data_as(C.c_void_p), a.nbytes),
                     "gvpm_read_device")
            o += (a.nbytes + 255) & ~255
        return rs

    def _download_staged(self, which, cls, fields):
        """the staging buffer `which` of gvpm_staging_peek as a `cls` set (arrays back to back, 256-byte aligned)"""
        dev, cnt = C.c_void_p(), C.c_size_t()
        self._ck(self.lib.gvpm_staging_peek(self.h, which, C.byref(dev), C.byref(cnt)), "gvpm_staging_peek")
        out = cls(cnt.value)
        o = 0
        for name, _, _ in fields:
            a = getattr(out, name)
            if a.nbytes:
                self._ck(self.lib.gvpm_read_device(self.h, C.c_void_p(dev.value + o), a.ctypes.data_as(C.c_void_p),
                                                   a.nbytes), "gvpm_read_device")
            o += (a.nbytes + 255) & ~255
        return out

    def download_beams(self):
        """parity aid: the current beam set (uploaded or traced) as a BeamSet"""
        from . import records as R
        return self._download_staged(2, R.BeamSet, R._BEAM_FIELDS)

    def download_planes(self):
        """parity aid: the current plane set (uploaded or made from beams) as a PlaneSet"""
        from . import records as R
        return self._download_staged(3, R.PlaneSet, R._PLANE_FIELDS)

    # ---- rays
    def upload_rays(self, rays):
        cs = rays.as_c()
        self._ck(self.lib.gvpm_upload_rays(self.h, C.byref(cs), rays.n), "gvpm_upload_rays")
        self.n_rays = rays.n

    def ray_staging(self, n):
        dev, nbytes = C.c_void_p(), C.c_size_t()
        self._ck(self.lib.gvpm_ray_staging(self.h, n, C.byref(dev), C.byref(nbytes)), "gvpm_ray_staging")
        self.n_rays = n
        return dev.value, nbytes.value

    def commit_rays(self):
        self._ck(self.lib.gvpm_commit_rays(self.h), "gvpm_commit_rays")

    # ---- gathers
    def gather_bre(self, out=None, counts=True):
        """-> (out [n_rays,27] float32, counts [n_rays,2] uint32 or None), on the host."""
        n = self.n_rays
        if out is None:
            out = np.empty(n * N.GVPM_OUT_FLOATS, dtype=np.float32)
        cnt = np.empty(n * 2, dtype=np.uint32) if counts else None
        self._ck(self.lib.gvpm_gather_bre(self.h, out.ctypes.data_as(N.f32p),
                                          cnt.ctypes.data_as(N.u32p) if counts else None), "gvpm_gather_bre")
        return out.reshape(n, N.GVPM_OUT_FLOATS), (cnt.reshape(n, 2) if counts else None)

    def gather_sppm_bre(self, counts=True):
        """sppm primal BRE (needs config.sppm_primal): -> (out [n_rays,3] float32, counts [n_rays,2] or None)."""
        n = self.n_rays
        out = np.empty(n * 3, dtype=np.float32)
        cnt = np.empty(n * 2, dtype=np.uint32) if counts else None
        self._ck(self.lib.gvpm_gather_sppm_bre(self.h, out.ctypes.data_as(N.f32p),
                                               cnt.ctypes.data_as(N.u32p) if counts else None), "gvpm_gather_sppm_bre")
        return out.reshape(n, 3), (cnt.reshape(n, 2) if counts else None)

    def gather_bre_device(self):
        """Launch only; returns device pointers (out, counts) owned by the context."""
        o, c = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.gvpm_gather_bre_device(self.h, C.byref(o), C.byref(c)), "gvpm_gather_bre_device")
        return o.value, c.value

    def gather_bre_into(self, out_dev_ptr, counts_dev_ptr=None):
        self._ck(self.lib.gvpm_gather_bre_into(self.h, C.c_void_p(out_dev_ptr),
                                               C.c_void_p(counts_dev_ptr) if counts_dev_ptr else None),
                 "gvpm_gather_bre_into")

    def gather_bre_host(self, rays, out=None):
        """upload_rays + gather_bre + download, pipelined (rays / out should be pinned host memory)."""
        cs = rays.as_c()
        self.n_rays = rays.n
        if out is None:
            out = np.empty(rays.n * N.GVPM_OUT_FLOATS, dtype=np.float32)
        self._ck(self.lib.gvpm_gather_bre_host(self.h, C.byref(cs), rays.n, out.ctypes.data_as(N.f32p)),
                 "gvpm_gather_bre_host")
        return out.reshape(rays.n, N.GVPM_OUT_FLOATS)

    def _dump_neighbours(self, name, rows, *args):
        """gvpm_dump_neighbours_<name>: size query, then fill -> (offsets [rows+1] uint64, idx uint32 with bit 31 =
        contributes), every row's segment in ascending index order."""
        fn = getattr(self.lib, "gvpm_dump_neighbours_" + name)
        offsets = np.zeros(rows + 1, dtype=np.uint64)
        rc = fn(self.h, *args, offsets.ctypes.data_as(N.u64p), None, 0)
        total = int(offsets[rows])
        if rc != 0 and total == 0:
            self._ck(rc, "gvpm_dump_neighbours_" + name)
        idx = np.zeros(max(total, 1), dtype=np.uint32)
        if total:
            self._ck(fn(self.h, *args, offsets.ctypes.data_as(N.u64p), idx.ctypes.data_as(N.u32p), total),
                     "gvpm_dump_neighbours_" + name)
        return offsets, idx[:total]

    def dump_neighbours_bre(self):
        """-> (offsets [n_rays+1] uint64, idx uint32 with bit 31 = contributes), per-ray sorted."""
        return self._dump_neighbours("bre", self.n_rays)

    # ---- G-Beams 3D
    def upload_beams(self, beams):
        cs = beams.as_c()
        self._ck(self.lib.gvpm_upload_beams(self.h, C.byref(cs), beams.n), "gvpm_upload_beams")

    def build_beams(self, radius):
        self._ck(self.lib.gvpm_build_beams(self.h, C.c_float(radius)), "gvpm_build_beams")

    def n_subbeams(self):
        """sub-beams the uploaded beam set is cut into (SubBeamBVH, beams_accel.h:98-124)"""
        return int(self.lib.gvpm_beam_subbeam_count(self.h))

    def gather_beams_device(self, counts=False):
        """asynchronous, results stay on the device: -> (out pointer, counts pointer or None)"""
        o, c = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.gvpm_gather_beams_device(self.h, C.byref(o), C.byref(c) if counts else None),
                 "gvpm_gather_beams_device")
        return o.value, (c.value if counts else None)

    def gather_beams(self, counts=True, out=None):
        n = self.n_rays
        out = np.empty(n * N.GVPM_OUT_FLOATS, dtype=np.float32) if out is None else out.reshape(-1)
        cnt = np.empty(n * 2, dtype=np.uint32) if counts else None
        self._ck(self.lib.gvpm_gather_beams(self.h, out.ctypes.data_as(N.f32p),
                                            cnt.ctypes.data_as(N.u32p) if counts else None), "gvpm_gather_beams")
        return out.reshape(n, N.GVPM_OUT_FLOATS), (cnt.reshape(n, 2) if counts else None)

    def dump_neighbours_beams(self):
        return self._dump_neighbours("beams", self.n_rays)

    # ---- sppm primal photon beams
    def gather_sppm_beams(self, technique, counts=True):
        """sppm primal beam gather (volTechnique beam1d | beam3d_naive | beam3d_egsr | beam3d):
        -> (out [n_rays,3] float32, counts [n_rays,2] or None)."""
        tech = N.BEAM_TECHNIQUES[technique] if isinstance(technique, str) else int(technique)
        n = self.n_rays
        out = np.empty(n * 3, dtype=np.float32)
        cnt = np.empty(n * 2, dtype=np.uint32) if counts else None
        self._ck(self.lib.gvpm_gather_sppm_beams(self.h, tech, out.ctypes.data_as(N.f32p),
                                                 cnt.ctypes.data_as(N.u32p) if counts else None),
                 "gvpm_gather_sppm_beams")
        return out.reshape(n, 3), (cnt.reshape(n, 2) if counts else None)

    def dump_neighbours_sppm_beams(self, technique):
        tech = N.BEAM_TECHNIQUES[technique] if isinstance(technique, str) else int(technique)
        return self._dump_neighbours("sppm_beams", self.n_rays, tech)

    # ---- G-Planes 0D
    def upload_planes(self, planes):
        cs = planes.as_c()
        self._ck(self.lib.gvpm_upload_planes(self.h, C.byref(cs), planes.n), "gvpm_upload_planes")

    def build_planes(self):
        self._ck(self.lib.gvpm_build_planes(self.h), "gvpm_build_planes")

    def gather_planes_device(self, counts=False):
        o, c = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.gvpm_gather_planes_device(self.h, C.byref(o), C.byref(c) if counts else None),
                 "gvpm_gather_planes_device")
        return o.value, (c.value if counts else None)

    def gather_planes(self, counts=True, out=None):
        n = self.n_rays
        out = np.empty(n * N.GVPM_OUT_FLOATS, dtype=np.float32) if out is None else out.reshape(-1)
        cnt = np.empty(n * 2, dtype=np.uint32) if counts else None
        self._ck(self.lib.gvpm_gather_planes(self.h, out.ctypes.data_as(N.f32p),
                                             cnt.ctypes.data_as(N.u32p) if counts else None), "gvpm_gather_planes")
        return out.reshape(n, N.GVPM_OUT_FLOATS), (cnt.reshape(n, 2) if counts else None)

    def dump_neighbours_planes(self):
        return self._dump_neighbours("planes", self.n_rays)

    # ---- G-VPM
    def upload_vpm_samples(self, samples):
        cs = samples.as_c()
        self._ck(self.lib.gvpm_upload_vpm_samples(self.h, C.byref(cs), samples.n), "gvpm_upload_vpm_samples")
        self.n_samples = samples.n

    def generate_vpm_samples(self, nb_camera_samples=40, seed=0, radius=None, radius_per_ray=None, stratified=False,
                             epsilon=1e-4):
        """the distance samples of the current ray set drawn on the device (what synth_vpm_samples draws, in place of
        upload_vpm_samples); radius: one radius for every ray, or radius_per_ray: a device pointer (int) or an object
        with data_ptr(), such as a CUDA float32 tensor of n_rays.  -> number of samples drawn"""
        ptr = None
        if radius_per_ray is not None:
            if hasattr(radius_per_ray, "data_ptr"):
                if str(getattr(radius_per_ray, "dtype", "float32")).rsplit(".", 1)[-1] != "float32":
                    raise ValueError("radius_per_ray must hold float32")
                if getattr(radius_per_ray, "is_cuda", True) is False:
                    raise ValueError("radius_per_ray must be in device memory")
                if hasattr(radius_per_ray, "numel") and radius_per_ray.numel() < self.n_rays:
                    raise ValueError(f"radius_per_ray holds {radius_per_ray.numel()} values for {self.n_rays} rays")
                ptr = radius_per_ray.data_ptr()
            else:
                ptr = int(radius_per_ray)
        n = C.c_size_t(0)
        self._ck(self.lib.gvpm_generate_vpm_samples(self.h, int(nb_camera_samples), int(bool(stratified)),
                                                    C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF),
                                                    C.c_float(epsilon), C.c_float(0.0 if radius is None else radius),
                                                    C.c_void_p(ptr) if ptr else None, C.byref(n)),
                 "gvpm_generate_vpm_samples")
        self.n_samples = int(n.value)
        return self.n_samples

    def download_vpm_samples(self):
        """parity aid: the current distance samples (uploaded or drawn on the device) as a VpmSampleSet"""
        from . import records as R
        return self._download_staged(4, R.VpmSampleSet, R._VPM_FIELDS)

    def gather_vpm_device(self, nb_camera_samples):
        o, m = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.gvpm_gather_vpm_device(self.h, nb_camera_samples, C.byref(o), C.byref(m)),
                 "gvpm_gather_vpm_device")
        return o.value, m.value

    def gather_vpm(self, nb_camera_samples, out=None, mvol=None, sample_counts=True):
        """-> (out [n_rays,27], mvol [n_rays] uint32, sample_counts [n_samples,2] uint32 or None), on the host."""
        n, ns = self.n_rays, self.n_samples
        out = np.empty(n * N.GVPM_OUT_FLOATS, dtype=np.float32) if out is None else out.reshape(-1)
        mvol = np.empty(n, dtype=np.uint32) if mvol is None else mvol
        sc = np.empty(ns * 2, dtype=np.uint32) if sample_counts else None
        self._ck(self.lib.gvpm_gather_vpm(self.h, nb_camera_samples, out.ctypes.data_as(N.f32p),
                                          mvol.ctypes.data_as(N.u32p), sc.ctypes.data_as(N.u32p) if sample_counts else None),
                 "gvpm_gather_vpm")
        return out.reshape(n, N.GVPM_OUT_FLOATS), mvol, (sc.reshape(ns, 2) if sample_counts else None)

    def dump_neighbours_vpm(self, nb_camera_samples):
        return self._dump_neighbours("vpm", self.n_samples, nb_camera_samples)

    def compute_gradient(self, acc, w, h, use_abs=False, reuse_primal=False, inv_emitted=1.0):
        """computeGradient (gvpm.cpp:1205-1306); reuse_primal: throughput by gvpm.cpp:503-532 (inv_emitted = 1 for the
        APA estimators, 1 / totalEmittedVolume for G-VPM)"""
        acc = np.ascontiguousarray(acc, dtype=np.float32).reshape(-1)
        assert acc.size == w * h * N.GVPM_OUT_FLOATS
        thr, gx, gy = (np.empty(w * h * 3, dtype=np.float32) for _ in range(3))
        if reuse_primal:
            self._ck(self.lib.gvpm_compute_gradient_reuse_primal(self.h, acc.ctypes.data_as(N.f32p), w, h, int(use_abs),
                                                                 C.c_float(inv_emitted), thr.ctypes.data_as(N.f32p),
                                                                 gx.ctypes.data_as(N.f32p), gy.ctypes.data_as(N.f32p)),
                     "gvpm_compute_gradient_reuse_primal")
        else:
            self._ck(self.lib.gvpm_compute_gradient(self.h, acc.ctypes.data_as(N.f32p), w, h, int(use_abs),
                                                    thr.ctypes.data_as(N.f32p), gx.ctypes.data_as(N.f32p),
                                                    gy.ctypes.data_as(N.f32p)), "gvpm_compute_gradient")
        return thr.reshape(h, w, 3), gx.reshape(h, w, 3), gy.reshape(h, w, 3)

    def poisson_solve(self, throughput, dx, dy, direct=None, preset="L2D", **params):
        """Screened-Poisson reconstruction (poisson::Solver).  Planes [h, w, 3] float32; throughput / direct may be
        None.  preset: L1D | L1Q | L1L | L2D | L2Q; params override its fields (alpha, cg_iter_max, ...)."""
        p = poisson_params(preset, **params)
        h, w, _ = dx.shape
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=np.float32) for a in (throughput, dx, dy, direct)]
        ptr = [None if a is None else a.ctypes.data_as(N.f32p) for a in arrs]
        rec = np.empty((h, w, 3), dtype=np.float32)
        self._ck(self.lib.gvpm_poisson_solve(self.h, w, h, ptr[0], ptr[1], ptr[2], ptr[3], C.byref(p),
                                             rec.ctypes.data_as(N.f32p)), "gvpm_poisson_solve")
        return rec

    def reconstruct(self, acc, w, h, direct=None, preset="L2D", use_abs=False, **params):
        """computeGradient + Poisson reconstruction in one call -> (throughput, gx, gy, reconstruction), [h, w, 3]."""
        p = poisson_params(preset, **params)
        acc = np.ascontiguousarray(acc, dtype=np.float32).reshape(-1)
        assert acc.size == w * h * N.GVPM_OUT_FLOATS
        d = None if direct is None else np.ascontiguousarray(direct, dtype=np.float32)
        thr, gx, gy, rec = (np.empty((h, w, 3), dtype=np.float32) for _ in range(4))
        self._ck(self.lib.gvpm_reconstruct(self.h, acc.ctypes.data_as(N.f32p), w, h, int(use_abs),
                                           None if d is None else d.ctypes.data_as(N.f32p), C.byref(p),
                                           thr.ctypes.data_as(N.f32p), gx.ctypes.data_as(N.f32p),
                                           gy.ctypes.data_as(N.f32p), rec.ctypes.data_as(N.f32p)), "gvpm_reconstruct")
        return thr, gx, gy, rec

    # ---- per-pixel accumulators on the device (gvpm_accum_*)
    def accum_reset(self, w, h, channels=N.GVPM_OUT_FLOATS, apa=True):
        """zeroed accumulators of w x h pixels: channels 27 (gvpm) or 3 (sppm); apa=False for G-VPM's plain sum"""
        self._ck(self.lib.gvpm_accum_reset(self.h, int(w), int(h), int(channels), int(bool(apa))), "gvpm_accum_reset")
        self._accum_shape = (int(h), int(w), int(channels))

    def accum_add(self):
        """add the per-ray results of the last gather on the current ray set to their pixels"""
        self._ck(self.lib.gvpm_accum_add(self.h), "gvpm_accum_add")

    def accum_fold(self, it, n_paths):
        """end of iteration `it` (from 1) of n_paths light paths: APA running mean, or the emitted total (G-VPM)"""
        self._ck(self.lib.gvpm_accum_fold(self.h, int(it), C.c_uint64(int(n_paths))), "gvpm_accum_fold")

    def accum_read(self, normalized=False):
        """-> (acc [h,w,C] float32, have_smoke [h,w] uint8, emitted-path total)"""
        h, w, c = getattr(self, "_accum_shape", (0, 0, 0))
        acc = np.empty((h, w, c), dtype=np.float32)
        smoke = np.empty((h, w), dtype=np.uint8)
        total = C.c_uint64(0)
        self._ck(self.lib.gvpm_accum_read(self.h, int(bool(normalized)), acc.ctypes.data_as(N.f32p),
                                          smoke.ctypes.data_as(N.u8p), C.byref(total)), "gvpm_accum_read")
        return acc, smoke, int(total.value)

    def accum_device(self):
        """-> (acc device pointer, have_smoke device pointer), owned by the context"""
        a, s = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.gvpm_accum_device(self.h, C.byref(a), C.byref(s)), "gvpm_accum_device")
        return a.value, s.value

    def compute_gradient_accum(self, use_abs=False, reuse_primal=False, inv_emitted=1.0):
        """compute_gradient on the device accumulators -> (throughput, gx, gy), [h, w, 3]"""
        h, w, _ = getattr(self, "_accum_shape", (0, 0, 0))
        thr, gx, gy = (np.empty((h, w, 3), dtype=np.float32) for _ in range(3))
        self._ck(self.lib.gvpm_compute_gradient_accum(self.h, int(use_abs), int(reuse_primal), C.c_float(inv_emitted),
                                                      thr.ctypes.data_as(N.f32p), gx.ctypes.data_as(N.f32p),
                                                      gy.ctypes.data_as(N.f32p)), "gvpm_compute_gradient_accum")
        return thr, gx, gy

    def reconstruct_accum(self, direct=None, preset="L2D", use_abs=False, **params):
        """reconstruct on the device accumulators -> (throughput, gx, gy, reconstruction), [h, w, 3]"""
        p = poisson_params(preset, **params)
        h, w, _ = getattr(self, "_accum_shape", (0, 0, 0))
        d = None if direct is None else np.ascontiguousarray(direct, dtype=np.float32)
        thr, gx, gy, rec = (np.empty((h, w, 3), dtype=np.float32) for _ in range(4))
        self._ck(self.lib.gvpm_reconstruct_accum(self.h, int(use_abs), None if d is None else d.ctypes.data_as(N.f32p),
                                                 C.byref(p), thr.ctypes.data_as(N.f32p), gx.ctypes.data_as(N.f32p),
                                                 gy.ctypes.data_as(N.f32p), rec.ctypes.data_as(N.f32p)),
                 "gvpm_reconstruct_accum")
        return thr, gx, gy, rec

    def last_poisson_ms(self):
        return float(self.lib.gvpm_last_poisson_ms(self.h))

    def sync(self):
        self._ck(self.lib.gvpm_sync(self.h), "gvpm_sync")

    def stream(self):
        return self.lib.gvpm_stream(self.h)

    def last_timings(self):
        b, g = C.c_float(), C.c_float()
        self._ck(self.lib.gvpm_last_timings(self.h, C.byref(b), C.byref(g)), "gvpm_last_timings")
        return b.value, g.value

    def last_gather_detail(self):
        """-> (traverse_ms, shade_ms, contributing pairs) of the last gather."""
        t, s, p = C.c_float(), C.c_float(), C.c_uint64()
        self._ck(self.lib.gvpm_last_gather_detail(self.h, C.byref(t), C.byref(s), C.byref(p)),
                 "gvpm_last_gather_detail")
        return t.value, s.value, int(p.value)

    def launch_count(self):
        return int(self.lib.gvpm_launch_count(self.h))


def poisson_params(preset="L2D", **params):
    """gvpm_poisson_preset + field overrides -> PoissonParams"""
    p = N.PoissonParams()
    if N.load_lib().gvpm_poisson_preset(preset.encode(), C.byref(p)) != 0:
        raise ValueError(f"unknown Poisson preset {preset!r}")
    for k, v in params.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p
