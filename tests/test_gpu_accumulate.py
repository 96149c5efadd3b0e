"""Per-pixel accumulators on the device (gvpm_accum_*): the fold of every gather technique against a numpy restatement
of the host mirror's foldIteration, bit for bit, fed the per-ray output of the same gather (the float-atomic gathers
are not bit-reproducible between runs, so each is compared with its own output); the plane gather (no atomics)
against the host mirror itself; device-made iterations, ray batches, image shards, a pair-list overflow, the image
hand-off, and the call-order errors."""
import ctypes as C

import numpy as np
import pytest

import gvpm_b200 as g
import gvpm_testlib as H
from gvpm_b200 import _native as N
from gvpm_b200 import records as R
from gvpm_b200 import shard

pytestmark = pytest.mark.gpu
F32 = np.float32


class Restated:
    """VolumeGatherB200 / SPPMVolumeGatherB200::foldIteration and computeVolumeGradientPhoton in numpy float32"""

    def __init__(self, w, h, channels=27, apa=True):
        self.w, self.h, self.c, self.apa = w, h, channels, apa
        self.acc = np.zeros((h * w, channels), dtype=F32)
        self.pix = np.zeros((h * w, channels), dtype=F32)
        self.smoke = np.zeros(h * w, dtype=np.uint8)
        self.total = 0

    def add(self, out, px, py):
        m = (px >= 0) & (py >= 0) & (px < self.w) & (py < self.h)
        p = py[m].astype(np.int64) * self.w + px[m]
        self.smoke[p] = 1
        np.add.at(self.pix if self.apa else self.acc, p, np.asarray(out, dtype=F32)[m][:, :self.c])   # ray order

    def fold(self, it, n_paths):
        if not self.apa:
            self.total += n_paths
            return
        rnb, rit = F32(1.0) / F32(n_paths), F32(1.0) / F32(it)
        self.acc = (self.acc * F32(it - 1) + self.pix * rnb) * rit
        self.pix[:] = 0

    def image(self, normalized=False):
        a = self.acc.copy()
        if normalized and not self.apa and self.total:
            a *= F32(1.0) / F32(self.total)
        return a.reshape(self.h, self.w, self.c)


def _same_bits(got, ref, what):
    got, ref = np.ascontiguousarray(got, dtype=F32), np.ascontiguousarray(ref, dtype=F32)
    assert got.shape == ref.shape, what
    bad = int(np.count_nonzero(got.view(np.uint32) != ref.view(np.uint32)))
    assert bad == 0, f"{what}: {bad} of {got.size} values differ"


def _check(ctx, ref, what, normalized=False):
    acc, smoke, total = ctx.accum_read(normalized)
    _same_bits(acc, ref.image(normalized), what)
    np.testing.assert_array_equal(smoke.reshape(-1), ref.smoke, err_msg=what)
    assert total == ref.total
    assert np.abs(acc).max() > 0, what


def _read_out(ctx, ptr, n, stride=N.GVPM_OUT_FLOATS):
    a = np.empty((n, stride), dtype=F32)
    if n:
        ctx._ck(ctx.lib.gvpm_read_device(ctx.h, C.c_void_p(ptr), a.ctypes.data_as(C.c_void_p), a.nbytes),
                "gvpm_read_device")
    return a


def _scrambled(rays, w, h, seed):
    """shuffled rays, a third of them moved onto random pixels (several records per pixel), a few outside the film"""
    rng = np.random.default_rng(seed)
    idx = np.concatenate([np.arange(rays.n), rng.integers(0, rays.n, rays.n // 2)])
    r = rays.take(rng.permutation(idx))
    k = rng.choice(r.n, r.n // 3, replace=False)
    r.px[k] = rng.integers(0, w, k.size)
    r.py[k] = rng.integers(0, h, k.size)
    r.px[:4], r.py[4:7], r.px[7:9], r.py[9:11] = -1, -2, w, h
    return r


def _ctx(medium, config, tri=None):
    from gvpm_b200.api import Context
    ctx = Context(0)
    ctx.set_medium(medium)
    ctx.set_config(config)
    ctx.set_occluders(g.synth_occluders() if tri is None else tri)
    return ctx


W, HH = 40, 24


def _iteration(tech, ctx, it):
    """one iteration's inputs uploaded and gathered -> (per-ray output of that gather, rays, n_paths)"""
    seed = 0xACC + 101 * it
    if tech == "planes":
        c = H.make_plane_case(n_planes=1500, w=W, h=HH, seed=seed)
        rays = _scrambled(c.rays, W, HH, seed)
        ctx.upload_planes(c.planes)
        ctx.build_planes()
        ctx.upload_rays(rays)
        return _read_out(ctx, ctx.gather_planes_device()[0], rays.n), rays, c.n_paths
    c = H.make_case(n_photons=20000, w=W, h=HH, scale=3.0, seed=seed)
    rays = _scrambled(c.rays, W, HH, seed)
    if tech in ("beam3d", "beam1d", "sppm_beam3d"):
        beams, n_paths = R.synth_beams(4000, c.medium, seed=seed + 3, threads=4)
        ctx.upload_beams(beams)
        ctx.build_beams(c.radius)
        ctx.upload_rays(rays)
        if tech == "sppm_beam3d":
            return ctx.gather_sppm_beams("beam3d", counts=False)[0], rays, n_paths
        if it == 2:
            return _read_out(ctx, ctx.gather_beams_device()[0], rays.n), rays, n_paths
        return ctx.gather_beams(counts=False)[0], rays, n_paths
    ctx.upload_photons(c.photons)
    ctx.build_points(c.radius)
    ctx.upload_rays(rays)
    if tech == "vpm":
        rad = np.full(rays.n, c.radius, dtype=F32) * np.random.default_rng(it).uniform(0.5, 1.0, rays.n).astype(F32)
        ctx.upload_vpm_samples(g.synth_vpm_samples(rays, c.medium, rad, nb_camera_samples=8, seed=99 + it))
        if it == 2:
            return _read_out(ctx, ctx.gather_vpm_device(8)[0], rays.n), rays, c.n_paths
        return ctx.gather_vpm(8, sample_counts=False)[0], rays, c.n_paths
    if tech == "sppm_bre":
        return ctx.gather_sppm_bre(counts=False)[0], rays, c.n_paths
    if it == 2:   # asynchronous: accum_add completes it
        return None, rays, c.n_paths
    return ctx.gather_bre(counts=False)[0], rays, c.n_paths


TECHS = {  # technique: (config overrides, channels, apa)
    "bre3d": ({}, 27, True),
    "bre2d": ({"kernel_3d": False, "use_shift_null": False}, 27, True),
    "beam3d": ({}, 27, True),
    "beam1d": ({"beam_kernel_1d": True}, 27, True),
    "planes": ({}, 27, True),
    "vpm": ({}, 27, False),
    "sppm_bre": ({"sppm_primal": True}, 3, True),
    "sppm_beam3d": ({"sppm_primal": True, "rng_seed": 7}, 3, True),
}


@pytest.mark.parametrize("tech", list(TECHS))
def test_fold_equals_the_restatement(built, tech):
    cfg, channels, apa = TECHS[tech]
    ctx = _ctx(g.make_medium(), g.make_config(W, HH, **cfg))
    ctx.accum_reset(W, HH, channels, apa)
    ref = Restated(W, HH, channels, apa)
    for it in (1, 2, 3):
        out, rays, n_paths = _iteration(tech, ctx, it)
        if out is None:
            ptr, _ = ctx.gather_bre_device()
            ctx.accum_add()
            out = _read_out(ctx, ptr, rays.n)
        else:
            ctx.accum_add()
        ctx.accum_fold(it, n_paths)
        ref.add(out, rays.px, rays.py)
        ref.fold(it, n_paths)
        _check(ctx, ref, f"{tech} iteration {it}")
    if not apa:
        _check(ctx, ref, f"{tech} normalised", normalized=True)
    ctx.close()


def test_planes_fold_equals_the_host_mirror(built):
    """the plane gather has no float atomics: the host mirror's whole iteration (gather + foldIteration) and a second
    context's gather + add + fold give the same accumulators"""
    from test_gpu_host_drivers import _create, _host_lib
    hl = _host_lib()
    c0 = H.make_plane_case(n_planes=64, w=W, h=HH)
    tri = g.synth_occluders()
    hd, err = _create(hl, W, HH, c0.medium, tri, initialScaleVolume=1.0, volTechnique=4)   # EVolPlane0D
    ctx = _ctx(c0.medium, g.make_config(W, HH), tri)
    ctx.accum_reset(W, HH)
    for it in (1, 2, 3):
        c = H.make_plane_case(n_planes=1500, w=W, h=HH, seed=0xC0FFEE + it)
        rays = _scrambled(c.rays, W, HH, it)
        cp, cr = c.planes.as_c(), rays.as_c()
        assert hl.gvpm_host_planes_iteration(hd, it, C.byref(cp), c.planes.n, C.byref(cr), rays.n, c.n_paths, err,
                                             512) == 0, err.value
        ctx.upload_planes(c.planes)
        ctx.build_planes()
        ctx.upload_rays(rays)
        ctx.gather_planes_device()
        ctx.accum_add()
        ctx.accum_fold(it, c.n_paths)
        mirror = np.ctypeslib.as_array(hl.gvpm_host_accumulators(hd), shape=(HH, W, 27)).copy()
        acc, _, _ = ctx.accum_read()
        assert np.abs(mirror).max() > 0
        _same_bits(acc, mirror, f"planes, host mirror, iteration {it}")
    hl.gvpm_host_destroy(hd)
    ctx.close()


def _device_iterations(prims, w=64, h=48, iters=4):
    scene = g.box_scene_default()
    cam = g.pinhole_camera(w, h) if prims == "photons" else g.pinhole_camera(w, h, cam_dist=-0.05, cover=0.45)
    medium = g.make_medium()
    ctx = _ctx(medium, g.make_config(w, h))
    ctx.accum_reset(w, h)
    ref = Restated(w, h)
    scale = 3.0
    for it in range(1, iters + 1):
        seed = 0xD0 + it
        ctx.generate_rays(scene, cam, seed, block=-32)
        radius = g.bre_radius(scale)
        if prims == "photons":
            n_paths = ctx.trace_photons(scene, 40000, seed, direct=True)
            ctx.build_points_for_rays(radius, want_kept=False)
            ptr, _ = ctx.gather_bre_device()
        else:
            n_paths = ctx.trace_beams(scene, 3000, seed)
            ctx.planes_from_beams(seed + 7)
            ctx.build_planes()
            ptr, _ = ctx.gather_planes_device()
        ctx.accum_add()
        ctx.accum_fold(it, n_paths)
        rays = ctx.download_rays()
        ref.add(_read_out(ctx, ptr, rays.n), rays.px, rays.py)
        ref.fold(it, n_paths)
        scale *= ((it - 1 + 0.7) / it) ** (1.0 / 3.0)
    _check(ctx, ref, f"device-made {prims}, {iters} iterations")
    assert ref.smoke.all()
    ctx.close()


def test_device_made_bre_iterations(built):
    _device_iterations("photons")


def test_device_made_plane_iterations(built):
    """camera inside the medium, as the plane technique requires"""
    _device_iterations("planes")


def test_batches_equal_one_batch(built):
    """an iteration whose rays come as two row ranges of gvpm_generate_rays == the restatement over their concatenation"""
    w, h = 64, 48
    scene, cam = g.box_scene_default(), g.pinhole_camera(w, h)
    ctx = _ctx(g.make_medium(), g.make_config(w, h))
    ctx.accum_reset(w, h)
    ref = Restated(w, h)
    for it in (1, 2):
        n_paths = ctx.trace_photons(scene, 40000, 77 + it, direct=True)
        for y0, y1 in ((0, 20), (20, h)):
            ctx.generate_rays(scene, cam, 5 + it, block=-32, y0=y0, y1=y1)
            ctx.build_points_for_rays(g.bre_radius(3.0), want_kept=False)
            ptr, _ = ctx.gather_bre_device()
            ctx.accum_add()
            rays = ctx.download_rays()
            ref.add(_read_out(ctx, ptr, rays.n), rays.px, rays.py)
        ctx.accum_fold(it, n_paths)
        ref.fold(it, n_paths)
    _check(ctx, ref, "two row ranges per iteration")
    ctx.close()


def test_image_shards_sum_to_the_whole(built):
    """two contexts holding the two column-band halves of an uploaded ray set: their accumulators sum to the
    restatement over all rays, bit for bit"""
    ranks = [None, None]
    ref = Restated(W, HH)
    for r in (0, 1):
        ranks[r] = _ctx(g.make_medium(), g.make_config(W, HH))
        ranks[r].accum_reset(W, HH)
    for it in (1, 2):
        c = H.make_case(n_photons=20000, w=W, h=HH, scale=3.0, seed=0x5A + it)
        rays = _scrambled(c.rays, W, HH, it)
        outs, parts = [], []
        for r, ctx in enumerate(ranks):
            part = rays.take(shard.band_indices(rays.px, rays.py, W, HH, 2, r))
            ctx.upload_photons(c.photons)
            ctx.build_points(c.radius)
            ctx.upload_rays(part)
            outs.append(ctx.gather_bre(counts=False)[0])
            parts.append(part)
            ctx.accum_add()
            ctx.accum_fold(it, c.n_paths)
        ref.add(np.concatenate(outs), np.concatenate([p.px for p in parts]), np.concatenate([p.py for p in parts]))
        ref.fold(it, c.n_paths)
    (a0, s0, _), (a1, s1, _) = (ctx.accum_read() for ctx in ranks)
    _same_bits(a0 + a1, ref.image(), "sum of two column-band shards")
    np.testing.assert_array_equal((s0 | s1).reshape(-1), ref.smoke)
    assert not (s0 & s1).any()
    for ctx in ranks:
        ctx.close()


def test_add_completes_an_overflowed_asynchronous_gather(built):
    """dense case of test_gpu_pair_overflow on a fresh context: gather_bre_device, then accum_add with no sync"""
    from oracle import binding as ob
    c = H.make_case(n_photons=150000, w=32, h=24, scale=14.0)
    ref_out = ob.bre_gather(c.photons, c.rays, c.medium, c.config, c.tri, c.radius, mode="brute").out
    ctx = H.gpu_context(c)
    ctx.accum_reset(c.w, c.h)
    ctx.gather_bre_device()
    ctx.accum_add()
    ctx.accum_fold(1, c.n_paths)
    assert ctx.last_gather_detail()[2] > max(1 << 20, 16 * c.rays.n)   # the list did overflow
    acc, _, _ = ctx.accum_read()
    blocking = Restated(c.w, c.h)
    blocking.add(ctx.gather_bre(counts=False)[0], c.rays.px, c.rays.py)
    blocking.fold(1, c.n_paths)
    oracle = Restated(c.w, c.h)
    oracle.add(ref_out, c.rays.px, c.rays.py)
    oracle.fold(1, c.n_paths)
    # the two gathers sum the same pairs by float atomics in different orders (measured 2.0e-6 on a B200); 1e-5 is the
    # tolerance test_gpu_pair_overflow allows between two gathers of the same inputs
    assert float(H.rel_err(acc, blocking.image()).max()) <= 1e-5
    H.assert_radiance_close(acc.reshape(-1, 27), oracle.image().reshape(-1, 27), 1e-4, "overflowed gather, folded")
    ctx.close()


@pytest.mark.parametrize("apa", [True, False])
def test_image_hand_off(built, apa):
    """compute_gradient_accum / reconstruct_accum == compute_gradient / reconstruct on accum_read()'s array"""
    ctx = _ctx(g.make_medium(), g.make_config(W, HH))
    ctx.accum_reset(W, HH, apa=apa)
    for it in (1, 2):
        out, rays, n_paths = _iteration("bre3d", ctx, it)
        if out is None:
            ctx.gather_bre_device()
        ctx.accum_add()
        ctx.accum_fold(it, n_paths)
    acc, _, total = ctx.accum_read()
    inv = 1.0 if apa else float(F32(1.0) / F32(total))
    for reuse in (False, True):
        got = ctx.compute_gradient_accum(use_abs=True, reuse_primal=reuse, inv_emitted=inv)
        want = ctx.compute_gradient(acc, W, HH, use_abs=True, reuse_primal=reuse, inv_emitted=inv)
        for a, b, name in zip(got, want, ("throughput", "gx", "gy")):
            _same_bits(a, b, f"gradient {name}, reuse_primal={reuse}")
    for preset in ("L2D", "L1D"):
        got = ctx.reconstruct_accum(preset=preset, alpha=0.2)
        want = ctx.reconstruct(acc, W, HH, preset=preset, alpha=0.2)
        for a, b, name in zip(got, want, ("throughput", "gx", "gy", "reconstruction")):
            _same_bits(a, b, f"reconstruct {preset} {name}")
    ctx.close()


def _fails(ctx, fn, *args):
    rc = fn(ctx.h, *args)
    assert rc == -1, rc   # GVPM_ERR_INVALID
    msg = ctx.lib.gvpm_last_error(ctx.h).decode()
    assert msg, "no message"
    return msg


def test_call_order_errors(built):
    c = H.make_case(n_photons=20000, w=W, h=HH, scale=3.0)
    ctx = H.gpu_context(c)
    lib = ctx.lib
    f = np.empty(W * HH * 27, dtype=F32)
    fp = f.ctypes.data_as(N.f32p)
    # before any reset
    _fails(ctx, lib.gvpm_accum_add)
    _fails(ctx, lib.gvpm_accum_fold, 1, 10)
    _fails(ctx, lib.gvpm_accum_read, 0, fp, None, None)
    _fails(ctx, lib.gvpm_accum_device, None, None)
    _fails(ctx, lib.gvpm_compute_gradient_accum, 0, 0, C.c_float(1.0), fp, fp, fp)
    p = N.PoissonParams()
    lib.gvpm_poisson_preset(b"L2D", C.byref(p))
    _fails(ctx, lib.gvpm_reconstruct_accum, 0, None, C.byref(p), None, None, None, fp)
    # reset arguments
    _fails(ctx, lib.gvpm_accum_reset, 0, HH, 27, 1)
    _fails(ctx, lib.gvpm_accum_reset, W, -1, 27, 1)
    _fails(ctx, lib.gvpm_accum_reset, W, HH, 9, 1)
    ctx.accum_reset(W, HH)
    _fails(ctx, lib.gvpm_accum_fold, 0, 10)
    _fails(ctx, lib.gvpm_accum_fold, 1, 0)
    # no gather since the last ray-set change
    assert "ray set" in _fails(ctx, lib.gvpm_accum_add)
    ctx.gather_bre(counts=False)
    ctx.upload_rays(c.rays)
    assert "ray set" in _fails(ctx, lib.gvpm_accum_add)
    ctx.gather_bre_device()
    ctx.ray_staging(c.rays.n)
    assert "ray set" in _fails(ctx, lib.gvpm_accum_add)
    ctx.generate_rays(g.box_scene_default(), g.pinhole_camera(W, HH), 3)
    assert "ray set" in _fails(ctx, lib.gvpm_accum_add)
    # added twice
    ctx.upload_rays(c.rays)
    ctx.gather_bre_device()
    ctx.accum_add()
    assert "already" in _fails(ctx, lib.gvpm_accum_add)
    # the last gather wrote to caller memory
    import torch
    buf = torch.empty(c.rays.n * 27, dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    ctx.gather_bre_into(buf.data_ptr())
    assert "caller memory" in _fails(ctx, lib.gvpm_accum_add)
    ctx.sync()
    # 27 channels from a gather that writes 3 floats per ray
    beams, _ = R.synth_beams(3000, c.medium, seed=3, threads=4)
    ctx.set_config(g.make_config(W, HH, sppm_primal=True))
    ctx.upload_beams(beams)
    ctx.build_beams(c.radius)
    ctx.gather_sppm_beams("beam3d", counts=False)
    assert "fewer floats" in _fails(ctx, lib.gvpm_accum_add)
    # the image hand-off needs 27 channels
    ctx.accum_reset(W, HH, channels=3)
    ctx.accum_add()   # the sppm beam output fits a 3-channel accumulator
    assert "27" in _fails(ctx, lib.gvpm_compute_gradient_accum, 0, 0, C.c_float(1.0), fp, fp, fp)
    assert "27" in _fails(ctx, lib.gvpm_reconstruct_accum, 0, None, C.byref(p), None, None, None, fp)
    ctx.close()


def test_gather_bre_host_is_accumulated(built):
    """the pipelined host gather leaves the whole ray set and its output in the context: it can be added"""
    c = H.make_case(n_photons=20000, w=W, h=HH, scale=3.0)
    ctx = H.gpu_context(c)
    ctx.accum_reset(W, HH)
    rays = _scrambled(c.rays, W, HH, 5)
    out = ctx.gather_bre_host(rays).copy()
    ctx.accum_add()
    ctx.accum_fold(1, c.n_paths)
    ref = Restated(W, HH)
    ref.add(out, rays.px, rays.py)
    ref.fold(1, c.n_paths)
    _check(ctx, ref, "gvpm_gather_bre_host")
    ctx.close()
