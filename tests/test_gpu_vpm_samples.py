"""G-VPM camera distance samples drawn on the device (gvpm_generate_vpm_samples):
  1. bit for bit equal to the CPU restatement (tests/vpm_samples_ref.cpp) over uploaded and generated ray sets;
  2. the gather on them against the CPU oracle (counts, index sets and MVol exact, radiance within 1e-4);
  3. the context they leave equals an upload of the same arrays (float-atomic radiance within 1e-6);
  4. a three-iteration device G-VPM render equals the same render fed the samples through the host;
  5. every refusal, including samples drawn for an earlier ray set."""
import ctypes as C

import numpy as np
import pytest

import gvpm_b200 as g
import gvpm_testlib as H
import vpm_samples_ref as P
from gvpm_b200.api import Context, GvpmError

pytestmark = pytest.mark.gpu
F32 = np.float32
FIELDS = ("ray", "t", "transmittance", "pdf_success", "pdf_sel", "radius")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def _device_array(torch, a):
    t = torch.tensor(np.asarray(a, dtype=F32), device="cuda:0")
    torch.cuda.synchronize()   # the context's stream does not wait for torch's copy
    return t


def _same_samples(got, ref, what):
    assert got.n == ref.n, f"{what}: {got.n} samples, restatement {ref.n}"
    for f in FIELDS:
        a, b = getattr(got, f), getattr(ref, f)
        bad = int(np.count_nonzero(a.view(np.uint32) != b.view(np.uint32)))
        assert bad == 0, f"{what}: {f} differs in {bad} of {a.size} values"


def _with_short_segments(rays, seed):
    """some segments empty, some at or just above the 4 epsilon threshold"""
    rng = np.random.default_rng(seed)
    idx = rng.choice(rays.n, 200, replace=False)
    rays.edge_len[idx[:60]] = 0.0
    rays.edge_len[idx[60:90]] = F32(4e-4)
    rays.edge_len[idx[90:]] = rng.uniform(2e-4, 3e-3, 110).astype(F32)
    rays.maxt[idx] = np.maximum(rays.edge_len[idx] - F32(1e-4), 0)
    return rays


def _context(medium, rays_source, w, h, seed):
    """a context holding a ray set: uploaded synthetic rays, or gvpm_generate_rays (whole image or a band of rows)"""
    ctx = Context(0)
    ctx.set_medium(medium)
    if rays_source == "uploaded":
        ctx.upload_rays(_with_short_segments(g.synth_rays(w, h, seed=seed), seed))
    else:
        y0, y1 = (0, h) if rays_source == "generated" else (h // 4, 3 * h // 4)
        ctx.generate_rays(g.box_scene_default(), g.pinhole_camera(w, h), seed, block=-32, y0=y0, y1=y1)
    return ctx


# ---- 1. bit for bit against the restatement ---------------------------------------------------------------------------
@pytest.mark.parametrize("rays_source", ["uploaded", "generated", "row_band"])
@pytest.mark.parametrize("stratified", [False, True])
@pytest.mark.parametrize("nb", [1, 8, 40])
@pytest.mark.parametrize("per_ray", [False, True])
def test_device_samples_equal_the_restatement(built, torch_cuda, rays_source, stratified, nb, per_ray):
    w, h, seed = 72, 40, 0x5EED + nb
    medium = g.make_medium(sigma_t=2.5, albedo=0.7)
    ctx = _context(medium, rays_source, w, h, seed)
    rays = ctx.download_rays()
    rad = np.random.default_rng(seed).uniform(0.005, 0.04, rays.n).astype(F32) if per_ray else None
    kw = dict(nb_camera_samples=nb, seed=seed, stratified=stratified, epsilon=1e-4)
    if per_ray:
        n = ctx.generate_vpm_samples(radius_per_ray=_device_array(torch_cuda, rad), **kw)
        ref = P.vpm_samples(rays, medium, radius_per_ray=rad, **kw)
    else:
        n = ctx.generate_vpm_samples(radius=0.02, **kw)
        ref = P.vpm_samples(rays, medium, radius=0.02, **kw)
    assert n == ref.n > 0.5 * nb * rays.n
    _same_samples(ctx.download_vpm_samples(), ref, f"{rays_source}, nb {nb}, stratified {stratified}")
    ctx.close()


# ---- 2. the gather on device-drawn samples against the oracle ----------------------------------------------------------
def _vpm_case(nb=8, **kw):
    c = H.make_case(n_photons=60000, w=40, h=24, scale=3.0, **kw)
    c.nb = nb
    return c


@pytest.mark.parametrize("kw,per_ray", [
    ({}, True),
    ({"phase": "hg", "hg_g": 0.4}, False),
    ({"use_shift_null": False}, True),
])
def test_gather_on_device_samples_matches_oracle(built, torch_cuda, kw, per_ray):
    from oracle import binding as ob
    c = _vpm_case(**kw)
    ctx = H.gpu_context(c)
    if per_ray:
        rad = (F32(c.radius) * np.random.default_rng(2).uniform(0.4, 1.0, c.rays.n)).astype(F32)
        ctx.generate_vpm_samples(c.nb, seed=99, radius_per_ray=_device_array(torch_cuda, rad))
    else:
        ctx.generate_vpm_samples(c.nb, seed=99, radius=c.radius)
    samples = ctx.download_vpm_samples()
    ref = ob.vpm_gather(c.photons, c.rays, samples, c.medium, c.config, c.tri, c.nb, mode="brute", neighbours=True)
    out, mvol, sc = ctx.gather_vpm(c.nb)
    offsets, idx = ctx.dump_neighbours_vpm(c.nb)
    np.testing.assert_array_equal(sc, ref.sample_counts)
    np.testing.assert_array_equal(mvol.astype(F32), ref.mvol)
    np.testing.assert_array_equal(offsets, ref.offsets)
    np.testing.assert_array_equal(idx, ref.idx)
    H.assert_radiance_close(out, ref.out, 1e-4, f"vpm on device samples {kw}")
    assert ref.sample_counts[:, 0].sum() > 2000
    ctx.close()


def test_sppm_shaped_pass_on_device_samples(built):
    """sppm's point-photon volume pass: no valid offset path"""
    from oracle import binding as ob
    c = _vpm_case(max_depth=6)
    c.rays = c.rays.copy()
    c.rays.off_valid[:] = 0
    ctx = H.gpu_context(c)
    ctx.generate_vpm_samples(c.nb, seed=5, radius=c.radius, stratified=True)
    samples = ctx.download_vpm_samples()
    ref = ob.vpm_gather(c.photons, c.rays, samples, c.medium, c.config, c.tri, c.nb, mode="brute")
    out, mvol, sc = ctx.gather_vpm(c.nb)
    np.testing.assert_array_equal(sc, ref.sample_counts)
    np.testing.assert_array_equal(mvol.astype(F32), ref.mvol)
    H.assert_radiance_close(out, ref.out, 1e-4, "sppm-shaped vpm on device samples")
    assert not out.reshape(-1, 9, 3)[:, 1:5].any()
    ctx.close()


# ---- 3. the same context state as an upload of the same arrays ---------------------------------------------------------
def test_drawn_samples_leave_the_state_of_an_upload(built, torch_cuda):
    c = _vpm_case(nb=12)
    ctx = H.gpu_context(c)
    rad = (F32(c.radius) * np.random.default_rng(4).uniform(0.5, 1.0, c.rays.n)).astype(F32)
    n = ctx.generate_vpm_samples(c.nb, seed=3, radius_per_ray=_device_array(torch_cuda, rad))
    out_d, mvol_d, sc_d = ctx.gather_vpm(c.nb)
    samples = ctx.download_vpm_samples()
    assert samples.n == n
    ctx.upload_vpm_samples(samples)
    out_u, mvol_u, sc_u = ctx.gather_vpm(c.nb)
    np.testing.assert_array_equal(sc_d, sc_u)
    np.testing.assert_array_equal(mvol_d, mvol_u)
    H.assert_radiance_close(out_d, out_u, 1e-6, "drawn vs uploaded samples")
    # sample_radius_max: a build radius below the largest sample radius is refused either way
    ctx.generate_vpm_samples(c.nb, seed=3, radius=c.radius * 1.5)
    with pytest.raises(GvpmError, match="smaller than a sample radius"):
        ctx.gather_vpm(c.nb)
    ctx.upload_vpm_samples(ctx.download_vpm_samples())
    with pytest.raises(GvpmError, match="smaller than a sample radius"):
        ctx.gather_vpm(c.nb)
    ctx.close()


# ---- 4. a three-iteration device G-VPM render against the host-sample render -------------------------------------------
def test_device_vpm_render_equals_host_sample_render(built):
    w, h, nb = 64, 48, 8
    scene, cam, medium = g.box_scene_default(), g.pinhole_camera(w, h), g.make_medium()
    ctxs = []
    for _ in range(2):
        ctx = Context(0)
        ctx.set_medium(medium)
        ctx.set_config(g.make_config(w, h))
        ctx.set_occluders(g.synth_occluders())
        ctx.accum_reset(w, h, apa=False)
        ctxs.append(ctx)
    dev, host = ctxs
    scale = 3.0
    for it in range(1, 4):
        seed = 0xB0 + it
        radius = g.bre_radius(scale)
        paths = []
        for ctx in ctxs:
            paths.append(ctx.trace_photons(scene, 40000, seed, direct=True))
            ctx.generate_rays(scene, cam, seed, block=-32)
            ctx.build_points_for_rays(radius, want_kept=False)
        assert paths[0] == paths[1]
        dev.generate_vpm_samples(nb, seed=seed, radius=radius)
        host.upload_vpm_samples(dev.download_vpm_samples())
        for ctx, n_paths in zip(ctxs, paths):
            ctx.gather_vpm_device(nb)
            ctx.accum_add()
            ctx.accum_fold(it, n_paths)
        scale *= ((it - 1 + 0.7) / it) ** (1.0 / 3.0)
    acc_d, smoke_d, tot_d = dev.accum_read(normalized=True)
    acc_h, smoke_h, tot_h = host.accum_read(normalized=True)
    assert tot_d == tot_h > 0
    np.testing.assert_array_equal(smoke_d, smoke_h)
    assert np.abs(acc_h).max() > 0
    H.assert_radiance_close(acc_d.reshape(-1, 27), acc_h.reshape(-1, 27), 1e-6, "device vs host-sample render")
    for ctx in ctxs:
        ctx.close()


# ---- 5. refusals -------------------------------------------------------------------------------------------------------
def _refused(ctx, match, **kw):
    args = dict(nb_camera_samples=8, seed=1, radius=0.02)
    args.update(kw)
    with pytest.raises(GvpmError, match=match):
        ctx.generate_vpm_samples(**args)


def test_refusals(built, torch_cuda):
    w, h = 48, 32
    medium = g.make_medium()
    ctx = Context(0)
    _refused(ctx, "no committed ray set")
    ctx.upload_rays(g.synth_rays(w, h, seed=3))
    _refused(ctx, "gvpm_set_medium first")
    ctx.set_medium(medium)
    ctx.ray_staging(w * h)   # a ray set being staged is not committed
    _refused(ctx, "no committed ray set")
    ctx.upload_rays(g.synth_rays(w, h, seed=3))
    _refused(ctx, "nbCameraSamples must be positive", nb_camera_samples=0)
    _refused(ctx, "nbCameraSamples must be positive", nb_camera_samples=-3)
    _refused(ctx, "epsilon must be > 0", epsilon=0.0)
    _refused(ctx, "epsilon must be > 0", epsilon=float("nan"))
    for r in (None, 0.0, -1.0, float("inf"), float("nan")):
        _refused(ctx, "radius must be finite and > 0", radius=r)
    _refused(ctx, "exceeds 0xfffffff0", nb_camera_samples=0xfffffff0 // (w * h) + 1)
    rad = np.full(w * h, 0.02, dtype=F32)
    rays = ctx.download_rays()
    drawing = np.flatnonzero(rays.edge_len > F32(4e-4))
    for bad in (-0.01, float("nan"), float("inf")):
        r = rad.copy()
        r[drawing[7]] = bad
        _refused(ctx, "per-ray radius must be finite and >= 0", radius=None, radius_per_ray=_device_array(torch_cuda, r))
    # a bad radius of a ray that draws nothing is never read
    r = rad.copy()
    r[np.flatnonzero(rays.edge_len <= F32(4e-4))] = -1.0
    assert ctx.generate_vpm_samples(8, seed=1, radius_per_ray=_device_array(torch_cuda, r)) > 0
    assert ctx.generate_vpm_samples(8, seed=1, radius_per_ray=_device_array(torch_cuda, rad)) > 0
    ctx.close()


def test_samples_drawn_for_another_ray_set_are_refused(built):
    c = _vpm_case()
    ctx = H.gpu_context(c)
    ctx.generate_vpm_samples(c.nb, seed=1, radius=c.radius)
    ctx.gather_vpm(c.nb)
    ctx.generate_rays(g.box_scene_default(), g.pinhole_camera(c.w, c.h), 9)
    stale = "drawn for another ray set: draw them again"
    with pytest.raises(GvpmError, match=stale):
        ctx.gather_vpm(c.nb)
    with pytest.raises(GvpmError, match=stale):
        ctx.gather_vpm_device(c.nb)
    with pytest.raises(GvpmError, match=stale):
        ctx.dump_neighbours_vpm(c.nb)
    ctx.upload_rays(c.rays)   # the same rays again: still a new ray set
    with pytest.raises(GvpmError, match=stale):
        ctx.gather_vpm(c.nb)
    ctx.generate_vpm_samples(c.nb, seed=1, radius=c.radius)
    ctx.gather_vpm(c.nb)
    # uploaded samples keep their behaviour: a new ray set of the same size does not refuse them
    ctx.upload_vpm_samples(ctx.download_vpm_samples())
    ctx.upload_rays(c.rays)
    ctx.gather_vpm(c.nb)
    ctx.close()
