"""Photon dispatch between ranks (gvpm_dispatch_*, csrc/dispatch.cu; SURVEY.md §8e): every rank classifies its slice of
the photon set against every receiver's perspective grid and writes the records a receiver can reach into that
receiver's inbox.  Here the "ranks" are contexts of one process on one GPU (wired directly instead of through CUDA IPC;
the kernels, the control flags and the build over the inbox are the ones the multi-process bench runs): each rank's
gather over what it was sent must equal the CPU oracle's gather of that rank's rays against the WHOLE photon set -
bit-exact neighbour index sets, radiance within 1e-4 - while an inbox holds a fraction of the set."""
import numpy as np
import pytest

import gvpm_testlib as H
from gvpm_b200 import shard

pytestmark = pytest.mark.gpu


def _ranks(case, world, cycles, view_dir=None):
    from gvpm_b200.api import Context
    n = case.photons.n
    assert n % world == 0
    n_slice = n // world
    ctxs, rays = [], []
    for rank in range(world):
        idx = shard.band_indices(case.rays.px, case.rays.py, case.w, case.h, world, rank, cycles)
        r = case.rays.take(idx)
        ctx = Context(0)
        ctx.set_medium(case.medium)
        ctx.set_config(case.config)
        ctx.set_occluders(case.tri)
        if view_dir is not None:   # every rank projects on the same plane: photons are classified once (owner map)
            ctx.set_view_direction(view_dir)
        ctx.upload_rays(r)
        ctx.photon_staging(n)
        ctx.upload_photons_slice(case.photons.take(np.arange(rank * n_slice, (rank + 1) * n_slice)), n, rank * n_slice)
        ctxs.append(ctx)
        rays.append(r)
    blobs = [c.dispatch_export(world, n_slice) for c in ctxs]
    for rank, c in enumerate(ctxs):
        c.dispatch_connect(blobs, rank)
    return ctxs, rays, n_slice


def _oracle(case, rays):
    from oracle import binding as ob
    return ob.bre_gather(case.photons, rays, case.medium, case.config, case.tri, case.radius, mode="brute", neighbours=True)


@pytest.mark.parametrize("world,cycles,view_dir", [(2, 2, None), (4, 1, None), (4, 2, (0.0, 0.0, 1.0)), (8, 1, (0.05, -0.02, 1.0)),
                                                   (8, 1, (0.0, 0.0, 1.0))])
def test_dispatched_gather_equals_oracle(built, world, cycles, view_dir):
    case = H.make_case(n_photons=120000, w=256, h=64, scale=1.0)
    ctxs, rays, n_slice = _ranks(case, world, cycles, view_dir)
    n = case.photons.n
    received = 0
    for it in range(3):   # three iterations: both inboxes, and a reuse of the first one (release / free flags)
        b = it & 1
        for rank, c in enumerate(ctxs):   # every sender first: one host thread drives all ranks here
            c.dispatch_photons(b, n, rank * n_slice, n_slice, case.radius)
        for rank, c in enumerate(ctxs):
            kept = c.build_dispatched(b, case.radius, want_kept=True)
            assert c.accel_kind() == "frustum"
            out, counts = c.gather_bre()
            c.dispatch_release(b)
            if it != 2 and rank not in (0, world - 1):
                continue
            ref = _oracle(case, rays[rank])
            np.testing.assert_array_equal(counts, ref.counts)
            H.assert_radiance_close(out, ref.out, 1e-4, f"dispatched, rank {rank}/{world}, iteration {it}")
            offsets, idx = c.dump_neighbours_bre()
            np.testing.assert_array_equal(offsets, ref.offsets)
            np.testing.assert_array_equal(idx, ref.idx)
            got = c.dispatch_status(b)
            # the owner map of the shared-frame dispatch is a (dilated) superset of each receiver's own keep test
            assert (0.999 if view_dir is None else 0.8) * sum(got) <= kept <= sum(got) and all(g <= n_slice for g in got)
            assert kept >= len(np.unique(ref.idx & 0x7fffffff))
            if it == 2:
                received += kept
    # what the ranks received in one iteration: far less than `world` copies of the set (the all-gather exchange)
    assert received < n * min(world, 2.2 + 0.25 * world), (received, n)
    for c in ctxs:
        c.close()


def test_dispatch_needs_concurrent_rays_and_matching_sizes(built):
    from gvpm_b200.api import Context
    case = H.make_case(n_photons=4096, w=32, h=16, scale=2.0)
    ctx = Context(0)
    ctx.set_medium(case.medium)
    ctx.set_config(case.config)
    ctx.set_occluders(case.tri)
    with pytest.raises(RuntimeError):
        ctx.dispatch_export(2, 2048)          # no rays yet
    r = case.rays.take(np.arange(64))
    r.view("d")[:] = r.view("d")[0]   # parallel rays: their lines have no common point
    ctx.upload_rays(r)
    with pytest.raises(RuntimeError):
        ctx.dispatch_export(2, 2048)
    ctx.upload_rays(case.rays)
    blob = ctx.dispatch_export(1, 4096)
    ctx.dispatch_connect([blob], 0)
    ctx.photon_staging(case.photons.n)
    ctx.upload_photons(case.photons)
    with pytest.raises(RuntimeError):
        ctx.dispatch_photons(0, case.photons.n, 0, 8192, case.radius)   # slice beyond the set
    # one rank dispatching to itself: the plain frustum build, through the inbox
    ctx.dispatch_photons(0, case.photons.n, 0, case.photons.n, case.radius)
    ctx.build_dispatched(0, case.radius)
    out, counts = ctx.gather_bre()
    ref = _oracle(case, case.rays)
    np.testing.assert_array_equal(counts, ref.counts)
    H.assert_radiance_close(out, ref.out, 1e-4, "self dispatch")
    ctx.close()
