"""CPU tests: the C-ABI library loads and exports every symbol include/gvpm_b200.h declares, fails
loudly without a device, host-side logic (radius reduction, tile sharding incl. a world-size-2 gloo
run).  No compute calls here."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from gvpm_b200 import _native
    return _native.load_lib()


def test_header_symbols_exported(lib):
    from gvpm_b200 import _native
    hdr = open(os.path.join(ROOT, "include", "gvpm_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(gvpm_[a-z_0-9]+)\s*\(", hdr))
    assert len(declared) >= 20
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/gvpm_b200.h but not exported"
    assert declared == set(_native.ABI_SYMBOLS), declared ^ set(_native.ABI_SYMBOLS)
    assert lib.gvpm_abi_version() == 1


def test_struct_sizes_match_header(lib):
    from gvpm_b200 import _native as N
    assert C.sizeof(N.Medium) == 36
    assert C.sizeof(N.Config) == 64
    assert C.sizeof(N.PhotonSoA) == 13 * 8
    assert C.sizeof(N.RaySoA) == 16 * 8


def test_no_device_fails_loudly(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from gvpm_b200.api import Context, GvpmError
    with pytest.raises(GvpmError, match="no CUDA device|CPU fallback"):
        Context(0)


def test_product_never_imports_oracle():
    """The product package must not reference oracle/ (only tests, smoke and bench may)."""
    pkg = os.path.join(ROOT, "gvpm_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "oracle" not in txt.lower(), f"{os.path.join(dp, f)} mentions the oracle"


def _host():
    import __graft_entry__ as ge
    ge.build()
    h = C.CDLL(os.path.join(ROOT, "gvpm_b200", "host", "libgvpm_host.so"))
    return h


class HostParams(C.Structure):
    _fields_ = [("maxDepth", C.c_int), ("minDepth", C.c_int), ("alpha", C.c_double),
                ("initialScaleVolume", C.c_double), ("volTechnique", C.c_int),
                ("lightingInteractionMode", C.c_int), ("useMIS", C.c_int), ("useShiftNull", C.c_int),
                ("pathSet", C.c_int), ("powerHeuristic", C.c_int), ("use3DKernelReduction", C.c_int),
                ("forceAPA", C.c_char * 8)]


def host_params(**kw):
    p = HostParams(maxDepth=12, minDepth=0, alpha=0.7, initialScaleVolume=1.0, volTechnique=1,
                   lightingInteractionMode=(1 << 2) | (1 << 4), useMIS=1, useShiftNull=1, pathSet=1,
                   powerHeuristic=0, use3DKernelReduction=0, forceAPA=b"")
    for k, v in kw.items():
        setattr(p, k, v)
    return p


@pytest.mark.parametrize("tech,force,expo", [(1, b"", 1 / 3), (0, b"", 1 / 2), (1, b"1D", 1.0), (0, b"3D", 1 / 3),
                                             (3, b"", 1 / 3), (2, b"", 1 / 3), (5, b"", 1.0), (4, b"", 1.0)])
def test_scale_volume_apa_schedule(tech, force, expo):
    """r_{i+1} = r_i * ((i-1+alpha)/i)^(1/d)  (gvpm.cpp:181-215), d by kernel dimension / forceAPA."""
    h = _host()
    h.gvpm_host_scale_apa.argtypes = [C.POINTER(C.c_double), C.c_int, C.POINTER(HostParams), C.c_char_p, C.c_size_t]
    p = host_params(volTechnique=tech, forceAPA=force, alpha=0.7, initialScaleVolume=0.1)
    s = C.c_double(0.1)
    want = 0.1
    err = C.create_string_buffer(256)
    for it in range(1, 30):
        assert h.gvpm_host_scale_apa(C.byref(s), it, C.byref(p), err, 256) == 0
        want *= ((it - 1 + 0.7) / it) ** expo
        assert abs(s.value - want) < 1e-15 * 10
    bad = host_params(forceAPA=b"7D")
    assert h.gvpm_host_scale_apa(C.byref(s), 1, C.byref(bad), err, 256) == -1
    assert b"No Force APA" in err.value


class HostExtra(C.Structure):
    _fields_ = [("rrDepth", C.c_int), ("photonCount", C.c_int), ("volumePhotonCount", C.c_int), ("maxPasses", C.c_int),
                ("dumpIteration", C.c_int), ("reconstructL1", C.c_int), ("reconstructL2", C.c_int),
                ("reconstructAlpha", C.c_double), ("useManifold", C.c_int), ("noMediumShift", C.c_int),
                ("convertLong", C.c_int), ("newShiftBeam", C.c_int), ("deterministic", C.c_int),
                ("nbCameraSamples", C.c_int), ("minCameraDepth", C.c_int), ("maxCameraDepth", C.c_int),
                ("cameraSphere", C.c_double)]


def _load_config(text):
    h = _host()
    p, x = HostParams(), HostExtra()
    err = C.create_string_buffer(512)
    rc = h.gvpm_host_config_load(text.encode(), C.byref(p), C.byref(x), err, 512)
    return rc, p, x, err.value.decode()


def test_gpm_config_load_defaults_and_paper_preset():
    """GPMConfig::load (gvpm_struct.h:181-333): XML parameter names, defaults, string parsing."""
    rc, p, x, err = _load_config("")
    assert rc == 0, err
    # plugin defaults: volTechnique "distance" (point photons), all2all, MIS by area, no mixed shift, pathSet on
    assert (p.maxDepth, p.minDepth, p.volTechnique, p.useMIS, p.useShiftNull, p.pathSet, p.powerHeuristic) == (-1, 0, 2, 1, 0, 1, 0)
    assert p.lightingInteractionMode == 0b11110 and p.alpha == pytest.approx(0.7) and p.initialScaleVolume == 1.0
    assert (x.rrDepth, x.photonCount, x.volumePhotonCount, x.maxPasses, x.nbCameraSamples) == (12, 250000, 250000, -1, 40)
    assert (x.reconstructL1, x.reconstructL2, x.newShiftBeam) == (0, 1, 0) and x.reconstructAlpha == pytest.approx(0.2)
    # the paper's generator script (scripts/scene/generatorGVPM.py:44-76): G-BRE 3D, mixed shift, volume only
    rc, p, x, err = _load_config("volTechnique=bre\nuseShiftNull=true\nuseMIS=Area\nmaxDepth=12\nrrDepth=1\n"
                                 "interactionMode=all2media\ninitialScaleVolume=0.1\nvolumePhotonCount=10000000")
    assert rc == 0, err
    assert (p.volTechnique, p.useShiftNull, p.useMIS, p.maxDepth, x.rrDepth) == (1, 1, 1, 12, 1)
    assert p.lightingInteractionMode == (1 << 2) | (1 << 4) and p.initialScaleVolume == pytest.approx(0.1)
    assert x.photonCount == 0 and x.volumePhotonCount == 10000000      # surface photons forced to 0 (:304-306)
    for name, tech in (("bre2d", 0), ("bre3d", 1), ("distance", 2), ("beam3d", 3), ("beam3d_optimized", 3),
                       ("plane0d", 4), ("beam", 5), ("beam1d", 5)):
        rc, p, x, err = _load_config(f"volTechnique={name}")
        assert rc == 0 and p.volTechnique == tech, (name, err)
        assert x.newShiftBeam == (1 if tech == 5 else 0)               # gvpm.cpp:96-98
    rc, p, x, err = _load_config("lightingInteractionMode=media2media\ninteractionMode=all2surf")
    assert rc == 0 and p.lightingInteractionMode == 1 << 4               # the first key wins (:291-294)


@pytest.mark.parametrize("text,msg", [
    ("maxDepth=1", "Maximum depth must be set"),
    ("maxPasses=0", "Maximum number of passes"),
    ("useMIS=balance", "useMIS: need to be 'none' or 'area'"),
    ("relaxME=0.5", "relaxME options need to be 0 or 1."),
    ("volTechnique=bre2d\nuseShiftNull=true", "Not possible to shift null without using 3D kernel"),
    ("volTechnique=raymarching", "Unknow vol technique"),
    ("volTechnique=beam3d_egsr", "Not supported kernel type"),
    ("interactionMode=some2all", "Invalid media interaction mode"),
    ("deterministic=true", "pathSet and deterministic"),
    ("minCameraDepth=-1", "minCamera depth"),
    ("bounceRoughness=0", "Bad roughtness constant"),
    ("pathSet=maybe", "wrong type"),
    ("maxDepth=twelve", "wrong type"),
])
def test_gpm_config_load_errors(text, msg):
    """SLog(EError, ...) of GPMConfig::load becomes an exception with the reference's message."""
    rc, _, _, err = _load_config(text)
    assert rc == -1 and msg in err, (text, err)


class SppmHostParams(C.Structure):
    _fields_ = [("maxDepth", C.c_int), ("minDepth", C.c_int), ("alpha", C.c_double), ("initialScaleVolume", C.c_double),
                ("volTechnique", C.c_int), ("rngSeed", C.c_uint), ("forceAPA", C.c_char * 8)]


@pytest.mark.parametrize("tech,force,expo", [(1, b"", 1 / 3), (0, b"", 1 / 2), (2, b"", 1.0), (3, b"", 1 / 3),
                                             (5, b"", 1 / 3), (2, b"3D", 1 / 3)])
def test_sppm_scale_volume_apa_schedule(tech, force, expo):
    """sppm.cpp:255-290: 3-D kernels (bre3d, the three 3-D beam techniques) shrink by the cube root, bre2d by the
    square root, beam1d linearly; forceAPA overrides."""
    h = _host()
    h.gvpm_host_sppm_scale_apa.argtypes = [C.POINTER(C.c_double), C.c_int, C.POINTER(SppmHostParams), C.c_char_p, C.c_size_t]
    p = SppmHostParams(maxDepth=-1, minDepth=0, alpha=0.7, initialScaleVolume=0.3, volTechnique=tech, rngSeed=0, forceAPA=force)
    s, want = C.c_double(0.3), 0.3
    err = C.create_string_buffer(256)
    for it in range(1, 20):
        assert h.gvpm_host_sppm_scale_apa(C.byref(s), it, C.byref(p), err, 256) == 0
        want *= ((it - 1 + 0.7) / it) ** expo
        assert abs(s.value - want) < 1e-14
    p.forceAPA = b"9D"
    assert h.gvpm_host_sppm_scale_apa(C.byref(s), 1, C.byref(p), err, 256) == -1 and b"No Force APA" in err.value


class SppmHostExtra(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("photonCount", "volumePhotonCount", "rrDepth", "maxPasses", "dumpIteration",
                                       "nbCameraSamples", "surfaceRendering", "volumeRendering", "convertLong",
                                       "deterministic", "minCameraDepth", "maxCameraDepth")] + [("cameraSphere", C.c_double)]


def _load_sppm(text):
    h = _host()
    p, x = SppmHostParams(), SppmHostExtra()
    err = C.create_string_buffer(512)
    rc = h.gvpm_host_sppm_config_load(text.encode(), C.byref(p), C.byref(x), err, 512)
    return rc, p, x, err.value.decode()


def test_sppm_config_load():
    """SPPMIntegrator's constructor (sppm.cpp:163-241): names, defaults, technique strings, error messages."""
    rc, p, x, err = _load_sppm("volTechnique=beam3d_egsr\nmaxDepth=8\ninitialScaleVolume=0.5\nforceAPA=2D")
    assert rc == 0, err
    assert (p.volTechnique, p.maxDepth, p.minDepth, p.forceAPA) == (4, 8, 0, b"2D") and p.initialScaleVolume == 0.5
    assert (x.rrDepth, x.photonCount, x.volumePhotonCount, x.nbCameraSamples, x.surfaceRendering) == (3, 250000, 250000, 40, 1)
    for name, tech in (("bre2d", 0), ("bre", 1), ("bre3d", 1), ("beam", 2), ("beam1d", 2), ("beam3d_naive", 3),
                       ("beam3d_egsr", 4), ("beam3d", 5), ("beam3d_optimized", 5), ("distance", 6), ("plane0d", 7)):
        rc, p, _, err = _load_sppm(f"volTechnique={name}")
        assert rc == 0 and p.volTechnique == tech, (name, err)
    for text, msg in (("", "Unknow vol technique: raymarching"),            # the default is not a known name (:208-209)
                      ("volTechnique=bre\nmaxDepth=0", "Maximum depth must be set"),
                      ("volTechnique=bre\nmaxPasses=-3", "Maximum number of Passes"),
                      ("volTechnique=bre\nmaxRenderingTime=60", "Max pass and time is incompatible!"),
                      ("volTechnique=bre\nvolumePhotonCount=0", "No volume photons/beams"),
                      ("volTechnique=bre\nphotonCount=0", "No surface photons"),
                      ("volTechnique=bre\nminCameraDepth=-2", "minCamera depth")):
        rc, _, _, err = _load_sppm(text)
        assert rc == -1 and msg in err, (text, err)
    rc, _, _, err = _load_sppm("volTechnique=bre\nphotonCount=0\nsurfaceRendering=false")
    assert rc == 0, err


def test_tile_sharding_partitions_every_ray_once():
    from gvpm_b200 import shard
    w, h = 100, 70
    py, px = np.mgrid[0:h, 0:w]
    px, py = px.ravel(), py.ravel()
    for world in (1, 2, 4, 8):
        seen = np.zeros(px.size, dtype=int)
        sizes = []
        for r in range(world):
            idx = shard.local_indices(px, py, w, world, r)
            seen[idx] += 1
            sizes.append(len(idx))
        assert (seen == 1).all()
        assert max(sizes) - min(sizes) <= 32 * 32 * 2
    parts = [np.arange(27, dtype=np.float32)[None, :] + shard.local_indices(px, py, w, 2, r)[:, None] for r in (0, 1)]
    full = shard.assemble(parts, [shard.local_indices(px, py, w, 2, r) for r in (0, 1)], px.size)
    np.testing.assert_array_equal(full[:, 0], np.arange(px.size))
    img = shard.to_image(full, px, py, w, h)
    assert img.shape == (h, w, 27) and img[3, 5, 0] == 3 * w + 5


def test_band_sharding_partitions_every_ray_once_in_compact_bands():
    from gvpm_b200 import shard
    w, h = 1920, 1080
    py, px = np.mgrid[0:h:8, 0:w:8]          # one ray per 8x8 pixels is enough to see every block
    px, py = px.ravel(), py.ravel()
    for world in (1, 2, 4, 8):
        for cycles in (1, 2, 4):
            owner = shard.band_owner(px, py, w, h, world, cycles)
            sizes = np.bincount(owner, minlength=world)
            assert sizes.sum() == px.size and sizes.min() > 0
            # equal block counts up to one block per run (the last block row / column is partial)
            assert sizes.max() - sizes.min() <= (cycles + 1) * 16 + 0.03 * sizes.mean()
            seen = np.zeros(px.size, dtype=int)
            for r in range(world):
                idx = shard.band_indices(px, py, w, h, world, r, cycles)
                seen[idx] += 1
                # a rank's rays lie in at most cycles + 1 vertical bands: few distinct block columns
                cols = np.unique(px[idx] // 32)
                assert len(cols) <= (60 // (cycles * world) + 2) * cycles
            assert (seen == 1).all()
    # degenerate deal: one run per block = round robin over the column-major block list
    o = shard.band_owner(px, py, w, h, 2, cycles=60 * 34)
    assert set(np.unique(o)) == {0, 1}


def test_weighted_bands_balance_cost_and_still_partition():
    """band_owner_weighted: every ray owned once, contiguous column-major runs, costs per rank within a few per cent of
    each other for a centre-weighted density (the uniform deal is far off), identical to band_owner for uniform costs"""
    from gvpm_b200 import shard
    w, h = 1920, 1080
    py, px = np.mgrid[0:h:8, 0:w:8]
    px, py = px.ravel(), py.ravel()
    tiles_x, tiles_y = 60, 34
    bx = np.repeat(np.arange(tiles_x), tiles_y)
    by = np.tile(np.arange(tiles_y), tiles_x)
    cost = 1.0 + 8.0 * np.exp(-((bx - 30) / 9.0) ** 2 - ((by - 17) / 7.0) ** 2)     # bright centre
    t = shard.block_index(px, py, h)
    ray_cost = cost[t]
    for world in (2, 4, 8):
        for cycles in (1, 2):
            o = shard.band_owner_weighted(px, py, w, h, world, cost, cycles)
            assert o.min() == 0 and o.max() == world - 1
            per = np.array([ray_cost[o == r].sum() for r in range(world)])
            assert per.max() / per.mean() < 1.05, (world, cycles, per / per.mean())
            uni = shard.band_owner(px, py, w, h, world, cycles)
            per_u = np.array([ray_cost[uni == r].sum() for r in range(world)])
            assert per_u.max() / per_u.mean() >= per.max() / per.mean()
            # runs are contiguous in the column-major block order: a rank owns at most `cycles` intervals of it
            for r in range(world):
                blocks = np.unique(t[o == r])
                assert (np.diff(blocks) > 1).sum() <= cycles - 1 + 0
    np.testing.assert_array_equal(shard.band_owner_weighted(px, py, w, h, 8, np.ones(tiles_x * tiles_y), 2),
                                  shard.band_owner(px, py, w, h, 8, 2))


GLOO_WORKER = r"""
import os, sys
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from gvpm_b200 import shard
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
w, h = 96, 80
py, px = np.mgrid[0:h, 0:w]; px, py = px.ravel(), py.ravel()
# replicated "photon set": broadcast from rank 0 like the iteration's photons
photons = torch.arange(1000, dtype=torch.float32) if rank == 0 else torch.zeros(1000)
dist.broadcast(photons, src=0)
assert float(photons.sum()) == 999 * 1000 / 2
mode = sys.argv[2] if len(sys.argv) > 2 else "tile"
def indices(r):
    if mode == "weighted":
        return np.nonzero(owner_w == r)[0]
    return shard.band_indices(px, py, w, h, world, r, 2) if mode == "band" else shard.local_indices(px, py, w, world, r)
if mode == "weighted":
    # bench.py rebalance_bands: every rank measures the cost of its equal-size bands (here: a centre-weighted density),
    # the per-block costs are summed over the ranks, and every rank derives the SAME cost-balanced partition from them
    t = shard.block_index(px, py, h)
    mine0 = shard.band_indices(px, py, w, h, world, rank, 2)
    dens = 1.0 + 6.0 * np.exp(-((px - w / 2) / 20.0) ** 2 - ((py - h / 2) / 15.0) ** 2)
    n_tiles = ((w + 31) // 32) * ((h + 31) // 32)
    cost = torch.from_numpy(np.bincount(t[mine0], weights=dens[mine0], minlength=n_tiles))
    dist.all_reduce(cost)
    owner_w = shard.band_owner_weighted(px, py, w, h, world, cost.numpy(), 2)
    sizes = torch.tensor([float(dens[owner_w == r].sum()) for r in range(world)], dtype=torch.float64)
    other = sizes.clone(); dist.broadcast(other, src=0)
    assert torch.equal(sizes, other)                       # identical partition on every rank
idx = indices(rank)
n_pad = torch.tensor([len(idx)]); dist.all_reduce(n_pad, op=dist.ReduceOp.MAX); n_pad = int(n_pad)
out = torch.zeros(n_pad, 27)
out[:len(idx)] = torch.from_numpy((px[idx] * 1000 + py[idx]).astype(np.float32))[:, None] + torch.arange(27.0)
gathered = [torch.empty_like(out) for _ in range(world)] if rank == 0 else None
dist.gather(out, gathered, dst=0)
if rank == 0:
    lists = [indices(r) for r in range(world)]
    full = shard.assemble([g.numpy() for g in gathered], lists, px.size)
    want = (px * 1000 + py).astype(np.float32)[:, None] + np.arange(27, dtype=np.float32)
    assert np.array_equal(full, want)
    print("GLOO_OK")
dist.destroy_process_group()
"""


@pytest.mark.parametrize("mode", ["tile", "band", "weighted"])
def test_sharded_gather_world2_gloo(tmp_path, mode):
    """The N > 1 plumbing of bench.py (broadcast photons, gather per-rank results of unequal size, reassemble) on
    2 CPU ranks over gloo, for the round-robin, the column-band and the cost-balanced column-band partition (costs
    all-reduced over the ranks as in bench.py rebalance_bands)."""
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", {"tile": "29533", "band": "29534", "weighted": "29535"}[mode], str(script), ROOT, mode]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert res.returncode == 0, res.stderr[-2000:]
    assert "GLOO_OK" in res.stdout


@pytest.mark.parametrize("arm", ["code", "port"])
def test_bench_reference_arm_contract_on_cpu(arm):
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours) needs no GPU: one JSON line with the
    contract's keys, e2e = value with zero copy bytes.  "code": the reference's own compiled G-BRE path
    (oracle/_ref/libgvpm_functor_ref.so, kind "reference"; it also reports the restated port on the same rays and their
    agreement); "port": the oracle restatement (what runs where that library is absent)."""
    import json
    from oracle import functor_binding as fb
    if arm == "code" and not fb.have_ref():
        pytest.skip("prebuilt reference library absent")
    env = dict(os.environ, GVPM_REFERENCE_ARM=arm)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1",
                        "--steps", "1", "--warmup", "1", "--cpu-seconds", "1"], capture_output=True, text=True, timeout=300,
                       env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "rays/s" and line["higher_is_better"] is True
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["value"] > 0 and line["vs_baseline"] is None and "workload" in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == ("reference" if arm == "code" else "port")
    assert cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    if arm == "code":
        chk = cb["restated_port_on_same_rays"]
        assert chk["max_rel_diff"] < 2e-6 and chk["port_value"] > 0 and chk["reference_value"] > 0
    else:
        assert cb["reference_code_not_timed"] == "GVPM_REFERENCE_ARM=port"
    assert line["e2e"] == {"value": line["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@pytest.mark.parametrize("workload,photons", [("cfg2", 20000), ("cfg3", 3000), ("cfg4", 1500)])
def test_bench_technique_reference_arm_runs_the_reference_code(workload, photons):
    """The reference arms of the other techniques time the reference's own structures + functors too (kind "reference")."""
    import json
    from oracle import functor_binding as fb
    if not fb.have_ref():
        pytest.skip("prebuilt reference library absent")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload,
                        "--photons", str(photons), "--steps", "1", "--warmup", "1", "--cpu-seconds", "1"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    cb = line["cpu_baseline"]
    assert line["impl"] == "reference" and cb["kind"] == "reference" and cb["value"] == line["value"] > 0
    assert "own compiled code" in cb["sample"]


def test_bench_poisson_reference_arm_on_cpu():
    """`bench.py --workload poisson720 --impl reference`: the reference's own poisson::Solver (OpenMP backend, compiled from
    /root/reference into oracle/_ref) on the host cores, one JSON line with the contract's keys."""
    import json
    from oracle import poisson_ref as pr
    if not pr.available():
        pytest.skip("prebuilt reference solver absent")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "poisson720",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "pixels/s" and line["cpu_baseline"]["kind"] == "reference"
    assert line["value"] > 0 and line["config"]["pixels"] == 1280 * 720


def test_bench_rejects_arguments_it_cannot_honour():
    """No timed step, or outputs of a path that has none on the device: refused before anything runs."""
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                           timeout=120)
        assert p.returncode == 2 and "error:" in p.stderr, (extra, p.stderr[-2000:])


def _bench_dump(tmp_path, *args):
    """run bench.py with --dump-outputs on one GPU -> (its JSON line, the dumped arrays by name)"""
    import json
    d = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                        "--dump-outputs", str(d)] + list(args), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    z = {f.stem: np.load(f) for f in d.glob("*.npy")}
    assert all(a.dtype in (np.float32, np.float64) for a in z.values())
    assert sum(a.nbytes for a in z.values()) <= 64 << 20
    return line, z


def _check_gather_dump(z, rays, out, mvol=None):
    """the dumped rows are the gather output of the rays they name (index and pixel), all rays where there are few"""
    assert sorted(z) == sorted(["gather_out", "ray_index", "ray_pixel"] + (["gather_mvol"] if mvol is not None else []))
    np.testing.assert_array_equal(z["ray_index"], np.arange(rays.n))
    np.testing.assert_array_equal(z["ray_pixel"], np.stack([rays.px, rays.py], axis=1))
    assert z["gather_out"].dtype == np.float32 and np.count_nonzero(z["gather_out"][:, :3]) > rays.n // 10
    import gvpm_testlib as H
    H.assert_radiance_close(z["gather_out"], out, 1e-4, "bench dump")
    if mvol is not None:
        np.testing.assert_array_equal(z["gather_mvol"], mvol)


@pytest.mark.gpu
def test_bench_dump_outputs_of_the_point_gather(tmp_path, built):
    """`bench.py --dump-outputs DIR` (cfg1, resident G-BRE path): the dump equals the same gather run directly through
    the C ABI on the bench's seeded inputs, row by row (27 floats per ray, float32), with each ray's index and pixel."""
    import types
    import bench
    from gvpm_b200.api import Context
    _, z = _bench_dump(tmp_path, "--workload", "cfg1")
    inp = bench.make_inputs(types.SimpleNamespace(workload="cfg1", photons=None, scale=None, impl="ours"), 0, 1, pin=False)
    ctx = Context(0)
    ctx.set_medium(inp["medium"])
    ctx.set_config(inp["cfg"])
    ctx.set_occluders(inp["tri"])
    ctx.upload_photons(inp["photons"])
    ctx.upload_rays(inp["rays"])
    ctx.build_points_for_rays(inp["radius"], want_kept=False)
    out, _ = ctx.gather_bre(counts=False)
    ctx.close()
    _check_gather_dump(z, inp["rays"], out)


@pytest.mark.gpu
def test_bench_dump_outputs_of_the_vpm_gather(tmp_path, built):
    """The technique path (cfg2, G-VPM, device pointers of the last gather): radiance and MVol, the per-ray photon count
    that drives the radius update, equal the same gather run directly through the C ABI on the bench's inputs."""
    import types
    import bench
    from gvpm_b200.api import Context
    _, z = _bench_dump(tmp_path, "--workload", "cfg2", "--photons", "20000")
    d = bench.technique_inputs(types.SimpleNamespace(workload="cfg2", photons=20000, scale=None), 0, 1)
    ctx = Context(0)
    ctx.set_medium(d["medium"])
    ctx.set_config(d["cfg"])
    ctx.set_occluders(d["tri"])
    ctx.upload_photons(d["photons"])
    ctx.build_points(d["radius"])
    ctx.upload_rays(d["rays"])
    ctx.upload_vpm_samples(d["samples"])
    out, mvol, _ = ctx.gather_vpm(d["nb"], sample_counts=False)
    ctx.close()
    assert mvol.max() > 0
    _check_gather_dump(z, d["rays"], out, mvol)


@pytest.mark.gpu
def test_bench_dump_outputs_of_the_poisson_solve(tmp_path, built):
    """The Poisson path (poisson720): the dumped reconstruction is the solve of the bench's seeded image set."""
    import importlib.util
    from gvpm_b200.api import Context
    line, z = _bench_dump(tmp_path, "--workload", "poisson720")
    assert line["warmup"] == 3 and sorted(z) == ["reconstruction"]
    spec = importlib.util.spec_from_file_location("make_poisson_golden", os.path.join(ROOT, "tests", "golden", "make_poisson_golden.py"))
    G = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(G)
    _, tp, dx, dy, direct = G.images(720, 1280, 11)
    ctx = Context(0)
    want = ctx.poisson_solve(tp, dx, dy, direct, preset="L2D")
    ctx.close()
    assert z["reconstruction"].shape == (720, 1280, 3) and z["reconstruction"].dtype == np.float32
    np.testing.assert_allclose(z["reconstruction"], want, rtol=0, atol=1e-6 * np.abs(want).max())
