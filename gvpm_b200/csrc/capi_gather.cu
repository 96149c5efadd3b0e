// capi_gather.cu — G-BRE and sppm BRE gathers (pair list, asynchronous ring, pipelined host gather), G-VPM, and the
// pair-list growth and neighbour dump steps the primitive gathers share.
#include "capi_internal.cuh"

// growth policy of the pair list: room for the count that overflowed it, and some
static unsigned long long grown_pairs(unsigned long long total) { return total + total / 8 + 1024; }

int grid_incomplete(gvpm_ctx *ctx) {
  return fail(ctx, GVPM_ERR_INVALID,
              "the perspective grid is incomplete - a peer's photon dispatch never arrived or overflowed its region "
              "(gvpm_dispatch_status names which): the gather did not run.  Build again and gather again");
}

int gather_params(gvpm_ctx *ctx, GatherParams &P, bool built, const char *not_built) {
  if (!ctx->have_medium || !ctx->have_cfg) return fail(ctx, GVPM_ERR_INVALID, "medium/config not set");
  if (!built) return fail(ctx, GVPM_ERR_INVALID, not_built);
  if (!ctx->rays_loaded) return fail(ctx, GVPM_ERR_INVALID, "no rays uploaded");
  memset(&P, 0, sizeof(P));
  P.rays = ctx->rays.as<float4>();
  P.n_rays = ctx->n_rays;
  for (int i = 0; i < 3; ++i) {
    P.sigma_s[i] = ctx->medium.sigma_s[i];
    P.sigma_t[i] = ctx->medium.sigma_s[i] + ctx->medium.sigma_a[i];
  }
  P.phase_type = ctx->medium.phase_type;
  P.hg_g = ctx->medium.hg_g;
  P.sampling_weight = ctx->medium.sampling_weight;
  P.cfg = ctx->cfg;
  P.work_counter = ctx->work_counter.as<uint32_t>();
  return GVPM_OK;
}

int fill_params(gvpm_ctx *ctx, GatherParams &P, float *out_dev, uint32_t *counts_dev) {
  int rc = gather_params(ctx, P, ctx->built, "gvpm_build_points has not been called");
  if (rc) return rc;
  if (ctx->pruned && ctx->pruned_for_gen != ctx->rays_gen)
    return fail(ctx, GVPM_ERR_INVALID, "the hierarchy was built by gvpm_build_points_for_rays for another ray set: rebuild");
  P.tree = ctx->tree;
  if (ctx->accel == gvpm_ctx::ACCEL_FRUSTUM) {
    P.grid = ctx->grid;
    P.cell_start = ctx->cell_start.as<uint32_t>();
    P.build_ovf = ctx->build_ovf;
  }
  P.planes = ctx->planes.as<float4>();
  P.aos = ctx->records();
  P.orig = ctx->orig.as<uint32_t>();
  const float r = ctx->radius;
  P.radius = r;
  P.radius_sq = r * r;
  // Float kernelVol = (4.0/3.0)*M_PI*pow(r,3) evaluated in double (shift_volume_photon.cpp:707)
  if (ctx->cfg.kernel_3d)
    P.kernel_vol = (float)((4.0 / 3.0) * (double)GVPM_PI * std::pow((double)r, 3));
  else
    P.kernel_vol = (float)((double)GVPM_PI * std::pow((double)r, 2));
  P.bounds = ctx->bounds.as<float>();
  P.tri = ctx->tri.as<float>();
  P.tri_plane = ctx->tri_plane.as<float4>();
  P.tri_aux = ctx->tri_aux.as<float2>();
  P.n_tri = ctx->n_tri;
  P.out = out_dev;
  P.counts = counts_dev;
  P.pair_counter = (unsigned long long *)(ctx->work_counter.as<char>() + 8);
  P.ray_begin = 0;
  P.ray_end = ctx->n_rays;
  P.pairs = ctx->pairs.as<uint2>();
  P.pair_cap = ctx->pair_cap;
  // packets whose rays drift apart by more than this are traversed ray by ray (performance only)
  P.packet_spread_max = 0.f;  // derived in the kernel from the photon bounds
  return GVPM_OK;
}

int reserve_pairs(gvpm_ctx *ctx, size_t entries) {
  if (ctx->pair_cap >= entries) return GVPM_OK;
  cudaError_t e = ctx->pairs.reserve(entries * sizeof(uint2));
  ctx->pair_cap = ctx->pairs.cap / sizeof(uint2);   // 0 when the allocation failed: nothing is stored through a stale pointer
  if (e != cudaSuccess) return fail(ctx, GVPM_ERR_CUDA, std::string("pair list: ") + cudaGetErrorString(e));
  return GVPM_OK;
}

// One host sync per attempt.  `clear` resets what the traversal accumulates into; `traverse` launches it between
// ev[4] and ev[5] (gvpm_last_gather_detail times that span).  An overflowed list grows and the traversal runs again,
// `attempts` runs at most (0: no limit).  within_budget: the list grows only within half of the free device memory; if
// it may not, *total is left above the capacity and the caller splits the work.
int traverse_growing(gvpm_ctx *ctx, GatherParams &P, int attempts, const char *overflow_msg, bool within_budget,
                     const std::function<int()> &clear, const std::function<int()> &traverse, unsigned long long *total) {
  for (int attempt = 1;; ++attempt) {
    P.pairs = ctx->pairs.as<uint2>();
    P.pair_cap = ctx->pair_cap;
    int rc = clear();
    if (rc) return rc;
    CK(cudaEventRecord(ctx->ev[4], ctx->stream));
    rc = traverse();
    if (rc) return rc;
    CK(cudaEventRecord(ctx->ev[5], ctx->stream));
    ctx->split_timed = true;
    CK(cudaMemcpyAsync(ctx->pair_count_host, P.pair_counter, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *total = *ctx->pair_count_host;
    if (*total <= ctx->pair_cap) return GVPM_OK;
    if (attempt == attempts) return fail(ctx, GVPM_ERR_CUDA, overflow_msg);
    const unsigned long long want = grown_pairs(*total);
    if (within_budget) {
      size_t freeB = 0, totalB = 0;
      cudaMemGetInfo(&freeB, &totalB);
      if (want > (freeB / 2 + ctx->pairs.cap) / sizeof(uint2)) return GVPM_OK;
    }
    rc = reserve_pairs(ctx, want);
    if (rc) return rc;
  }
}

int copy_back(gvpm_ctx *ctx, float *out, size_t out_bytes, uint32_t *counts, size_t counts_bytes, bool wait) {
  if (out_bytes) CK(cudaMemcpyAsync(out, ctx->out.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (counts && counts_bytes) CK(cudaMemcpyAsync(counts, ctx->counts.p, counts_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (wait) CK(cudaStreamSynchronize(ctx->stream));
  return GVPM_OK;
}

int dump_neighbours(gvpm_ctx *ctx, size_t rows, uint64_t *offsets, uint32_t *idx, size_t cap, bool pair_list,
                    const std::function<int(uint32_t *counts)> &count, const std::function<int(uint64_t total)> &fill) {
  std::vector<uint32_t> counts(2 * rows + 2);
  int rc = count(counts.data());
  if (rc) return rc;
  uint64_t total = 0;
  for (size_t i = 0; i < rows; ++i) { offsets[i] = total; total += counts[2 * i]; }
  offsets[rows] = total;
  if (total > cap || (total && !idx)) return fail(ctx, GVPM_ERR_INVALID, "neighbour buffer too small");
  if (total == 0) return GVPM_OK;
  ctx->out_state = gvpm_ctx::OUT_NONE;   // the fill pass may leave other values in the gather output
  if (pair_list) {   // the gather fills a flat list of (row, index) pairs: bucket it by row
    CK(ctx->nbr_idx.reserve(total * sizeof(uint2)));
    rc = fill(total);
    if (rc) return rc;
    std::vector<uint2> flat(total);
    CK(cudaMemcpyAsync(flat.data(), ctx->nbr_idx.p, total * sizeof(uint2), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    std::vector<uint64_t> cursor(offsets, offsets + rows);
    for (const uint2 &p : flat) idx[cursor[p.x]++] = p.y;
  } else {           // the gather writes every row's entries from its offset on
    CK(ctx->nbr_offsets.reserve((rows + 1) * 8));
    CK(ctx->nbr_idx.reserve(total * 4));
    CK(cudaMemcpyAsync(ctx->nbr_offsets.p, offsets, (rows + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    rc = fill(total);
    if (rc) return rc;
    CK(cudaMemcpyAsync(idx, ctx->nbr_idx.p, total * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  // canonical order: ascending index; entries of one index (the naive beam technique lists a beam once per accepted
  // sub-beam) by their flag bit
  for (size_t i = 0; i < rows; ++i)
    std::sort(idx + offsets[i], idx + offsets[i + 1], [](uint32_t a, uint32_t b) {
      const uint32_t ai = a & 0x7fffffffu, bi = b & 0x7fffffffu;
      return ai != bi ? ai < bi : a < b;
    });
  return GVPM_OK;
}

// ---- G-BRE gather: traverse + shade without a host round trip in between ---------------------------------------------
// The shading kernel reads the pair count on the device, so a ray range is two back-to-back launches; the count is
// copied to a pinned slot behind them and looked at later (gather_finish / pending_poll).  If the pair list turns out to
// have overflowed, the range is run again the slow way (gather_range_sync: grow the list or split the range, one host
// sync per attempt).  The list is grow-only, so after the first iteration of a render this does not happen again.
static int enqueue_range(gvpm_ctx *ctx, GatherParams &P, uint32_t r0, uint32_t r1, unsigned long long *host_slot) {
  if (r1 <= r0) { *host_slot = 0; return GVPM_OK; }
  P.ray_begin = r0;
  P.ray_end = r1;
  P.pairs = ctx->pairs.as<uint2>();
  P.pair_cap = ctx->pair_cap;
  CK(cudaMemsetAsync(ctx->work_counter.p, 0, 16, ctx->stream));
  CK(cudaEventRecord(ctx->ev[4], ctx->stream));
  CK(launch_bre_traverse(P, false, ctx->sm_count, ctx->stream));
  CK(cudaEventRecord(ctx->ev[5], ctx->stream));
  ctx->split_timed = true;
  CK(launch_bre_shade(P, ~0ull, ctx->sm_count, ctx->stream));
  ctx->launches += 2;
  CK(cudaMemcpyAsync(host_slot, P.pair_counter, 8, cudaMemcpyDeviceToHost, ctx->stream));
  return GVPM_OK;
}

// the slow path.  Rows [r0, r1) of P.out are cleared first.
static int gather_range_sync(gvpm_ctx *ctx, GatherParams &P, uint32_t r0, uint32_t r1, int depth) {
  if (r1 <= r0) return GVPM_OK;
  P.ray_begin = r0;
  P.ray_end = r1;
  unsigned long long total = 0;
  int rc = traverse_growing(
      ctx, P, 0, nullptr, true,
      [&]() -> int {
        CK(cudaMemsetAsync(ctx->work_counter.p, 0, 16, ctx->stream));
        CK(cudaMemsetAsync(P.out + (size_t)r0 * GVPM_OUT_FLOATS, 0, (size_t)(r1 - r0) * GVPM_OUT_FLOATS * sizeof(float),
                           ctx->stream));
        return GVPM_OK;
      },
      [&]() -> int {
        CK(launch_bre_traverse(P, false, ctx->sm_count, ctx->stream));
        ctx->launches += 1;
        return GVPM_OK;
      },
      &total);
  if (rc) return rc;
  if (total <= ctx->pair_cap) {
    ctx->last_pairs += total;
    CK(launch_bre_shade(P, total, ctx->sm_count, ctx->stream));
    if (total) ctx->launches += 1;
    return GVPM_OK;
  }
  // the grown list would not fit in device memory: halve the range
  if (r1 - r0 <= 1 || depth > 40) return fail(ctx, GVPM_ERR_CUDA, "pair list does not fit in device memory");
  const uint32_t mid = r0 + (r1 - r0) / 2;
  rc = gather_range_sync(ctx, P, r0, mid, depth + 1);
  if (rc) return rc;
  return gather_range_sync(ctx, P, mid, r1, depth + 1);
}

// a gather over all rays whose pair list overflowed, run again the slow way
static int gather_rerun(gvpm_ctx *ctx, float *out_dev, uint32_t *counts_dev) {
  GatherParams P;
  int rc = fill_params(ctx, P, out_dev, counts_dev);
  if (rc) return rc;
  ctx->last_pairs = 0;
  rc = gather_range_sync(ctx, P, 0, ctx->n_rays, 0);
  if (rc) return rc;
  CK(cudaEventRecord(ctx->ev[3], ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GVPM_OK;
}

// Asynchronous gathers (gvpm_gather_bre_into / _device) in flight: their pair counts are looked at without blocking when
// the next call comes in, and for good at gvpm_sync, which re-runs the latest gather if its list overflowed and nothing
// it depends on has changed since.
int pending_check(gvpm_ctx *ctx, bool block) {
  while (ctx->ring_n > 0) {
    gvpm_ctx::AsyncGather &g = ctx->ring[ctx->ring_tail];
    if (!block) {
      cudaError_t q = cudaEventQuery(g.done);
      if (q == cudaErrorNotReady) break;
      if (q != cudaSuccess) return fail(ctx, GVPM_ERR_CUDA, std::string("cudaEventQuery: ") + cudaGetErrorString(q));
    } else {
      CK(cudaEventSynchronize(g.done));
    }
    const unsigned long long total = ctx->pair_count_host[8 + ctx->ring_tail];
    ctx->ring_tail = (ctx->ring_tail + 1) % gvpm_ctx::kRing;
    --ctx->ring_n;
    ctx->last_pairs = total;
    if (total <= g.cap) continue;
    if (total >= kBuildOverflow) return grid_incomplete(ctx);   // a peer's dispatch timed out or overflowed: nothing was gathered
    // overflow: make the list large enough for the next one
    cudaStreamSynchronize(ctx->stream);
    int rc = reserve_pairs(ctx, grown_pairs(total));
    if (rc) return rc;
    const bool latest = ctx->ring_n == 0 && g.gen == ctx->state_gen;
    if (!(block && latest))
      return fail(ctx, GVPM_ERR_INVALID,
                  "an asynchronous gather (gvpm_gather_bre_into / _device) overflowed its pair list and its inputs have "
                  "been replaced since: its results are incomplete.  Call gvpm_sync after such a gather before the next "
                  "upload / build / gather (the list has been enlarged)");
    rc = gather_rerun(ctx, g.out, g.counts);   // same photons, rays and output buffers
    if (rc) return rc;
  }
  return GVPM_OK;
}

static int gather_common(gvpm_ctx *ctx, float *out_dev, uint32_t *counts_dev, unsigned long long *host_slot) {
  GatherParams P;
  int rc = fill_params(ctx, P, out_dev, counts_dev);
  if (rc) return rc;
  CK(cudaEventRecord(ctx->ev[2], ctx->stream));
  const size_t n = ctx->n_rays;
  *host_slot = 0;
  if (n) {
    if (ctx->pair_cap == 0) {
      rc = reserve_pairs(ctx, std::max<size_t>(1u << 20, 16 * n));
      if (rc) return rc;
      P.pairs = ctx->pairs.as<uint2>();
      P.pair_cap = ctx->pair_cap;
    }
    CK(cudaMemsetAsync(out_dev, 0, n * GVPM_OUT_FLOATS * sizeof(float), ctx->stream));
    rc = enqueue_range(ctx, P, 0, (uint32_t)n, host_slot);
    if (rc) return rc;
  }
  CK(cudaEventRecord(ctx->ev[3], ctx->stream));
  ctx->timed_gather = true;
  if (out_dev == ctx->out.as<float>()) out_written(ctx);
  else ctx->out_state = gvpm_ctx::OUT_ELSEWHERE;
  return GVPM_OK;
}

// blocking tail of a gather whose results the caller reads right away: wait, check the pair count, re-run on overflow.
static int gather_finish(gvpm_ctx *ctx, float *out_dev, uint32_t *counts_dev, const unsigned long long *host_slot,
                         bool *redone) {
  CK(cudaStreamSynchronize(ctx->stream));
  if (redone) *redone = false;
  const unsigned long long total = *host_slot;
  ctx->last_pairs = total;
  if (total <= ctx->pair_cap) return GVPM_OK;
  if (total >= kBuildOverflow) return grid_incomplete(ctx);
  int rc = reserve_pairs(ctx, grown_pairs(total));
  if (rc) return rc;
  rc = gather_rerun(ctx, out_dev, counts_dev);
  if (rc) return rc;
  if (redone) *redone = true;
  return GVPM_OK;
}

// asynchronous variant: the count goes to a ring slot that pending_check looks at later
static int gather_async(gvpm_ctx *ctx, float *out_dev, uint32_t *counts_dev) {
  int rc = pending_check(ctx, false);
  if (rc) return rc;
  if (ctx->ring_n == gvpm_ctx::kRing) {       // ring full: wait for the oldest
    gvpm_ctx::AsyncGather &g = ctx->ring[ctx->ring_tail];
    CK(cudaEventSynchronize(g.done));
    rc = pending_check(ctx, false);
    if (rc) return rc;
  }
  const int slot = (ctx->ring_tail + ctx->ring_n) % gvpm_ctx::kRing;
  gvpm_ctx::AsyncGather &g = ctx->ring[slot];
  rc = gather_common(ctx, out_dev, counts_dev, ctx->pair_count_host + 8 + slot);
  if (rc) return rc;
  g.gen = ctx->state_gen;
  g.out = out_dev;
  g.counts = counts_dev;
  g.cap = ctx->pair_cap;
  CK(cudaEventRecord(g.done, ctx->stream));
  ++ctx->ring_n;
  return GVPM_OK;
}

// ---- G-VPM ----------------------------------------------------------------------------------------------------------
static int vpm_params(gvpm_ctx *ctx, GatherParams &P, int nb_camera_samples) {
  if (ctx->built && ctx->accel == gvpm_ctx::ACCEL_FRUSTUM) {
    // the range queries walk the box hierarchy: build it (over the photons the rays can reach) in place of the grid
    int rcb = build_pruned_bvh(ctx, ctx->radius, nullptr);
    if (rcb) return rcb;
  }
  int rc = fill_params(ctx, P, ctx->out.as<float>(), nullptr);
  if (rc) return rc;
  if (!ctx->samples_loaded) return fail(ctx, GVPM_ERR_INVALID, "no VPM samples uploaded");
  if (ctx->samples_drawn && ctx->samples_rays_gen != ctx->rays_gen)
    return fail(ctx, GVPM_ERR_INVALID, "VPM samples were drawn for another ray set: draw them again");
  if (nb_camera_samples <= 0) return fail(ctx, GVPM_ERR_INVALID, "nbCameraSamples must be positive");
  if (ctx->sample_radius_max > ctx->radius)
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_build_points radius is smaller than a sample radius");
  P.samples = ctx->samples.as<float4>();
  P.n_samples = ctx->n_samples;
  P.sample_counts = ctx->sample_counts.as<uint32_t>();
  P.vpm_normalization = 1.0f / (float)nb_camera_samples;
  return GVPM_OK;
}

extern "C" {

int gvpm_gather_bre_into(gvpm_ctx *ctx, float *out_dev, uint32_t *counts_dev) {
  if (!ctx || !out_dev) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  return gather_async(ctx, out_dev, counts_dev);
}

int gvpm_gather_bre_device(gvpm_ctx *ctx, const float **out_dev, const uint32_t **counts_dev) {
  if (!ctx) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  int rc = gather_async(ctx, ctx->out.as<float>(), ctx->counts.as<uint32_t>());
  if (rc) return rc;
  if (out_dev) *out_dev = ctx->out.as<float>();
  if (counts_dev) *counts_dev = ctx->counts.as<uint32_t>();
  return GVPM_OK;
}

int gvpm_gather_bre(gvpm_ctx *ctx, float *out, uint32_t *counts) {
  if (!ctx || !out) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  int rc = pending_check(ctx, true);
  if (rc) return rc;
  uint32_t *cdev = counts ? ctx->counts.as<uint32_t>() : nullptr;   // no counts wanted: the traversal filters before queueing
  rc = gather_common(ctx, ctx->out.as<float>(), cdev, ctx->pair_count_host);
  if (rc) return rc;
  const size_t out_bytes = (size_t)ctx->n_rays * GVPM_OUT_FLOATS * sizeof(float), counts_bytes = (size_t)ctx->n_rays * 8;
  // the copies are queued behind the gather before the host waits for it; a re-run after an overflow copies again
  rc = copy_back(ctx, out, out_bytes, counts, counts_bytes, false);
  if (rc) return rc;
  bool redone = false;
  rc = gather_finish(ctx, ctx->out.as<float>(), cdev, ctx->pair_count_host, &redone);
  if (rc) return rc;
  return redone ? copy_back(ctx, out, out_bytes, counts, counts_bytes) : GVPM_OK;
}

// sppm's primal BRE (bre.cpp:167-259 driven as sppm.cpp:926-981): same traverse + shade kernels with
// gvpm_config.sppm_primal set; only the primal (first) spectrum of every ray is produced.
int gvpm_gather_sppm_bre(gvpm_ctx *ctx, float *out, uint32_t *counts) {
  if (!ctx || !out) return GVPM_ERR_INVALID;
  if (!ctx->have_cfg || !ctx->cfg.sppm_primal)
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_gather_sppm_bre needs gvpm_config.sppm_primal = 1");
  cudaSetDevice(ctx->device);
  int rc = pending_check(ctx, true);
  if (rc) return rc;
  rc = gather_common(ctx, ctx->out.as<float>(), ctx->counts.as<uint32_t>(), ctx->pair_count_host);
  if (rc) return rc;
  rc = gather_finish(ctx, ctx->out.as<float>(), ctx->counts.as<uint32_t>(), ctx->pair_count_host, nullptr);
  if (rc) return rc;
  const size_t n = ctx->n_rays;
  if (n)
    CK(cudaMemcpy2DAsync(out, 3 * sizeof(float), ctx->out.p, GVPM_OUT_FLOATS * sizeof(float), 3 * sizeof(float), n,
                         cudaMemcpyDeviceToHost, ctx->stream));
  return copy_back(ctx, nullptr, 0, counts, n * 8);
}

// Pipelined iteration tail: rays are uploaded in chunks on a copy stream while earlier chunks are packed, traversed
// and shaded on the compute stream and their results stream back on a third one, so PCIe (both directions) and the
// SMs work at the same time.  Equivalent to gvpm_upload_rays + gvpm_gather_bre.
int gvpm_gather_bre_host(gvpm_ctx *ctx, const gvpm_ray_soa *r, size_t n, float *out) {
  if (!ctx || (n && (!r || !out))) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  int rc = gvpm_ray_staging(ctx, n, nullptr, nullptr);
  if (rc) return rc;
  CK(ctx->rays.reserve((size_t)n * GVPM_RAY_FLOAT4 * 16 + 256));
  CK(ctx->out.reserve((size_t)n * GVPM_OUT_FLOATS * 4 + 256));
  CK(ctx->counts.reserve((size_t)n * 8 + 256));
  ctx->rays_loaded = true;
  GatherParams P;
  rc = fill_params(ctx, P, ctx->out.as<float>(), nullptr);
  if (rc) return rc;
  rc = pending_check(ctx, true);
  if (rc) return rc;
  CK(cudaEventRecord(ctx->ev[2], ctx->stream));
  ctx->last_pairs = 0;
  int used = 0;
  size_t per = 0;
  if (n) {
    if (ctx->pair_cap == 0) {
      rc = reserve_pairs(ctx, std::max<size_t>(1u << 20, 16 * n));
      if (rc) return rc;
    }
    // chunks of whole 32-ray tiles, ~256k rays each
    int nChunks = (int)std::min<size_t>(32, std::max<size_t>(1, n / 262144));
    per = ((n + nChunks - 1) / nChunks + 31) & ~(size_t)31;
    const RayStaging S = staging_ptrs<RaySoA>(ctx->ray_staging.p, n);
    // the staging buffer may still be read by work queued earlier on the compute stream
    CK(cudaEventRecord(ctx->pipe_ev[64], ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_in, ctx->pipe_ev[64], 0));
    CK(cudaStreamWaitEvent(ctx->copy_out, ctx->pipe_ev[64], 0));
    for (int c = 0; c < nChunks; ++c) {
      const size_t r0 = (size_t)c * per, r1 = std::min(n, r0 + per);
      if (r0 >= r1) break;
      rc = copy_soa<RaySoA>(ctx, *r, ctx->ray_staging.p, n, r0, r0, r1 - r0, ctx->copy_in);
      if (rc) return rc;
      CK(cudaEventRecord(ctx->pipe_ev[2 * c], ctx->copy_in));
      used = c + 1;
    }
    for (int c = 0; c < used; ++c) {
      const size_t r0 = (size_t)c * per, r1 = std::min(n, r0 + per);
      CK(cudaStreamWaitEvent(ctx->stream, ctx->pipe_ev[2 * c], 0));
      launch_pack_rays_range(S, (uint32_t)r0, (uint32_t)r1, ctx->rays.as<float4>(), ctx->stream);
      ctx->launches += 1;
      CK(cudaMemsetAsync(ctx->out.as<float>() + r0 * GVPM_OUT_FLOATS, 0, (r1 - r0) * GVPM_OUT_FLOATS * sizeof(float),
                         ctx->stream));
      rc = enqueue_range(ctx, P, (uint32_t)r0, (uint32_t)r1, ctx->pair_count_host + 16 + c);
      if (rc) return rc;
      CK(cudaEventRecord(ctx->pipe_ev[2 * c + 1], ctx->stream));
      CK(cudaStreamWaitEvent(ctx->copy_out, ctx->pipe_ev[2 * c + 1], 0));
      CK(cudaMemcpyAsync(out + r0 * GVPM_OUT_FLOATS, ctx->out.as<float>() + r0 * GVPM_OUT_FLOATS,
                         (r1 - r0) * GVPM_OUT_FLOATS * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_out));
    }
  }
  CK(cudaEventRecord(ctx->ev[3], ctx->stream));
  ctx->timed_gather = true;
  CK(cudaStreamSynchronize(ctx->copy_out));
  CK(cudaStreamSynchronize(ctx->stream));
  // chunks whose pair list overflowed are run again the slow way (first iteration of a render at most)
  for (int c = 0; c < used; ++c) {
    const unsigned long long total = ctx->pair_count_host[16 + c];
    if (total <= ctx->pair_cap) { ctx->last_pairs += total; continue; }
    const size_t r0 = (size_t)c * per, r1 = std::min(n, r0 + per);
    rc = reserve_pairs(ctx, grown_pairs(total));
    if (rc) return rc;
    rc = gather_range_sync(ctx, P, (uint32_t)r0, (uint32_t)r1, 0);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out + r0 * GVPM_OUT_FLOATS, ctx->out.as<float>() + r0 * GVPM_OUT_FLOATS,
                       (r1 - r0) * GVPM_OUT_FLOATS * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  out_written(ctx);
  return GVPM_OK;
}

int gvpm_dump_neighbours_bre(gvpm_ctx *ctx, uint64_t *offsets, uint32_t *idx, size_t cap) {
  if (!ctx || !offsets) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const size_t n = ctx->n_rays;
  return dump_neighbours(
      ctx, n, offsets, idx, cap, false,
      [&](uint32_t *counts) -> int {
        int rc = pending_check(ctx, true);
        if (rc) return rc;
        rc = gather_common(ctx, ctx->out.as<float>(), ctx->counts.as<uint32_t>(), ctx->pair_count_host);
        if (rc) return rc;
        rc = gather_finish(ctx, ctx->out.as<float>(), ctx->counts.as<uint32_t>(), ctx->pair_count_host, nullptr);
        if (rc) return rc;
        return copy_back(ctx, nullptr, 0, counts, n * 8);
      },
      [&](uint64_t total) -> int {
        GatherParams P;
        int rc = fill_params(ctx, P, ctx->out.as<float>(), nullptr);
        if (rc) return rc;
        P.nbr_offsets = ctx->nbr_offsets.as<uint64_t>();
        P.nbr_idx = ctx->nbr_idx.as<uint32_t>();
        CK(cudaMemsetAsync(ctx->work_counter.p, 0, 16, ctx->stream));
        CK(launch_bre_traverse(P, true, ctx->sm_count, ctx->stream));
        ctx->launches += 1;
        if (ctx->aos_override) {   // dispatched set: report the photons by their index in the whole set
          launch_translate_idx(ctx->nbr_idx.as<uint32_t>(), total, ctx->aos_override, ctx->stream);
          ctx->launches += 1;
        }
        return GVPM_OK;
      });
}

// The sample staging buffer holds a set of n samples (n_dev: a count known on the device only, n is then its bound):
// one kernel packs them (2 float4 per sample), finds the largest sample radius and checks the ray indices and the
// radii (pack_prims.cu); the host reads the stats (and the count) with one copy of three words and checks them.
// Negative or non-finite radii are refused for drawn samples only (an uploaded set keeps the checks it always had).
static int commit_samples(gvpm_ctx *ctx, uint32_t n, const uint32_t *n_dev, bool drawn) {
  uint32_t *stats = ctx->work_counter.as<uint32_t>() + 8;   // words 8, 9 of the counter block (+ word 10: n_dev)
  CK(cudaMemsetAsync(stats, 0, 8, ctx->stream));
  launch_pack_samples(ctx->sample_staging.p, n, n_dev, ctx->n_rays, ctx->samples.as<float4>(), stats, ctx->stream);
  ctx->launches += n ? 1 : 0;
  CK(cudaGetLastError());
  uint32_t *host = ctx->sample_stats_host + 8;
  CK(cudaMemcpyAsync(host, stats, n_dev ? 12 : 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));   // the caller's arrays are only read during the call
  ctx->n_samples = n_dev ? host[2] : n;
  if (host[1] & 1u) {
    ctx->samples_loaded = false;
    return fail(ctx, GVPM_ERR_INVALID, "sample refers to a ray that is not uploaded");
  }
  if (drawn && (host[1] & 2u)) {
    ctx->samples_loaded = false;
    return fail(ctx, GVPM_ERR_INVALID, "per-ray radius must be finite and >= 0");
  }
  memcpy(&ctx->sample_radius_max, &host[0], 4);
  return GVPM_OK;
}

int gvpm_upload_vpm_samples(gvpm_ctx *ctx, const gvpm_vpm_sample_soa *s, size_t n) {
  if (!ctx || (n && !s) || n > 0xfffffff0u) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  ctx->n_samples = (uint32_t)n;
  ctx->samples_loaded = true;
  ctx->samples_drawn = false;
  ctx->sample_radius_max = 0.f;
  ++ctx->state_gen;
  if (n == 0) return GVPM_OK;
  CK(ctx->sample_staging.reserve(SoaLayout<SampleSoA>(n).bytes));
  CK(ctx->samples.reserve(2 * n * sizeof(float4)));
  CK(ctx->sample_counts.reserve(2 * n * sizeof(uint32_t)));
  int rc = copy_soa<SampleSoA>(ctx, *s, ctx->sample_staging.p, n, 0, 0, n, ctx->stream);
  if (rc) return rc;
  return commit_samples(ctx, (uint32_t)n, nullptr, false);
}

// Count -> scan -> emit over the rays (generate.cu), then the upload's pack and checks on the drawn set.  The buffers
// are sized for the bound n_rays * nb; the staging arrays are laid out for the count the scan finds, which the host
// learns from the pack's stats read-back.
int gvpm_generate_vpm_samples(gvpm_ctx *ctx, int nb_camera_samples, int stratified, uint64_t seed, float epsilon,
                              float radius, const float *radius_per_ray_dev, size_t *n_samples) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (!ctx->rays_loaded) return fail(ctx, GVPM_ERR_INVALID, "gvpm_generate_vpm_samples: no committed ray set");
  if (!ctx->have_medium) return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_medium first");
  if (nb_camera_samples <= 0) return fail(ctx, GVPM_ERR_INVALID, "nbCameraSamples must be positive");
  if (!(epsilon > 0.f)) return fail(ctx, GVPM_ERR_INVALID, "epsilon must be > 0");
  if (!radius_per_ray_dev && !(std::isfinite(radius) && radius > 0.f))
    return fail(ctx, GVPM_ERR_INVALID, "radius must be finite and > 0 (or give a per-ray radius array)");
  const uint32_t nr = ctx->n_rays;
  const size_t bound = (size_t)nr * (size_t)nb_camera_samples;
  if (bound > 0xfffffff0u) return fail(ctx, GVPM_ERR_INVALID, "n_rays * nb_camera_samples exceeds 0xfffffff0 samples");
  cudaSetDevice(ctx->device);
  ctx->n_samples = 0;
  ctx->samples_loaded = true;
  ctx->samples_drawn = true;
  ctx->samples_rays_gen = ctx->rays_gen;
  ctx->sample_radius_max = 0.f;
  ++ctx->state_gen;
  if (n_samples) *n_samples = 0;
  if (nr == 0) return GVPM_OK;
  const uint32_t tiles = (nr + 255) / 256;
  CK(ctx->sample_staging.reserve(SoaLayout<SampleSoA>(bound).bytes));
  CK(ctx->samples.reserve(2 * bound * sizeof(float4)));
  CK(ctx->sample_counts.reserve(2 * bound * sizeof(uint32_t)));
  CK(ctx->sample_scratch.reserve(4 * ((size_t)nr + tiles + 1)));
  const RayStaging R = staging_ptrs<RaySoA>(ctx->ray_staging.p, nr);
  uint32_t *total = ctx->work_counter.as<uint32_t>() + 10;   // word 10 of the counter block: read back by commit_samples
  VpmGenParams P{};
  P.o = R.o;
  P.d = R.d;
  P.edge_len = R.edge_len;
  P.radius_per_ray = radius_per_ray_dev;
  P.n_rays = nr;
  P.nb = nb_camera_samples;
  P.stratified = stratified ? 1 : 0;
  P.seed = seed;
  P.epsilon = epsilon;
  P.radius = radius;
  for (int c = 0; c < 3; ++c) P.sigma_t[c] = ctx->medium.sigma_s[c] + ctx->medium.sigma_a[c];
  P.counts = ctx->sample_scratch.as<uint32_t>();
  P.tile_tot = P.counts + nr;
  P.n_total = total;
  P.staging = ctx->sample_staging.p;
  launch_vpm_samples(P, total, ctx->sm_count, ctx->stream);
  ctx->launches += 3;
  CK(cudaGetLastError());
  const int rc = commit_samples(ctx, (uint32_t)bound, total, true);
  if (rc) return rc;
  if (n_samples) *n_samples = ctx->n_samples;
  return GVPM_OK;
}

int gvpm_gather_vpm_device(gvpm_ctx *ctx, int nb_camera_samples, const float **out_dev, const uint32_t **mvol_dev) {
  if (!ctx) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  GatherParams P;
  int rc = vpm_params(ctx, P, nb_camera_samples);
  if (rc) return rc;
  const size_t nr = ctx->n_rays, ns = ctx->n_samples;
  CK(ctx->mvol.reserve(nr * 4 + 256));
  P.mvol = ctx->mvol.as<uint32_t>();
  CK(cudaEventRecord(ctx->ev[2], ctx->stream));
  if (ctx->pair_cap == 0) {
    rc = reserve_pairs(ctx, std::max<size_t>(1u << 20, 8 * ns));
    if (rc) return rc;
  }
  unsigned long long total = 0;
  rc = traverse_growing(
      ctx, P, 3, "VPM pair list overflow", false,
      [&]() -> int {
        CK(cudaMemsetAsync(ctx->work_counter.p, 0, 16, ctx->stream));
        if (nr) CK(cudaMemsetAsync(ctx->out.p, 0, nr * GVPM_OUT_FLOATS * sizeof(float), ctx->stream));
        if (nr) CK(cudaMemsetAsync(ctx->mvol.p, 0, nr * 4, ctx->stream));
        return GVPM_OK;
      },
      [&]() -> int {
        CK(launch_vpm_traverse(P, false, ctx->sm_count, ctx->stream));
        ctx->launches += ns ? 1 : 0;
        return GVPM_OK;
      },
      &total);
  if (rc) return rc;
  ctx->last_pairs = total;
  CK(launch_vpm_shade(P, total, ctx->sm_count, ctx->stream));
  ctx->launches += total ? 1 : 0;
  CK(cudaEventRecord(ctx->ev[3], ctx->stream));
  ctx->timed_gather = true;
  out_written(ctx);
  if (out_dev) *out_dev = ctx->out.as<float>();
  if (mvol_dev) *mvol_dev = ctx->mvol.as<uint32_t>();
  return GVPM_OK;
}

int gvpm_gather_vpm(gvpm_ctx *ctx, int nb_camera_samples, float *out, uint32_t *mvol, uint32_t *sample_counts) {
  if (!ctx || !out) return GVPM_ERR_INVALID;
  int rc = gvpm_gather_vpm_device(ctx, nb_camera_samples, nullptr, nullptr);
  if (rc) return rc;
  const size_t nr = ctx->n_rays, ns = ctx->n_samples;
  if (nr) {
    CK(cudaMemcpyAsync(out, ctx->out.p, nr * GVPM_OUT_FLOATS * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (mvol) CK(cudaMemcpyAsync(mvol, ctx->mvol.p, nr * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (ns && sample_counts)
    CK(cudaMemcpyAsync(sample_counts, ctx->sample_counts.p, ns * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GVPM_OK;
}

int gvpm_dump_neighbours_vpm(gvpm_ctx *ctx, int nb_camera_samples, uint64_t *offsets, uint32_t *idx, size_t cap) {
  if (!ctx || !offsets) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  return dump_neighbours(
      ctx, ctx->n_samples, offsets, idx, cap, false,
      [&](uint32_t *counts) -> int {
        std::vector<float> tmp((size_t)ctx->n_rays * GVPM_OUT_FLOATS + 1);
        return gvpm_gather_vpm(ctx, nb_camera_samples, tmp.data(), nullptr, counts);
      },
      [&](uint64_t) -> int {
        GatherParams P;
        int rc = vpm_params(ctx, P, nb_camera_samples);
        if (rc) return rc;
        P.sample_counts = nullptr;
        P.nbr_offsets = ctx->nbr_offsets.as<uint64_t>();
        P.nbr_idx = ctx->nbr_idx.as<uint32_t>();
        CK(cudaMemsetAsync(ctx->work_counter.p, 0, 16, ctx->stream));
        CK(launch_vpm_traverse(P, true, ctx->sm_count, ctx->stream));
        ctx->launches += 1;
        return GVPM_OK;
      });
}

}  // extern "C"
