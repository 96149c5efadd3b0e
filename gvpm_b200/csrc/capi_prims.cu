// capi_prims.cu — photon planes (G-Planes 0D, uploaded or made from the beam set), photon beams (G-Beams) and sppm's
// primal photon beams.
#include "capi_internal.cuh"

// ---- G-Planes 0D -------------------------------------------------------------------------------
// A new plane set of n planes: the old one and its build are dropped, the staging arrays sized.
static int begin_plane_set(gvpm_ctx *ctx, size_t n) {
  ctx->n_planes = (uint32_t)n;
  ctx->planes_loaded = true;
  ctx->planes_built = false;
  ++ctx->state_gen;
  if (n) CK(ctx->plane_staging.reserve(SoaLayout<PlaneSoA>(n).bytes));
  return GVPM_OK;
}

// The staging arrays hold the plane set: pack the records, and reject a plane with a zero or non-finite edge length.
static int commit_planes(gvpm_ctx *ctx) {
  const uint32_t n = ctx->n_planes;
  if (n == 0) return GVPM_OK;
  CK(ctx->plane_raw.reserve(GVPM_PLANE_PLANES * (size_t)n * sizeof(float4)));
  CK(ctx->plane_pos.reserve(12 * (size_t)n));
  const PlaneStaging S = staging_ptrs<PlaneSoA>(ctx->plane_staging.p, n);
  uint32_t *flag = ctx->work_counter.as<uint32_t>() + 12;   // word 12 of the counter block
  CK(cudaMemsetAsync(flag, 0, 4, ctx->stream));
  launch_pack_planes(S, n, ctx->plane_raw.as<float4>(), ctx->plane_pos.as<float>(), flag, ctx->stream);
  ctx->launches += 1;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->sample_stats_host + 2, flag, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));   // the caller's arrays are only read during the call
  if (ctx->sample_stats_host[2]) {
    // PhotonPlane ctor asserts (plane_struct.h:45-46)
    ctx->planes_loaded = false;
    return fail(ctx, GVPM_ERR_INVALID, "photon plane with zero or non-finite edge length");
  }
  return GVPM_OK;
}

extern "C" {

int gvpm_upload_planes(gvpm_ctx *ctx, const gvpm_plane_soa *p, size_t n) {
  if (!ctx || (n && !p) || n > 0x0ffffff0u) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  int rc = begin_plane_set(ctx, n);
  if (rc || n == 0) return rc;
  rc = copy_soa<PlaneSoA>(ctx, *p, ctx->plane_staging.p, n, 0, 0, n, ctx->stream);
  return rc ? rc : commit_planes(ctx);
}

int gvpm_planes_from_beams(gvpm_ctx *ctx, uint64_t seed) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (!ctx->beams_loaded) return fail(ctx, GVPM_ERR_INVALID, "gvpm_planes_from_beams: no beam set (gvpm_upload_beams or gvpm_trace_beams first)");
  if (!ctx->have_medium) return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_medium first");
  if (ctx->medium.sampling_weight != 1.0f)
    // the reference reads an unset distance sample otherwise (gvpm_host::transformBeam)
    return fail(ctx, GVPM_ERR_INVALID, "transformBeam: mediumSamplingWeight must be 1 for photon planes");
  cudaSetDevice(ctx->device);
  const uint32_t n = ctx->n_beams;
  int rc = begin_plane_set(ctx, n);
  if (rc || n == 0) return rc;
  PlaneGenParams P{};
  P.beams = staging_ptrs<BeamSoA>(ctx->beam_staging.p, n);
  P.n = n;
  P.seed = seed;
  P.sigma_t1 = ctx->medium.sigma_s[1] + ctx->medium.sigma_a[1];   // the balance strategy's sampling density
  P.hg_g = ctx->medium.hg_g;
  P.phase_type = ctx->medium.phase_type;
  writable_view<PlaneSoA>(P.origin, staging_ptrs<PlaneSoA>(ctx->plane_staging.p, n));
  launch_planes_from_beams(P, ctx->stream);
  ctx->launches += 1;
  CK(cudaGetLastError());
  return commit_planes(ctx);
}

int gvpm_build_planes(gvpm_ctx *ctx) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (!ctx->planes_loaded) return fail(ctx, GVPM_ERR_INVALID, "no planes uploaded");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  const uint32_t n = ctx->n_planes;
  CK(cudaEventRecord(ctx->ev[0], st));
  const uint32_t nLeaves = (n + 31) / 32;
  if (n > 0) {
    CK(ctx->plane_bounds.reserve(256));
    CK(ctx->bounds_partial.reserve((size_t)bounds_blocks(n) * 6 * sizeof(float)));
    int rc = reserve_sort(ctx, n);
    if (rc) return rc;
    CK(ctx->plane_rec.reserve(GVPM_PLANE_PLANES * (size_t)n * sizeof(float4)));
    CK(ctx->plane_orig.reserve(4 * (size_t)n));
    CK(ctx->plane_box_lo.reserve(16 * (size_t)nLeaves));
    CK(ctx->plane_box_hi.reserve(16 * (size_t)nLeaves));
    launch_bounds(ctx->plane_pos.as<float>(), n, ctx->bounds_partial.as<float>(), ctx->plane_bounds.as<float>(), st);
    launch_morton(ctx->plane_pos.as<float>(), n, ctx->plane_bounds.as<float>(), ctx->keys_in.as<uint32_t>(),
                  ctx->vals_in.as<uint32_t>(), st);
    CK(run_sort_bits(ctx->sort_temp.p, ctx->sort_temp.cap, ctx->keys_in.as<uint32_t>(), ctx->keys_out.as<uint32_t>(),
                     ctx->vals_in.as<uint32_t>(), ctx->vals_out.as<uint32_t>(), n, kHilbertBits, st));
    launch_plane_pack_sorted(ctx->plane_raw.as<float4>(), ctx->vals_out.as<uint32_t>(), n, ctx->plane_rec.as<float4>(),
                             ctx->plane_orig.as<uint32_t>(), st);
    launch_plane_leaf_boxes(ctx->plane_rec.as<float4>(), n, nLeaves, ctx->plane_box_lo.as<float4>(),
                            ctx->plane_box_hi.as<float4>(), st);
    ctx->launches += 4 + 4;
    CK(cudaGetLastError());
  }
  ctx->planes_built = true;
  CK(cudaEventRecord(ctx->ev[1], st));
  ctx->timed_build = true;
  return GVPM_OK;
}

static int plane_params(gvpm_ctx *ctx, GatherParams &P) {
  int rc = gather_params(ctx, P, ctx->planes_built, "gvpm_build_planes has not been called");
  if (rc) return rc;
  P.tree.lo = ctx->plane_box_lo.as<float4>();
  P.tree.hi = ctx->plane_box_hi.as<float4>();
  P.tree.n = ctx->n_planes;
  P.out = ctx->out.as<float>();
  P.counts = ctx->counts.as<uint32_t>();
  P.plane_rec = ctx->plane_rec.as<float4>();
  P.plane_orig = ctx->plane_orig.as<uint32_t>();
  P.n_planes = ctx->n_planes;
  return GVPM_OK;
}

int gvpm_gather_planes_device(gvpm_ctx *ctx, const float **out_dev, const uint32_t **counts_dev) {
  if (!ctx) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  GatherParams P;
  int rc = plane_params(ctx, P);
  if (rc) return rc;
  if (!counts_dev) P.counts = nullptr;
  CK(cudaEventRecord(ctx->ev[2], ctx->stream));
  CK(cudaMemsetAsync(ctx->work_counter.p, 0, 32, ctx->stream));
  ctx->split_timed = false;
  CK(launch_plane_gather(P, false, ctx->sm_count, ctx->stream));
  ctx->launches += ctx->n_rays ? 1 : 0;
  CK(cudaEventRecord(ctx->ev[3], ctx->stream));
  ctx->timed_gather = true;
  out_written(ctx);
  if (out_dev) *out_dev = ctx->out.as<float>();
  if (counts_dev) *counts_dev = ctx->counts.as<uint32_t>();
  return GVPM_OK;
}

int gvpm_gather_planes(gvpm_ctx *ctx, float *out, uint32_t *counts) {
  if (!ctx || !out) return GVPM_ERR_INVALID;
  const uint32_t *cd = nullptr;
  int rc = gvpm_gather_planes_device(ctx, nullptr, counts ? &cd : nullptr);
  if (rc) return rc;
  const size_t n = ctx->n_rays;
  return copy_back(ctx, out, n * GVPM_OUT_FLOATS * sizeof(float), counts, n * 8);
}

int gvpm_dump_neighbours_planes(gvpm_ctx *ctx, uint64_t *offsets, uint32_t *idx, size_t cap) {
  if (!ctx || !offsets) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  return dump_neighbours(
      ctx, ctx->n_rays, offsets, idx, cap, false,
      [&](uint32_t *counts) -> int {
        std::vector<float> tmp((size_t)ctx->n_rays * GVPM_OUT_FLOATS + 1);
        return gvpm_gather_planes(ctx, tmp.data(), counts);
      },
      [&](uint64_t) -> int {
        GatherParams P;
        int rc = plane_params(ctx, P);
        if (rc) return rc;
        P.counts = nullptr;
        P.nbr_offsets = ctx->nbr_offsets.as<uint64_t>();
        P.nbr_idx = ctx->nbr_idx.as<uint32_t>();
        CK(cudaMemsetAsync(ctx->work_counter.p, 0, 32, ctx->stream));
        CK(launch_plane_gather(P, true, ctx->sm_count, ctx->stream));
        ctx->launches += 1;
        return GVPM_OK;
      });
}

// ---- G-Beams 3D --------------------------------------------------------------------------------
}  // extern "C"

int begin_beam_set(gvpm_ctx *ctx, size_t n) {
  ctx->n_beams = (uint32_t)n;
  ctx->beams_loaded = true;
  ctx->beams_built = false;
  ctx->n_subs = 0;
  ctx->beam_subsize = 0.f;
  ++ctx->state_gen;
  if (n == 0) return GVPM_OK;
  CK(ctx->beam_staging.reserve(SoaLayout<BeamSoA>(n).bytes));
  CK(ctx->beams.reserve(8 * n * sizeof(float4)));
  CK(ctx->beam_len.reserve(4 * n));
  CK(ctx->beam_aux.reserve(64 + 4 * ((n + 255) / 256 + 1)));
  return GVPM_OK;
}

// A kernel assembles the 128-byte beam records from the staging arrays (pack_prims.cu).  The one thing that has to be
// sequential is the fp32 running sum of the beam lengths that fixes the sub-beam size (beams_accel.h:98-104), and with
// it the number of sub-beams (sizes the sort without a read-back in the build).  Uploaded beams: the host does the sum
// from the caller's arrays while the DMA runs.  Beams made on the device: one warp does it there (k_beam_subsize_seq),
// the sub-beams are counted (k_sub_count) and both numbers are read back.
int commit_beams(gvpm_ctx *ctx, const gvpm_beam_soa *b) {
  const uint32_t n = ctx->n_beams;
  if (n == 0) return GVPM_OK;
  launch_pack_beams(staging_ptrs<BeamSoA>(ctx->beam_staging.p, n), n, ctx->beams.as<float4>(), ctx->beam_len.as<float>(), ctx->stream);
  ctx->launches += 1;
  uint64_t total = 0;
  float subbeamSize = 0.f;
  if (b) {
    // host, under the DMA: PhotonBeam::setEndPoint lengths, sequential sum, sub-beam count (SubBeamBVH ctor)
    std::vector<float> len(n);
    float avgSize = 0.f;
    for (size_t i = 0; i < n; ++i) {
      const float *o = b->origin + 3 * i, *e = b->end + 3 * i;
      const float d[3] = {e[0] - o[0], e[1] - o[1], e[2] - o[2]};
      len[i] = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
      avgSize += len[i];
    }
    avgSize /= (float)n;
    subbeamSize = avgSize / 10;
    for (size_t i = 0; i < n; ++i) {
      int nSub = subbeamSize > 0.f ? (int)std::ceil(len[i] / subbeamSize) : 1;
      total += (uint64_t)(nSub < 1 ? 1 : nSub);
    }
  } else {
    // aux[0] = subbeamSize, aux[1] = sub-beam total (fewer than 11 per beam: no 32-bit overflow), aux[16..] block sums
    float *subsize = ctx->beam_aux.as<float>();
    uint32_t *aux = ctx->beam_aux.as<uint32_t>();
    launch_beam_subsize_seq(ctx->beam_len.as<float>(), n, subsize, ctx->stream);
    launch_sub_count(ctx->beam_len.as<float>(), n, subsize, aux + 16, aux + 1, ctx->stream);
    ctx->launches += 3;
    uint32_t *host = ctx->sample_stats_host + 4;   // pinned words 4, 5
    CK(cudaMemcpyAsync(host, aux, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memcpy(&subbeamSize, host, 4);
    total = host[1];
  }
  if (total > 0xfffffff0ull) return fail(ctx, GVPM_ERR_INVALID, "too many sub-beams");
  ctx->beam_subsize = subbeamSize;
  ctx->n_subs = (uint32_t)total;
  if (b) CK(cudaMemcpyAsync(ctx->beam_aux.p, &ctx->beam_subsize, 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream));   // the caller's arrays are only read during the call
  return GVPM_OK;
}

extern "C" {

int gvpm_upload_beams(gvpm_ctx *ctx, const gvpm_beam_soa *b, size_t n) {
  if (!ctx || (n && !b) || n > 0x0ffffff0u) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  int rc = begin_beam_set(ctx, n);
  if (rc || n == 0) return rc;
  rc = copy_soa<BeamSoA>(ctx, *b, ctx->beam_staging.p, n, 0, 0, n, ctx->stream);
  return rc ? rc : commit_beams(ctx, b);
}

int gvpm_build_beams(gvpm_ctx *ctx, float radius) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (!ctx->beams_loaded) return fail(ctx, GVPM_ERR_INVALID, "no beams uploaded");
  if (!(radius > 0.f)) return fail(ctx, GVPM_ERR_INVALID, "radius must be positive");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  const uint32_t nb = ctx->n_beams, n = ctx->n_subs;
  CK(cudaEventRecord(ctx->ev[0], st));
  Tree T{};
  uint32_t total = 0;
  int rc = bvh_levels(ctx, T, n, "too many sub-beams", &total);
  if (rc) return rc;
  const int levels = T.levels;
  CK(ctx->beam_bounds.reserve(256));
  if (n > 0) {
    CK(ctx->sub_pos.reserve(12 * (size_t)n));
    CK(ctx->sub_raw.reserve(16 * (size_t)n));
    CK(ctx->subs.reserve(16 * (size_t)n));
    rc = reserve_sort(ctx, n);
    if (rc) return rc;
    CK(ctx->bounds_partial.reserve((size_t)bounds_blocks(n) * 6 * sizeof(float)));
    CK(ctx->beam_box_lo.reserve(16 * (size_t)total));
    CK(ctx->beam_box_hi.reserve(16 * (size_t)total));
    // sub-beam cuts on the device (pack_prims.cu): per-beam counts -> offsets -> (midpoint, t1, t2, beam, flags)
    const float *subsize = ctx->beam_aux.as<float>();
    uint32_t *aux = ctx->beam_aux.as<uint32_t>();
    launch_sub_count(ctx->beam_len.as<float>(), nb, subsize, aux + 16, aux + 1, st);
    launch_sub_emit(ctx->beams.as<float4>(), ctx->beam_len.as<float>(), nb, subsize, aux + 16, n, ctx->sub_pos.as<float>(),
                    ctx->sub_raw.as<float4>(), st);
    launch_bounds(ctx->sub_pos.as<float>(), n, ctx->bounds_partial.as<float>(), ctx->beam_bounds.as<float>(), st);
    launch_morton(ctx->sub_pos.as<float>(), n, ctx->beam_bounds.as<float>(), ctx->keys_in.as<uint32_t>(),
                  ctx->vals_in.as<uint32_t>(), st);
    CK(run_sort_bits(ctx->sort_temp.p, ctx->sort_temp.cap, ctx->keys_in.as<uint32_t>(), ctx->keys_out.as<uint32_t>(),
                     ctx->vals_in.as<uint32_t>(), ctx->vals_out.as<uint32_t>(), n, kHilbertBits, st));
    launch_sub_gather(ctx->sub_raw.as<float4>(), ctx->vals_out.as<uint32_t>(), n, ctx->subs.as<float4>(), st);
    float4 *lo = ctx->beam_box_lo.as<float4>(), *hi = ctx->beam_box_hi.as<float4>();
    launch_subbeam_leaf_boxes(ctx->subs.as<float4>(), ctx->beams.as<float4>(), n, T.cnt[0], radius, lo, hi, st);
    for (int l = 1; l < levels; ++l)
      launch_level_boxes(lo + T.off[l - 1], hi + T.off[l - 1], T.cnt[l - 1], T.cnt[l], lo + T.off[l], hi + T.off[l], st);
    ctx->launches += 8 + (levels - 1) + 4;
    CK(cudaGetLastError());
  } else {
    CK(cudaMemsetAsync(ctx->beam_bounds.p, 0, 7 * sizeof(float), st));
  }
  T.lo = ctx->beam_box_lo.as<float4>();
  T.hi = ctx->beam_box_hi.as<float4>();
  ctx->beam_tree = T;
  ctx->beam_radius = radius;
  ctx->beams_built = true;
  ++ctx->state_gen;
  CK(cudaEventRecord(ctx->ev[1], st));
  ctx->timed_build = true;
  return GVPM_OK;
}

uint64_t gvpm_beam_subbeam_count(const gvpm_ctx *ctx) { return ctx ? ctx->n_subs : 0; }

static int beam_params(gvpm_ctx *ctx, GatherParams &P) {
  int rc = gather_params(ctx, P, ctx->beams_built, "gvpm_build_beams has not been called");
  if (rc) return rc;
  P.tree = ctx->beam_tree;
  const float r = ctx->beam_radius;
  P.radius = r;
  P.radius_sq = r * r;
  P.kernel_vol = (float)((4.0 / 3.0) * (double)GVPM_PI * std::pow((double)r, 3));
  P.weight_kernel = (float)(1.0 / P.kernel_vol);  // shift_volume_beams.h:272
  if (ctx->cfg.beam_kernel_1d) P.weight_kernel = 0.5f / r;  // :188
  P.bounds = ctx->beam_bounds.as<float>();
  P.out = ctx->out.as<float>();
  P.counts = ctx->counts.as<uint32_t>();
  P.pair_counter = (unsigned long long *)(ctx->work_counter.as<char>() + 8);
  P.dump_counter = (unsigned long long *)(ctx->work_counter.as<char>() + 16);
  P.ray_begin = 0;
  P.ray_end = ctx->n_rays;
  P.beams = ctx->beams.as<float4>();
  P.subs = ctx->subs.as<float4>();
  P.n_beams = ctx->n_beams;
  P.sppm_beam_technique = -1;
  return GVPM_OK;
}

// traverse + shade with pair-list growth; dump != nullptr: fill the flat geometric pair list instead of shading
static int beams_run(gvpm_ctx *ctx, GatherParams &P, bool want_counts) {
  const size_t nr = ctx->n_rays;
  if (ctx->pair_cap == 0) {
    int rc = reserve_pairs(ctx, std::max<size_t>(1u << 20, 64 * nr));
    if (rc) return rc;
  }
  const bool sppm = P.sppm_beam_technique >= 0;
  P.beam_prefilter = (want_counts || P.dump_pairs || sppm) ? 0 : 1;
  unsigned long long total = 0;
  int rc = traverse_growing(
      ctx, P, 4, "beam pair list overflow", false,
      [&]() -> int {
        CK(cudaMemsetAsync(ctx->work_counter.p, 0, 32, ctx->stream));
        return GVPM_OK;
      },
      [&]() -> int {
        CK(launch_beam_traverse(P, ctx->sm_count, ctx->stream));
        ctx->launches += nr ? 1 : 0;
        return GVPM_OK;
      },
      &total);
  if (rc) return rc;
  ctx->last_pairs = total;
  if (nr) {
    CK(cudaMemsetAsync(ctx->out.p, 0, nr * GVPM_OUT_FLOATS * sizeof(float), ctx->stream));
    CK(cudaMemsetAsync(ctx->counts.p, 0, nr * 8, ctx->stream));
  }
  CK(sppm ? launch_beam_shade_sppm(P, total, ctx->sm_count, ctx->stream)
          : launch_beam_shade(P, total, ctx->sm_count, ctx->stream));
  ctx->launches += total ? 1 : 0;
  return GVPM_OK;
}

int gvpm_gather_beams_device(gvpm_ctx *ctx, const float **out_dev, const uint32_t **counts_dev) {
  if (!ctx) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  GatherParams P;
  int rc = beam_params(ctx, P);
  if (rc) return rc;
  CK(cudaEventRecord(ctx->ev[2], ctx->stream));
  rc = beams_run(ctx, P, counts_dev != nullptr);
  if (rc) return rc;
  CK(cudaEventRecord(ctx->ev[3], ctx->stream));
  ctx->timed_gather = true;
  out_written(ctx);
  if (out_dev) *out_dev = ctx->out.as<float>();
  if (counts_dev) *counts_dev = ctx->counts.as<uint32_t>();
  return GVPM_OK;
}

int gvpm_gather_beams(gvpm_ctx *ctx, float *out, uint32_t *counts) {
  if (!ctx || !out) return GVPM_ERR_INVALID;
  const uint32_t *cd = nullptr;
  int rc = gvpm_gather_beams_device(ctx, nullptr, counts ? &cd : nullptr);
  if (rc) return rc;
  const size_t n = ctx->n_rays;
  return copy_back(ctx, out, n * GVPM_OUT_FLOATS * sizeof(float), counts, n * 8);
}

// the flat (ray, beam) list of the accepted pairs, gathered as the counts above were
static int dump_beam_pairs(gvpm_ctx *ctx, GatherParams &P, uint64_t total) {
  P.counts = nullptr;
  P.dump_pairs = ctx->nbr_idx.as<uint2>();
  P.dump_cap = total;
  return beams_run(ctx, P, true);
}

int gvpm_dump_neighbours_beams(gvpm_ctx *ctx, uint64_t *offsets, uint32_t *idx, size_t cap) {
  if (!ctx || !offsets) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  return dump_neighbours(
      ctx, ctx->n_rays, offsets, idx, cap, true,
      [&](uint32_t *counts) -> int {
        std::vector<float> tmp((size_t)ctx->n_rays * GVPM_OUT_FLOATS + 1);
        return gvpm_gather_beams(ctx, tmp.data(), counts);
      },
      [&](uint64_t total) -> int {
        GatherParams P;
        int rc = beam_params(ctx, P);
        return rc ? rc : dump_beam_pairs(ctx, P, total);
      });
}

// ---- sppm primal photon beams (sppm.cpp:823-860 + beams.h:29-223) ------------------------------------------------
static int sppm_beam_params(gvpm_ctx *ctx, int technique, GatherParams &P) {
  if (technique < GVPM_BEAM_1D || technique > GVPM_BEAM_3D_OPTIMIZED)
    return fail(ctx, GVPM_ERR_INVALID, "unknown gvpm_beam_technique");
  int rc = beam_params(ctx, P);
  if (rc) return rc;
  P.sppm_beam_technique = technique;
  return GVPM_OK;
}

int gvpm_gather_sppm_beams(gvpm_ctx *ctx, int technique, float *out, uint32_t *counts) {
  if (!ctx || !out) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  GatherParams P;
  int rc = sppm_beam_params(ctx, technique, P);
  if (rc) return rc;
  CK(cudaEventRecord(ctx->ev[2], ctx->stream));
  rc = beams_run(ctx, P, counts != nullptr);
  if (rc) return rc;
  CK(cudaEventRecord(ctx->ev[3], ctx->stream));
  ctx->timed_gather = true;
  out_written(ctx, 3);   // [n_rays][3]
  const size_t n = ctx->n_rays;
  return copy_back(ctx, out, n * 3 * sizeof(float), counts, n * 8);
}

int gvpm_dump_neighbours_sppm_beams(gvpm_ctx *ctx, int technique, uint64_t *offsets, uint32_t *idx, size_t cap) {
  if (!ctx || !offsets) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  return dump_neighbours(
      ctx, ctx->n_rays, offsets, idx, cap, true,
      [&](uint32_t *counts) -> int {
        std::vector<float> tmp((size_t)ctx->n_rays * 3 + 1);
        return gvpm_gather_sppm_beams(ctx, technique, tmp.data(), counts);
      },
      [&](uint64_t total) -> int {
        GatherParams P;
        int rc = sppm_beam_params(ctx, technique, P);
        return rc ? rc : dump_beam_pairs(ctx, P, total);
      });
}

}  // extern "C"
