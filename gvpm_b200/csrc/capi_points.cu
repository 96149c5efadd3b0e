// capi_points.cu — point hierarchies over the photons: full BVH, ray-region pruned BVH, perspective grid.
#include "capi_internal.cuh"

int reserve_sort(gvpm_ctx *ctx, uint32_t n) {
  CK(ctx->keys_in.reserve(8 * (size_t)n));
  CK(ctx->keys_out.reserve(8 * (size_t)n));
  CK(ctx->vals_in.reserve(4 * (size_t)n));
  CK(ctx->vals_out.reserve(4 * (size_t)n));
  CK(ctx->sort_temp.reserve(sort_temp_bytes(n)));
  return GVPM_OK;
}

// Level sizes of the implicit 32-ary hierarchy over n leaves' elements (gvpm_device.cuh Tree); *nodes = all levels' nodes.
int bvh_levels(gvpm_ctx *ctx, Tree &T, uint32_t n, const char *too_many, uint32_t *nodes) {
  T.n = n;
  uint32_t cnt = (n + 31) / 32, total = 0;
  int levels = 0;
  if (n > 0) {
    for (;;) {
      T.cnt[levels] = cnt;
      T.off[levels] = total;
      total += cnt;
      ++levels;
      if (cnt <= 32) break;
      if (levels >= GVPM_MAX_LEVELS) return fail(ctx, GVPM_ERR_INVALID, too_many);
      cnt = (cnt + 31) / 32;
    }
  }
  T.levels = levels;
  *nodes = total;
  return GVPM_OK;
}

// a point build has finished: its structure becomes the one the gathers use
static int points_built(gvpm_ctx *ctx, const Tree &T, float radius, int accel, bool pruned, uint32_t n_kept) {
  ctx->tree = T;
  ctx->radius = radius;
  ctx->built = true;
  ctx->accel = accel;
  ++ctx->state_gen;
  ctx->pruned = pruned;
  if (pruned) ctx->pruned_for_gen = ctx->rays_gen;
  ctx->n_kept = n_kept;
  CK(cudaEventRecord(ctx->ev[1], ctx->stream));
  ctx->timed_build = true;
  return GVPM_OK;
}

// Same hierarchy, over the photons the uploaded rays can reach only (tree_build.cu, "ray-region pruning").
int build_pruned_bvh(gvpm_ctx *ctx, float radius, uint32_t *n_kept) {
  cudaSetDevice(ctx->device);
  if (ctx->photons_direct) {   // records traced in place: no staged SoA to prune from, build over all of them
    int rc = gvpm_build_points(ctx, radius);
    if (rc == GVPM_OK) { ctx->pruned = false; if (n_kept) *n_kept = ctx->n_photons; }
    return rc;
  }
  const uint32_t n = ctx->n_photons;
  cudaStream_t st = ctx->stream;
  CK(cudaEventRecord(ctx->ev[0], st));
  const size_t gridOff = 32, maskOff = align256(gridOff + ray_grid_bytes()), keepOff = align256(maskOff + ray_mask_bytes());
  CK(ctx->ray_region.reserve(keepOff + 4 * ((size_t)n / 32 + 1)));
  char *rr = ctx->ray_region.as<char>();
  float *box = (float *)rr;
  uint32_t *mask = (uint32_t *)(rr + maskOff), *keepmask = (uint32_t *)(rr + keepOff);
  const float boxInit[8] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY, 0.f, 0.f};
  CK(cudaMemcpyAsync(box, boxInit, sizeof(boxInit), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(mask, 0, ray_mask_bytes(), st));
  launch_ray_region(ctx->rays.as<float4>(), ctx->n_rays, radius, box, rr + gridOff, mask, ctx->bounds.as<float>(),
                    ctx->sm_count, st);
  ctx->launches += ctx->n_rays ? 3 : 1;
  uint32_t kept = 0;
  if (n > 0) {
    int rc = reserve_sort(ctx, n);
    if (rc) return rc;
    CK(ctx->planes.reserve(16 * (size_t)n));
    CK(ctx->orig.reserve(4 * (size_t)n));
    CK(ctx->aos.reserve(128 * (size_t)n));
    const PhotonStaging S = staging_ptrs<PhotonSoA>(ctx->ph_staging.p, n);
    // kept indices in photon order (deterministic): per-CTA counts, exclusive scan, ordered compaction
    const uint32_t nb = (n + 255) / 256;
    CK(ctx->keepmask.reserve(4 * ((size_t)nb + 4)));
    uint32_t *block_kept = ctx->keepmask.as<uint32_t>();
    launch_keep_pruned(S.pos, n, rr + gridOff, mask, keepmask, block_kept, st);
    launch_scan_u32(block_kept, nb, block_kept + nb, st);
    launch_compact_kept(keepmask, block_kept, n, ctx->vals_in.as<uint32_t>(), st);
    ctx->launches += 3;
    // the number of kept photons sizes the sort and the hierarchy levels: one 4-byte read-back
    CK(cudaMemcpyAsync(ctx->pair_count_host, block_kept + nb, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    kept = *(const uint32_t *)ctx->pair_count_host;
  }
  Tree T{};
  uint32_t total = 0;
  int rc = bvh_levels(ctx, T, kept, "too many photons", &total);
  if (rc) return rc;
  const int levels = T.levels;
  if (kept > 0) {
    CK(ctx->box_lo.reserve(16 * (size_t)total));
    CK(ctx->box_hi.reserve(16 * (size_t)total));
    const PhotonStaging S = staging_ptrs<PhotonSoA>(ctx->ph_staging.p, n);
    launch_keys_kept(S.pos, ctx->vals_in.as<uint32_t>(), kept, rr + gridOff, ctx->keys_in.as<uint32_t>(), st);
    CK(run_sort_bits(ctx->sort_temp.p, ctx->sort_temp.cap, ctx->keys_in.as<uint32_t>(), ctx->keys_out.as<uint32_t>(),
                     ctx->vals_in.as<uint32_t>(), ctx->vals_out.as<uint32_t>(), kept, kHilbertBits, st));
    launch_pack_sorted_kept(S, n, keepmask, ctx->vals_out.as<uint32_t>(), kept, ctx->aos.as<float4>(),
                            ctx->planes.as<float4>(), ctx->orig.as<uint32_t>(), st);
    float4 *lo = ctx->box_lo.as<float4>(), *hi = ctx->box_hi.as<float4>();
    launch_leaf_boxes(ctx->planes.as<float4>(), kept, T.cnt[0], radius, lo, hi, st);
    for (int l = 1; l < levels; ++l)
      launch_level_boxes(lo + T.off[l - 1], hi + T.off[l - 1], T.cnt[l - 1], T.cnt[l], lo + T.off[l], hi + T.off[l], st);
    ctx->launches += 4 + (levels - 1) + 4;
    CK(cudaGetLastError());
  }
  if (n > 0) CK(cudaEventRecord(ctx->ev_free[ctx->ph_staging_sel], st));   // last read of the staging buffer
  T.lo = ctx->box_lo.as<float4>();
  T.hi = ctx->box_hi.as<float4>();
  if (n_kept) *n_kept = kept;
  return points_built(ctx, T, radius, gvpm_ctx::ACCEL_BVH, true, kept);
}


// ---- frustum grid (gvpm_device.cuh FrustumGrid) -------------------------------------------------------------------------
static float decode_max_key(unsigned key) {
  const unsigned b = (key & 0x80000000u) ? (key ^ 0x80000000u) : ~key;
  float f;
  memcpy(&f, &b, 4);
  return f;
}
// Are the uploaded rays concurrent (do their lines meet in one point)?  Two reductions over the packed rays and one
// read-back, cached until other rays are uploaded.
int analyse_rays(gvpm_ctx *ctx) {
  if (ctx->pin_gen == ctx->rays_gen) return GVPM_OK;
  gvpm_ctx::RayFit &F = ctx->pin;
  F.concurrent = false;
  ctx->pin_gen = ctx->rays_gen;
  const uint32_t n = ctx->n_rays;
  if (n == 0) return GVPM_OK;
  CK(ctx->pin_scratch.reserve(128 + (size_t)pinhole_blocks(n) * 16 * sizeof(double)));
  char *ps = ctx->pin_scratch.as<char>();
  launch_pinhole_fit(ctx->rays.as<float4>(), n, (double *)(ps + 128), (float *)ps, (unsigned *)(ps + 64), ctx->stream,
                     ctx->have_view_dir ? ctx->view_dir : nullptr);
  ctx->launches += 3;
  CK(cudaMemcpyAsync(ctx->pin_host, ps, 96, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const float *fit = ctx->pin_host;
  const unsigned *st = (const unsigned *)(ctx->pin_host + 16);
  F.count = fit[12];
  if (!(F.count >= 1.f) || !(fit[13] > 0.f)) return GVPM_OK;   // no active ray, or parallel rays (no common point)
  for (int k = 0; k < 3; ++k) { F.C[k] = fit[k]; F.m[k] = fit[3 + k]; F.u[k] = fit[6 + k]; F.v[k] = fit[9 + k]; }
  F.delta = decode_max_key(st[0]);
  F.cosmin = -decode_max_key(st[1]);
  F.xmin = -decode_max_key(st[2]); F.xmax = decode_max_key(st[3]);
  F.ymin = -decode_max_key(st[4]); F.ymax = decode_max_key(st[5]);
  F.concurrent = std::isfinite(F.delta) && F.cosmin > 0.35f && std::isfinite(F.xmin) && std::isfinite(F.xmax) &&
                 std::isfinite(F.ymin) && std::isfinite(F.ymax) && F.xmin <= F.xmax && F.ymin <= F.ymax;
  return GVPM_OK;
}

// The grid of a concurrent ray set (RayFit) for search radius `radius`: host arithmetic only, so that a rank that SENDS
// photons (dispatch.cu) derives the receiver's grid from the receiver's RayFit exactly as the receiver does.
FrustumGrid make_frustum_grid(const gvpm_ctx::RayFit &F, float radius, bool parity_split) {
  FrustumGrid G{};
  for (int k = 0; k < 3; ++k) { G.C[k] = F.C[k]; G.m[k] = F.m[k]; G.u[k] = F.u[k]; G.v[k] = F.v[k]; }
  G.xmin = F.xmin; G.xmax = F.xmax; G.ymin = F.ymin; G.ymax = F.ymax;
  G.pad_r = radius + F.delta;
  // about one ray per class-0 cell, square cells, at most 4 M of them; every class doubles the cell edge
  const double ex = std::max((double)F.xmax - F.xmin, 1e-9), ey = std::max((double)F.ymax - F.ymin, 1e-9);
  const double target = std::min(std::max((double)F.count, 64.0), 4.0e6);
  double cell = std::sqrt(ex * ey / target);
  cell = std::max(cell, std::max(ex, ey) / 4096.0);
  G.gx0 = F.xmin;
  G.gy0 = F.ymin;
  uint32_t total = 0;
  int classes = 0;
  for (int c = 0; c < GVPM_GRID_CLASSES; ++c) {
    G.csize[c] = (float)(cell * std::pow(2.0, (double)c));
    G.nx[c] = (uint32_t)std::floor(ex / G.csize[c]) + 2u;
    G.ny[c] = (uint32_t)std::floor(ey / G.csize[c]) + 2u;
    G.base[c] = total;
    total += G.nx[c] * G.ny[c];
    classes = c + 1;
    if (G.nx[c] <= 2 && G.ny[c] <= 2) break;
  }
  for (int c = classes; c < GVPM_GRID_CLASSES; ++c) { G.csize[c] = G.csize[classes - 1]; G.nx[c] = G.ny[c] = 1; G.base[c] = total; }
  G.classes = classes;
  G.n_cells = total;
  G.parity_split = parity_split ? 1 : 0;
  return G;
}

int build_frustum(gvpm_ctx *ctx, float radius, uint32_t *n_kept) {
  cudaSetDevice(ctx->device);
  const uint32_t n = ctx->n_photons;
  cudaStream_t st = ctx->stream;
  const gvpm_ctx::RayFit &F = ctx->pin;
  CK(cudaEventRecord(ctx->ev[0], st));
  const FrustumGrid G = make_frustum_grid(F, radius, ctx->have_cfg && ctx->cfg.path_set && !ctx->cfg.sppm_primal);
  const uint32_t total = G.n_cells;
  const uint32_t n_keys = (G.parity_split ? 2u : 1u) * total + 2;   // + NEAR + DROP
  CK(ctx->cell_start.reserve(((size_t)n_keys + 1) * 4));
  if (n > 0) {
    CK(ctx->keys_in.reserve(4 * (size_t)n));
    CK(ctx->vals_in.reserve(4 * (size_t)n));
    CK(ctx->sort_temp.reserve(cell_scan_temp_bytes(n_keys)));
    CK(ctx->cell_count.reserve(((size_t)n_keys + 2) * 4));
    CK(ctx->planes.reserve(16 * (size_t)n));
    CK(ctx->orig.reserve(4 * (size_t)n));
    CK(ctx->keepmask.reserve(4 * ((size_t)n / 32 + 2)));
    const bool direct = ctx->photons_direct;
    if (!direct) CK(ctx->aos.reserve(128 * (size_t)n));
    CK(ctx->grid_occ.reserve(frustum_occ_bytes()));
    uint32_t *keepmask = ctx->keepmask.as<uint32_t>(), *cell_count = ctx->cell_count.as<uint32_t>();
    // the word after the keep bits: set when the build is incomplete (gvpm_build_dispatched: a peer's dispatch timed out
    // or overflowed its region); the gather reports it instead of gathering
    uint32_t *ovf = keepmask + (n / 32 + 1);
    CK(cudaMemsetAsync(ovf, 0, 4, st));
    PhotonStaging S{};
    if (!direct) S = staging_ptrs<PhotonSoA>(ctx->ph_staging.p, n);
    // Counting sort: the key pass counts the photons of every cell and gives each its rank in the cell; the exclusive scan
    // of the counters IS cell_start; the packing pass (or a scatter pass over records that exist already) puts position
    // plane entry and index at cell_start[key] + rank.  Nothing to size from a count: dropped photons and the empty part
    // of a dispatched inbox are simply never written.  The order inside a cell follows the atomics (the gather's float
    // atomics are unordered anyway).
    CK(cudaMemsetAsync(cell_count, 0, ((size_t)n_keys + 2) * 4, st));
    if (direct)   // position = first three floats of the record, path parity = bit 10 of its meta word
      launch_frustum_keys(ctx->rays.as<float4>(), ctx->n_rays, (const float *)ctx->records(), 32u, (const uint32_t *)ctx->records() + 3, 32u, 10u, n,
                          G, ctx->grid_occ.as<uint32_t>(), ctx->keys_in.as<uint32_t>(), ctx->vals_in.as<uint32_t>(),
                          ctx->bounds.as<unsigned>() + 6, keepmask, cell_count, ctx->region_cap, ctx->region_count, ctx->sm_count, st);
    else
      launch_frustum_keys(ctx->rays.as<float4>(), ctx->n_rays, S.pos, 3u, S.path_id, 1u, 0u, n, G, ctx->grid_occ.as<uint32_t>(),
                          ctx->keys_in.as<uint32_t>(), ctx->vals_in.as<uint32_t>(), ctx->bounds.as<unsigned>() + 6, keepmask,
                          cell_count, 0, nullptr, ctx->sm_count, st);
    CK(launch_cell_scan(ctx->sort_temp.p, ctx->sort_temp.cap, cell_count, ctx->cell_start.as<uint32_t>(), n_keys, st));
    launch_pack_scatter(S, n, keepmask, ctx->keys_in.as<uint32_t>(), ctx->vals_in.as<uint32_t>(), ctx->cell_start.as<uint32_t>(),
                        ctx->records(), ctx->planes.as<float4>(), ctx->orig.as<uint32_t>(), st, direct,
                        ctx->cell_start.as<uint32_t>() + n_keys - 1, ctx->sm_count);
    ctx->build_ovf = ovf;
    CK(cudaEventRecord(ctx->ev_free[ctx->ph_staging_sel], st));   // last read of the staging buffer
    ctx->launches += 17;
    CK(cudaGetLastError());
  } else {
    CK(cudaMemsetAsync(ctx->bounds.p, 0, 7 * sizeof(float), st));
    CK(cudaMemsetAsync(ctx->cell_start.p, 0, ((size_t)n_keys + 1) * 4, st));
  }
  Tree T{};
  T.n = n;
  ctx->grid = G;
  int rc = points_built(ctx, T, radius, gvpm_ctx::ACCEL_FRUSTUM, true, n);
  if (rc) return rc;
  if (n_kept) {   // photons some ray can reach = everything in front of the DROP bucket (one read-back, only on request)
    CK(cudaMemcpyAsync(ctx->pair_count_host, ctx->cell_start.as<uint32_t>() + n_keys - 1, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    ctx->n_kept = *(const uint32_t *)ctx->pair_count_host;
    *n_kept = ctx->n_kept;
  }
  return GVPM_OK;
}

extern "C" {

int gvpm_build_points(gvpm_ctx *ctx, float radius) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (!ctx->photons_loaded) return fail(ctx, GVPM_ERR_INVALID, "no photons uploaded");
  if (!(radius > 0.f)) return fail(ctx, GVPM_ERR_INVALID, "radius must be positive");
  cudaSetDevice(ctx->device);
  const uint32_t n = ctx->n_photons;
  cudaStream_t st = ctx->stream;
  CK(cudaEventRecord(ctx->ev[0], st));
  Tree T{};
  uint32_t total = 0;
  int rc = bvh_levels(ctx, T, n, "too many photons", &total);
  if (rc) return rc;
  const int levels = T.levels;
  if (n > 0) {
    rc = reserve_sort(ctx, n);
    if (rc) return rc;
    CK(ctx->planes.reserve(16 * (size_t)n));
    CK(ctx->orig.reserve(4 * (size_t)n));
    CK(ctx->box_lo.reserve(16 * (size_t)total));
    CK(ctx->box_hi.reserve(16 * (size_t)total));
    const bool direct = ctx->photons_direct;
    PhotonStaging S{};
    if (!direct) S = staging_ptrs<PhotonSoA>(ctx->ph_staging.p, n);
    const float *pos = direct ? (const float *)ctx->records() : S.pos;
    const uint32_t stride = direct ? 32u : 3u;
    CK(ctx->bounds_partial.reserve((size_t)bounds_blocks(n) * 6 * sizeof(float)));
    launch_bounds(pos, n, ctx->bounds_partial.as<float>(), ctx->bounds.as<float>(), st, stride);
    launch_morton(pos, n, ctx->bounds.as<float>(), ctx->keys_in.as<uint32_t>(), ctx->vals_in.as<uint32_t>(), st, stride);
    CK(run_sort_bits(ctx->sort_temp.p, ctx->sort_temp.cap, ctx->keys_in.as<uint32_t>(), ctx->keys_out.as<uint32_t>(),
                     ctx->vals_in.as<uint32_t>(), ctx->vals_out.as<uint32_t>(), n, kHilbertBits, st));
    if (!direct) CK(ctx->aos.reserve(128 * (size_t)n));
    launch_pack_sorted(S, ctx->records(), ctx->vals_out.as<uint32_t>(), n, ctx->planes.as<float4>(),
                       ctx->orig.as<uint32_t>(), st, direct);
    CK(cudaEventRecord(ctx->ev_free[ctx->ph_staging_sel], st));   // last read of the staging buffer
    float4 *lo = ctx->box_lo.as<float4>(), *hi = ctx->box_hi.as<float4>();
    launch_leaf_boxes(ctx->planes.as<float4>(), n, T.cnt[0], radius, lo, hi, st);
    for (int l = 1; l < levels; ++l)
      launch_level_boxes(lo + T.off[l - 1], hi + T.off[l - 1], T.cnt[l - 1], T.cnt[l], lo + T.off[l], hi + T.off[l], st);
    ctx->launches += 6 + (levels - 1) + 4;  // + the radix sort's own passes (library, ~4 launches)
    CK(cudaGetLastError());
  } else {
    CK(cudaMemsetAsync(ctx->bounds.p, 0, 7 * sizeof(float), st));
  }
  T.lo = ctx->box_lo.as<float4>();
  T.hi = ctx->box_hi.as<float4>();
  return points_built(ctx, T, radius, gvpm_ctx::ACCEL_BVH, false, n);
}

int gvpm_build_points_for_rays(gvpm_ctx *ctx, float radius, uint32_t *n_kept) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (!ctx->photons_loaded) return fail(ctx, GVPM_ERR_INVALID, "no photons uploaded");
  if (!ctx->rays_loaded) return fail(ctx, GVPM_ERR_INVALID, "gvpm_build_points_for_rays needs the rays first (gvpm_upload_rays)");
  if (!(radius > 0.f)) return fail(ctx, GVPM_ERR_INVALID, "radius must be positive");
  cudaSetDevice(ctx->device);
  if (!ctx->force_bvh) {
    int rc = analyse_rays(ctx);
    if (rc) return rc;
    // concurrent rays whose common point is sharp compared with the search radius: perspective grid, no hierarchy
    if (ctx->pin.concurrent && ctx->pin.delta <= 0.25f * radius) return build_frustum(ctx, radius, n_kept);
  }
  return build_pruned_bvh(ctx, radius, n_kept);
}

}  // extern "C"
