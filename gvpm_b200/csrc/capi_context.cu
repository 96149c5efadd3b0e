// capi_context.cu — context lifetime, scene constants (medium, config, occluders and their any-hit path), timings and
// small queries.
#include "capi_internal.cuh"

static std::string g_create_error;

void triangle_planes(const float *tri, size_t n_tri, std::vector<float> &planes, std::vector<float> &aux) {
  planes.assign(4 * n_tri, 0.f);
  aux.assign(2 * n_tri, 0.f);
  for (size_t t = 0; t < n_tri; ++t) {
    const float *p = tri + 9 * t;
    double e1[3], e2[3], n[3];
    for (int a = 0; a < 3; ++a) { e1[a] = (double)p[3 + a] - p[a]; e2[a] = (double)p[6 + a] - p[a]; }
    n[0] = e1[1] * e2[2] - e1[2] * e2[1];
    n[1] = e1[2] * e2[0] - e1[0] * e2[2];
    n[2] = e1[0] * e2[1] - e1[1] * e2[0];
    double len = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    {
      // rounding slack of the strict ray-triangle parameter (bre_device.cuh occluded()): ~16 eps * |e1||e2|/|e1 x e2|
      // per unit of |o - p0| / |n.d|; aux = (that coefficient, largest |vertex coordinate|)
      const double l1 = std::sqrt(e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2]),
                   l2 = std::sqrt(e2[0] * e2[0] + e2[1] * e2[1] + e2[2] * e2[2]);
      double vmag = 0;
      for (int a = 0; a < 9; ++a) vmag = std::max(vmag, (double)std::fabs(p[a]));
      aux[2 * t] = (float)(len > 0 ? 2e-6 * (l1 * l2 / len) : 0.0);
      aux[2 * t + 1] = (float)vmag;
    }
    if (len > 0) {
      for (int a = 0; a < 3; ++a) n[a] /= len;
      planes[4 * t] = (float)n[0]; planes[4 * t + 1] = (float)n[1]; planes[4 * t + 2] = (float)n[2];
      planes[4 * t + 3] = (float)(-(n[0] * p[0] + n[1] * p[1] + n[2] * p[2]));
    } else {
      planes[4 * t] = planes[4 * t + 1] = planes[4 * t + 2] = planes[4 * t + 3] = 0.f;  // never culled
    }
  }
}

extern "C" {

int gvpm_abi_version(void) { return GVPM_ABI_VERSION; }

int gvpm_ctx_create(int device, gvpm_ctx **out) {
  if (!out) return GVPM_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_create_error = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count = 0") +
                     " (gvpm_b200 has no CPU fallback)";
    return GVPM_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= ndev) { g_create_error = "device index out of range"; return GVPM_ERR_INVALID; }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    g_create_error = cudaGetErrorString(e);
    return GVPM_ERR_CUDA;
  }
  if (prop.major != 10) {
    g_create_error = "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                     "; this library is built for sm_100a only";
    return GVPM_ERR_NO_DEVICE;
  }
  if ((e = cudaSetDevice(device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return GVPM_ERR_CUDA; }
  gvpm_ctx *ctx = new gvpm_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    g_create_error = cudaGetErrorString(e);
    delete ctx;
    return GVPM_ERR_CUDA;
  }
  for (auto &ev : ctx->ev) cudaEventCreate(&ev);
  cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking);
  for (auto &ev : ctx->pipe_ev) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  for (int b = 0; b < 2; ++b) {
    cudaEventCreateWithFlags(&ctx->ev_free[b], cudaEventDisableTiming | cudaEventInterprocess);
    cudaEventCreateWithFlags(&ctx->ev_pushed[b], cudaEventDisableTiming | cudaEventInterprocess);
  }
  for (auto &ps : ctx->push_streams) cudaStreamCreateWithFlags(&ps, cudaStreamNonBlocking);
  {
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    cudaStreamCreateWithPriority(&ctx->push_kernel_stream, cudaStreamNonBlocking, hi);
  }
  for (auto &ev : ctx->push_ev) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  ctx->work_counter.reserve(256);
  // [0,8): pair / kept-photon counters, the solver's 3-float residual; [8,16): async gather ring; [16,48): ray chunks
  cudaHostAlloc((void **)&ctx->pair_count_host, 48 * sizeof(unsigned long long), cudaHostAllocDefault);
  memset(ctx->pair_count_host, 0, 48 * sizeof(unsigned long long));
  for (auto &g : ctx->ring) cudaEventCreateWithFlags(&g.done, cudaEventDisableTiming);
  cudaHostAlloc((void **)&ctx->pin_host, 128, cudaHostAllocDefault);
  { const char *e = getenv("GVPM_ACCEL"); ctx->force_bvh = e && !strcmp(e, "bvh"); }
  cudaHostAlloc((void **)&ctx->sample_stats_host, 64, cudaHostAllocDefault);
  memset(ctx->sample_stats_host, 0, 64);
  ctx->bounds.reserve(256);
  ctx->bounds_partial.reserve(1024 * 6 * sizeof(float));
  *out = ctx;
  return GVPM_OK;
}

int gvpm_ctx_destroy(gvpm_ctx *ctx) {
  if (!ctx) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (int p = 0; p < ctx->disp.n_peers; ++p)
    if (ctx->disp.peer_mapped[p]) {
      for (int b = 0; b < 2; ++b) if (ctx->disp.peer_inbox[b][p]) cudaIpcCloseMemHandle(ctx->disp.peer_inbox[b][p]);
      if (ctx->disp.peer_ctrl[p]) cudaIpcCloseMemHandle(ctx->disp.peer_ctrl[p]);
    }
  for (int b = 0; b < 2; ++b) if (ctx->disp.grids_host[b]) cudaFreeHost(ctx->disp.grids_host[b]);
  for (void *q : ctx->disp.shared_opened) cudaIpcCloseMemHandle(q);
  for (void *q : ctx->disp.shared_owned) cudaFree(q);
  if (ctx->disp.ev_src) cudaEventDestroy(ctx->disp.ev_src);
  if (ctx->pair_count_host) cudaFreeHost(ctx->pair_count_host);
  if (ctx->sample_stats_host) cudaFreeHost(ctx->sample_stats_host);
  if (ctx->pin_host) cudaFreeHost(ctx->pin_host);
  for (auto &g : ctx->ring) if (g.done) cudaEventDestroy(g.done);
  for (auto &ps : ctx->push_streams) if (ps) { cudaStreamSynchronize(ps); cudaStreamDestroy(ps); }
  if (ctx->push_kernel_stream) { cudaStreamSynchronize(ctx->push_kernel_stream); cudaStreamDestroy(ctx->push_kernel_stream); }
  for (auto &ev : ctx->push_ev) if (ev) cudaEventDestroy(ev);
  for (int b = 0; b < 2; ++b) {
    for (int p = 0; p < ctx->n_peers; ++p) {
      if (p == ctx->peer_self) continue;
      if (ctx->peer_staging[b][p]) cudaIpcCloseMemHandle(ctx->peer_staging[b][p]);
      if (ctx->peer_free[b][p]) cudaEventDestroy(ctx->peer_free[b][p]);
      if (ctx->peer_pushed[b][p]) cudaEventDestroy(ctx->peer_pushed[b][p]);
    }
    if (ctx->ev_free[b]) cudaEventDestroy(ctx->ev_free[b]);
    if (ctx->ev_pushed[b]) cudaEventDestroy(ctx->ev_pushed[b]);
  }
  for (auto &ev : ctx->ev) if (ev) cudaEventDestroy(ev);
  for (auto &ev : ctx->pipe_ev) if (ev) cudaEventDestroy(ev);
  if (ctx->copy_in) { cudaStreamSynchronize(ctx->copy_in); cudaStreamDestroy(ctx->copy_in); }
  if (ctx->copy_out) { cudaStreamSynchronize(ctx->copy_out); cudaStreamDestroy(ctx->copy_out); }
  cudaStreamDestroy(ctx->stream);
  delete ctx;   // the DevBufs free their allocations
  return GVPM_OK;
}

const char *gvpm_last_error(const gvpm_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int gvpm_sync(gvpm_ctx *ctx) {
  if (!ctx) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  CK(cudaStreamSynchronize(ctx->stream));
  return pending_check(ctx, true);   // an asynchronous gather whose pair list overflowed is re-run here
}

void *gvpm_stream(gvpm_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

int gvpm_set_medium(gvpm_ctx *ctx, const gvpm_medium *m) {
  if (!ctx || !m) return GVPM_ERR_INVALID;
  const float st0 = m->sigma_s[0] + m->sigma_a[0];
  for (int i = 1; i < 3; ++i)
    if (m->sigma_s[i] + m->sigma_a[i] != st0)
      // the reference aborts the same way: homogeneous.cpp:188-201
      return fail(ctx, GVPM_ERR_UNSUPPORTED, "sigma_t must be equal across channels (balance strategy)");
  if (m->phase_type != GVPM_PHASE_ISOTROPIC && m->phase_type != GVPM_PHASE_HG)
    return fail(ctx, GVPM_ERR_UNSUPPORTED, "phase function must be isotropic or hg");
  ctx->medium = *m;
  ctx->have_medium = true;
  ++ctx->state_gen;
  return GVPM_OK;
}

int gvpm_set_config(gvpm_ctx *ctx, const gvpm_config *c) {
  if (!ctx || !c) return GVPM_ERR_INVALID;
  if (c->use_shift_null && !c->kernel_3d && !c->sppm_primal)
    // gvpm_struct.h:305-308: "Not possible to shift null without using 3D kernel"
    return fail(ctx, GVPM_ERR_UNSUPPORTED, "useShiftNull requires the 3D kernel");
  ctx->cfg = *c;
  ctx->have_cfg = true;
  ++ctx->state_gen;
  return GVPM_OK;
}

int gvpm_set_occluders(gvpm_ctx *ctx, const float *tri_xyz, size_t n_tri) {
  if (!ctx || (n_tri && !tri_xyz)) return GVPM_ERR_INVALID;
  if (n_tri > GVPM_MAX_OCCLUDERS)
    return fail(ctx, GVPM_ERR_INVALID, "more than GVPM_MAX_OCCLUDERS (2^24) occluder triangles");
  cudaSetDevice(ctx->device);
  ctx->n_tri = (uint32_t)n_tri;
  ctx->occ_built = false;
  ++ctx->state_gen;
  if (n_tri == 0) return GVPM_OK;
  std::vector<float> planes, aux;
  triangle_planes(tri_xyz, n_tri, planes, aux);
  CK(ctx->tri.reserve(9 * n_tri * sizeof(float)));
  CK(ctx->tri_plane.reserve(4 * n_tri * sizeof(float)));
  CK(ctx->tri_aux.reserve(2 * n_tri * sizeof(float)));
  CK(cudaMemcpyAsync(ctx->tri_aux.p, aux.data(), 2 * n_tri * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->tri.p, tri_xyz, 9 * n_tri * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->tri_plane.p, planes.data(), 4 * n_tri * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (occluder_use_bvh(ctx)) {
    const int rc = build_occluder_bvh(ctx);
    if (rc) ctx->n_tri = 0;   // no half-built set: the occluders are cleared
    return rc;
  }
  return GVPM_OK;
}

int gvpm_set_occluder_accel(gvpm_ctx *ctx, int mode) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (mode != GVPM_OCC_AUTO && mode != GVPM_OCC_LIST && mode != GVPM_OCC_BVH)
    return fail(ctx, GVPM_ERR_INVALID, "occluder accel must be GVPM_OCC_AUTO, GVPM_OCC_LIST or GVPM_OCC_BVH");
  ctx->occ_accel = mode;   // both paths give the same any-hit: the gathers' results do not change
  if (occluder_use_bvh(ctx) && !ctx->occ_built) {
    cudaSetDevice(ctx->device);
    return build_occluder_bvh(ctx);
  }
  return GVPM_OK;
}

int gvpm_occluder_accel_kind(const gvpm_ctx *ctx) {
  if (!ctx) return 0;
  return occluder_use_bvh(ctx) ? GVPM_OCC_BVH : GVPM_OCC_LIST;
}

int gvpm_occluded(gvpm_ctx *ctx, const float *o, const float *d, const float *mint, const float *maxt, size_t n,
                  uint8_t *hit) {
  if (!ctx || (n && (!o || !d || !mint || !maxt || !hit))) return GVPM_ERR_INVALID;
  if (n > 0xffffffffull) return fail(ctx, GVPM_ERR_INVALID, "more than 2^32 - 1 rays");
  if (n == 0) return GVPM_OK;
  cudaSetDevice(ctx->device);
  const size_t o_d = align256(12 * n), o_mint = o_d + align256(12 * n), o_maxt = o_mint + align256(4 * n),
               o_hit = o_maxt + align256(4 * n);
  CK(ctx->occ_query.reserve(o_hit + n));
  char *q = ctx->occ_query.as<char>();
  CK(cudaMemcpyAsync(q, o, 12 * n, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(q + o_d, d, 12 * n, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(q + o_mint, mint, 4 * n, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(q + o_maxt, maxt, 4 * n, cudaMemcpyHostToDevice, ctx->stream));
  GatherParams P;
  memset(&P, 0, sizeof(P));
  occluder_params(ctx, P);
  launch_occluded(P, P.occ_nodes != nullptr, (const float *)q, (const float *)(q + o_d), (const float *)(q + o_mint),
                  (const float *)(q + o_maxt), (uint32_t)n, (uint8_t *)(q + o_hit), ctx->stream);
  CK(cudaGetLastError());
  ++ctx->launches;
  CK(cudaMemcpyAsync(hit, q + o_hit, n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GVPM_OK;
}

int gvpm_measure_read_bandwidth(gvpm_ctx *ctx, size_t bytes, int reps, double *gb_per_s) {
  if (!ctx || !gb_per_s || bytes < 4096 || bytes > (1ull << 32) || reps < 1) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  CK(ctx->poisson_io.reserve(bytes + 256));
  CK(cudaMemsetAsync(ctx->poisson_io.p, 1, bytes + 256, ctx->stream));
  unsigned *sink = (unsigned *)(ctx->poisson_io.as<char>() + bytes);
  launch_l2_read(ctx->poisson_io.p, bytes, 2, sink, ctx->sm_count, ctx->stream);   // warm: the buffer is in L2 (if it fits)
  CK(cudaEventRecord(ctx->ev[2], ctx->stream));
  launch_l2_read(ctx->poisson_io.p, bytes, reps, sink, ctx->sm_count, ctx->stream);
  CK(cudaEventRecord(ctx->ev[3], ctx->stream));
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]));
  ctx->launches += 2;
  *gb_per_s = (double)(bytes / 16 * 16) * reps / ((double)ms * 1e-3) / 1e9;
  return GVPM_OK;
}

int gvpm_read_device(gvpm_ctx *ctx, const void *dev, void *host, size_t bytes) {
  if (!ctx || (bytes && (!dev || !host))) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (bytes) CK(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GVPM_OK;
}

int gvpm_staging_peek(gvpm_ctx *ctx, int which, void **dev, size_t *count) {
  if (!ctx || !dev || which < 0 || which > 4) return GVPM_ERR_INVALID;
  const DevBuf *buf[5] = {&ctx->ph_staging, &ctx->ray_staging, &ctx->beam_staging, &ctx->plane_staging, &ctx->sample_staging};
  const size_t n[5] = {ctx->n_photons, ctx->n_rays, ctx->n_beams, ctx->n_planes, ctx->n_samples};
  *dev = buf[which]->p;
  if (count) *count = n[which];
  return GVPM_OK;
}

int gvpm_accel_kind(const gvpm_ctx *ctx) { return ctx ? ctx->accel : 0; }

int gvpm_frustum_grid(gvpm_ctx *ctx, void *grid, size_t grid_bytes, uint32_t *cell_start, size_t cap, size_t *n_entries) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (grid_bytes != sizeof(FrustumGrid)) return fail(ctx, GVPM_ERR_INVALID, "grid_bytes is not sizeof(FrustumGrid)");
  if (!ctx->built || ctx->accel != gvpm_ctx::ACCEL_FRUSTUM)
    return fail(ctx, GVPM_ERR_INVALID, "no perspective grid built (gvpm_build_points_for_rays over concurrent rays)");
  const FrustumGrid &G = ctx->grid;
  const size_t n = (size_t)(G.parity_split ? 2u : 1u) * G.n_cells + 3;   // + NEAR, DROP and the end
  if (grid) memcpy(grid, &G, sizeof(FrustumGrid));
  if (n_entries) *n_entries = n;
  if (cell_start) {
    if (cap < n) return fail(ctx, GVPM_ERR_INVALID, "cell_start holds fewer than *n_entries entries");
    cudaSetDevice(ctx->device);
    CK(cudaMemcpyAsync(cell_start, ctx->cell_start.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return GVPM_OK;
}

int gvpm_set_view_direction(gvpm_ctx *ctx, const float dir[3]) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (dir) {
    const double l = std::sqrt((double)dir[0] * dir[0] + (double)dir[1] * dir[1] + (double)dir[2] * dir[2]);
    if (!(l > 0.0) || !std::isfinite(l)) return fail(ctx, GVPM_ERR_INVALID, "view direction must be a non-zero vector");
    for (int k = 0; k < 3; ++k) ctx->view_dir[k] = dir[k];
  }
  ctx->have_view_dir = dir != nullptr;
  ctx->pin_gen = ~0ull;   // the rays are analysed again with the new axis
  return GVPM_OK;
}

float gvpm_last_poisson_ms(const gvpm_ctx *ctx) { return ctx ? ctx->poisson_ms : 0.f; }

int gvpm_last_timings(gvpm_ctx *ctx, float *build_ms, float *gather_ms) {
  if (!ctx) return GVPM_ERR_INVALID;
  CK(cudaStreamSynchronize(ctx->stream));
  { int rc = pending_check(ctx, true); if (rc) return rc; }
  if (ctx->timed_build) CK(cudaEventElapsedTime(&ctx->build_ms, ctx->ev[0], ctx->ev[1]));
  if (ctx->timed_gather) CK(cudaEventElapsedTime(&ctx->gather_ms, ctx->ev[2], ctx->ev[3]));
  if (build_ms) *build_ms = ctx->build_ms;
  if (gather_ms) *gather_ms = ctx->gather_ms;
  return GVPM_OK;
}

int gvpm_last_gather_detail(gvpm_ctx *ctx, float *traverse_ms, float *shade_ms, uint64_t *pairs) {
  if (!ctx) return GVPM_ERR_INVALID;
  CK(cudaStreamSynchronize(ctx->stream));
  { int rc = pending_check(ctx, true); if (rc) return rc; }
  float t = 0.f, s = 0.f;
  if (ctx->timed_gather && ctx->n_rays && ctx->split_timed) {
    CK(cudaEventElapsedTime(&t, ctx->ev[4], ctx->ev[5]));
    CK(cudaEventElapsedTime(&s, ctx->ev[5], ctx->ev[3]));
  }
  if (traverse_ms) *traverse_ms = t;
  if (shade_ms) *shade_ms = s;
  if (pairs) *pairs = ctx->last_pairs;
  return GVPM_OK;
}

uint64_t gvpm_launch_count(const gvpm_ctx *ctx) { return ctx ? ctx->launches : 0; }

}  // extern "C"
