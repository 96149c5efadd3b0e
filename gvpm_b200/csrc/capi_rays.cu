// capi_rays.cu — ray staging, commit, upload and on-device camera-ray generation.
#include "capi_internal.cuh"

extern "C" {

int gvpm_ray_staging(gvpm_ctx *ctx, size_t n, void **dev, size_t *bytes) {
  if (!ctx || n > 0xfffffff0u) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const SoaLayout<RaySoA> L(n);
  CK(ctx->ray_staging.reserve(L.bytes ? L.bytes : 256));
  ctx->n_rays = (uint32_t)n;
  ctx->rays_loaded = false;
  ++ctx->rays_gen;
  ++ctx->state_gen;
  if (dev) *dev = ctx->ray_staging.p;
  if (bytes) *bytes = L.bytes;
  return GVPM_OK;
}

int gvpm_commit_rays(gvpm_ctx *ctx) {
  if (!ctx) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const uint32_t n = ctx->n_rays;
  CK(ctx->rays.reserve((size_t)n * GVPM_RAY_FLOAT4 * 16 + 256));
  CK(ctx->out.reserve((size_t)n * GVPM_OUT_FLOATS * 4 + 256));
  CK(ctx->counts.reserve((size_t)n * 8 + 256));
  if (n > 0) {
    launch_pack_rays(staging_ptrs<RaySoA>(ctx->ray_staging.p, n), n, ctx->rays.as<float4>(), ctx->stream);
    ctx->launches += 1;
    CK(cudaGetLastError());
  }
  ctx->rays_loaded = true;
  return GVPM_OK;
}

int gvpm_upload_rays(gvpm_ctx *ctx, const gvpm_ray_soa *r, size_t n) {
  if (!ctx || (n && !r)) return GVPM_ERR_INVALID;
  int rc = gvpm_ray_staging(ctx, n, nullptr, nullptr);
  if (rc) return rc;
  if (n > 0) {
    rc = copy_soa<RaySoA>(ctx, *r, ctx->ray_staging.p, n, 0, 0, n, ctx->stream);
    if (rc) return rc;
  }
  return gvpm_commit_rays(ctx);
}

int gvpm_generate_rays(gvpm_ctx *ctx, const gvpm_box_scene *scene, const gvpm_pinhole_camera *cam, uint64_t seed,
                       int block, int y0, int y1, float epsilon) {
  if (!ctx || !scene || !cam) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  int rc = check_scene(ctx, scene);
  if (rc) return rc;
  const bool zorder = block < 0;
  const int bs = zorder ? -block : block;
  if (bs < 1 || bs > 32 || (zorder && (bs & (bs - 1)))) return fail(ctx, GVPM_ERR_INVALID, "block must be in [1, 32] (a power of two for Z-order)");
  if (cam->film_w <= 0 || cam->film_h <= 0 || y0 < 0 || y1 > cam->film_h || y0 > y1)
    return fail(ctx, GVPM_ERR_INVALID, "bad film size / row range");
  const size_t n = (size_t)cam->film_w * (size_t)(y1 - y0);
  void *dev = nullptr;
  rc = gvpm_ray_staging(ctx, n, &dev, nullptr);
  if (rc) return rc;
  if (n) {
    const RayStaging S = staging_ptrs<RaySoA>(dev, n);
    RayGenParams P{};
    P.scene = *scene;
    P.cam = *cam;
    P.seed = seed;
    P.block = bs;
    P.zorder = zorder ? 1 : 0;
    P.y0 = y0;
    P.y1 = y1;
    P.epsilon = epsilon;
    writable_view<RaySoA>(P.o, S);
    launch_generate_rays(P, ctx->stream);
    ctx->launches += 1;
    CK(cudaGetLastError());
  }
  rc = gvpm_commit_rays(ctx);
  if (rc) return rc;
  ctx->pixel_rays_gen = ctx->rays_gen;   // one ray per pixel of rows [y0, y1): gvpm_accum_add needs no sort
  // The rays of a pinhole are concurrent by construction: what analyse_rays would measure on the device (and read back)
  // follows from the camera.  Every ray is pos + t * dir up to the rounding of the entry point (a few ulp of the
  // coordinates, bounded here by 4e-6 * (1 + |pos|)); projected directions span [-tx, tx] x rows [y0, y1).
  {
    gvpm_ctx::RayFit &F = ctx->pin;
    const float tx = cam->tan_half_fov_x, ty = tx * (float)cam->film_h / (float)cam->film_w;
    for (int k = 0; k < 3; ++k) { F.C[k] = cam->pos[k]; F.m[k] = F.u[k] = F.v[k] = 0.f; }
    F.m[2] = 1.f; F.u[0] = 1.f; F.v[1] = 1.f;
    F.xmin = -tx * 1.0001f; F.xmax = tx * 1.0001f;
    F.ymin = ((float)y0 / (float)cam->film_h - 0.5f) * 2.f * ty;
    F.ymax = ((float)y1 / (float)cam->film_h - 0.5f) * 2.f * ty;
    const float ypad = 1e-4f * ty + 1e-7f;
    F.ymin -= ypad; F.ymax += ypad;
    const float amax = std::max(std::fabs(cam->pos[0]), std::max(std::fabs(cam->pos[1]), std::fabs(cam->pos[2])));
    F.delta = 4e-6f * (1.f + amax);
    F.cosmin = 1.f / std::sqrt(1.f + tx * tx + ty * ty);
    F.count = (float)n;
    F.concurrent = n > 0 && F.cosmin > 0.35f;
    ctx->pin_gen = ctx->rays_gen;
    ctx->occ_ready = false;
  }
  return GVPM_OK;
}

}  // extern "C"

// The look-at frame: f = normalize(forward), r = normalize(cross(up, f)), u = cross(f, r), each operation rounded on its own
// in this order (the CPU restatement forms the same).  False when forward is zero or parallel to up.
__attribute__((optimize("fp-contract=off"))) static bool lookat_frame(const gvpm_lookat_camera &c, LookatCam &L) {
  auto unit = [](float &x, float &y, float &z) {
    const float l = std::sqrt((x * x + y * y) + z * z);
    if (!(l > 0.f) || !std::isfinite(l)) return false;
    const float il = 1.0f / l;
    x = x * il; y = y * il; z = z * il;
    return true;
  };
  float f[3] = {c.forward[0], c.forward[1], c.forward[2]};
  if (!unit(f[0], f[1], f[2])) return false;
  float r[3] = {c.up[1] * f[2] - c.up[2] * f[1], c.up[2] * f[0] - c.up[0] * f[2], c.up[0] * f[1] - c.up[1] * f[0]};
  if (!unit(r[0], r[1], r[2])) return false;
  const float u[3] = {f[1] * r[2] - f[2] * r[1], f[2] * r[0] - f[0] * r[2], f[0] * r[1] - f[1] * r[0]};
  for (int a = 0; a < 3; ++a) { L.pos[a] = c.pos[a]; L.f[a] = f[a]; L.r[a] = r[a]; L.u[a] = u[a]; }
  return true;
}

extern "C" {

int gvpm_generate_rays_mesh(gvpm_ctx *ctx, const gvpm_lookat_camera *cam, uint64_t seed, int block, int y0, int y1,
                            float epsilon) {
  if (!ctx || !cam) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (!ctx->mesh.ready) return fail(ctx, GVPM_ERR_INVALID, "no mesh scene: gvpm_set_trace_mesh first");
  const bool zorder = block < 0;
  const int bs = zorder ? -block : block;
  if (bs < 1 || bs > 32 || (zorder && (bs & (bs - 1)))) return fail(ctx, GVPM_ERR_INVALID, "block must be in [1, 32] (a power of two for Z-order)");
  if (cam->film_w <= 0 || cam->film_h <= 0 || y0 < 0 || y1 > cam->film_h || y0 > y1)
    return fail(ctx, GVPM_ERR_INVALID, "bad film size / row range");
  if (!(cam->tan_half_fov_x > 0.f) || !std::isfinite(cam->tan_half_fov_x))
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_lookat_camera: tan_half_fov_x must be positive and finite");
  MeshRayGenParams P{};
  for (int a = 0; a < 3; ++a)
    if (!std::isfinite(cam->pos[a])) return fail(ctx, GVPM_ERR_INVALID, "gvpm_lookat_camera: pos is not finite");
  if (!lookat_frame(*cam, P.cam))
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_lookat_camera: forward is zero or parallel to up");
  const gvpm_ctx::TraceMesh &M = ctx->mesh;
  bool inside = true;
  for (int a = 0; a < 3; ++a) inside = inside && cam->pos[a] > M.lo[a] && cam->pos[a] < M.hi[a];
  P.cam.tan_half_fov_x = cam->tan_half_fov_x;
  P.cam.film_w = cam->film_w;
  P.cam.film_h = cam->film_h;
  P.cam.inside_medium = inside ? 1 : 0;
  const size_t n = (size_t)cam->film_w * (size_t)(y1 - y0);
  void *dev = nullptr;
  int rc = gvpm_ray_staging(ctx, n, &dev, nullptr);
  if (rc) return rc;
  if (n) {
    P.scene = mesh_view(ctx);
    P.seed = seed;
    P.block = bs;
    P.zorder = zorder ? 1 : 0;
    P.y0 = y0;
    P.y1 = y1;
    P.epsilon = epsilon;
    writable_view<RaySoA>(P.o, staging_ptrs<RaySoA>(dev, n));
    launch_generate_rays(P, ctx->stream);
    ctx->launches += 1;
    CK(cudaGetLastError());
  }
  rc = gvpm_commit_rays(ctx);
  if (rc) return rc;
  ctx->pixel_rays_gen = ctx->rays_gen;   // one ray per pixel of rows [y0, y1): gvpm_accum_add needs no sort
  // the ray fit of the perspective grid is measured on the device (analyse_rays), as for uploaded rays
  return GVPM_OK;
}

}  // extern "C"
