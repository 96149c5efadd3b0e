// capi_accum.cu — the per-pixel accumulators of a progressive render, kept on the device (gvpm_accum_*): add the
// per-ray results of the gathers, fold them into the APA running mean (or the plain sum of G-VPM), hand them to the
// gradient and the Poisson solve.  Kernels in accumulate.cu.
#include "capi_internal.cuh"

static int accum_check(gvpm_ctx *ctx, const char *what) {
  if (!ctx->accum.ready) return fail(ctx, GVPM_ERR_INVALID, std::string(what) + ": gvpm_accum_reset has not been called");
  return GVPM_OK;
}

extern "C" {

int gvpm_accum_reset(gvpm_ctx *ctx, int w, int h, int channels, int apa) {
  if (!ctx) return GVPM_ERR_INVALID;
  if (w <= 0 || h <= 0 || (uint64_t)w * (uint64_t)h >= (1ull << 30))
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_accum_reset: w, h must be positive and w * h below 2^30");
  if (channels != 3 && channels != GVPM_OUT_FLOATS)
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_accum_reset: channels must be 27 (gvpm) or 3 (sppm)");
  cudaSetDevice(ctx->device);
  gvpm_ctx::Accum &A = ctx->accum;
  A.ready = false;
  const size_t npix = (size_t)w * h, bytes = npix * channels * sizeof(float);
  CK(A.acc.reserve(bytes));
  CK(A.smoke.reserve(npix));
  CK(cudaMemsetAsync(A.acc.p, 0, bytes, ctx->stream));
  CK(cudaMemsetAsync(A.smoke.p, 0, npix, ctx->stream));
  if (apa) {
    CK(A.pix.reserve(bytes));
    CK(cudaMemsetAsync(A.pix.p, 0, bytes, ctx->stream));
  }
  A.w = w;
  A.h = h;
  A.channels = channels;
  A.apa = apa != 0;
  A.total = 0;
  A.ready = true;
  return GVPM_OK;
}

int gvpm_accum_add(gvpm_ctx *ctx) {
  if (!ctx) return GVPM_ERR_INVALID;
  int rc = accum_check(ctx, "gvpm_accum_add");
  if (rc) return rc;
  cudaSetDevice(ctx->device);
  // an asynchronous gather whose pair list overflowed is run again here, before its output is read
  rc = pending_check(ctx, true);
  if (rc) return rc;
  if (ctx->out_state == gvpm_ctx::OUT_ELSEWHERE)
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_accum_add: the last gather wrote to caller memory (gvpm_gather_bre_into), "
                                       "not to the context's output");
  if (ctx->out_state == gvpm_ctx::OUT_NONE || ctx->out_gen != ctx->rays_gen)
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_accum_add: no gather has run on the current ray set");
  if (ctx->out_state == gvpm_ctx::OUT_ADDED)
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_accum_add: the output of the last gather has already been added");
  gvpm_ctx::Accum &A = ctx->accum;
  if ((uint32_t)A.channels > ctx->out_stride)
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_accum_add: the last gather wrote fewer floats per ray than the accumulator "
                                       "has channels");
  const uint32_t n = ctx->n_rays;
  const RayStaging S = staging_ptrs<RaySoA>(ctx->ray_staging.p, n);
  float *dst = A.apa ? A.pix.as<float>() : A.acc.as<float>();
  const float *out = ctx->out.as<float>();
  if (ctx->pixel_rays_gen == ctx->rays_gen) {
    launch_accum_scatter(out, ctx->out_stride, S.px, S.py, n, A.w, A.h, A.channels, dst, A.smoke.as<uint8_t>(),
                         ctx->sm_count, ctx->stream);
    ctx->launches += n ? 1 : 0;
  } else if (n) {
    // several records may share a pixel: sort (pixel, ray index) pairs - radix sort is stable, so each pixel's rays
    // stay in ray order - and add each pixel's run in order
    const size_t words = align256((size_t)n * 4);
    const size_t temp = sort_temp_bytes(n);
    CK(A.keys.reserve(4 * words + temp));
    char *k = A.keys.as<char>();
    uint32_t *kin = (uint32_t *)k, *vin = (uint32_t *)(k + words), *kout = (uint32_t *)(k + 2 * words),
             *vout = (uint32_t *)(k + 3 * words);
    const uint32_t npix = (uint32_t)A.w * (uint32_t)A.h;
    int bits = 1;
    while (bits < 32 && (npix >> bits)) ++bits;   // keys go up to npix (rays outside the film)
    launch_accum_keys(S.px, S.py, n, A.w, A.h, kin, vin, ctx->stream);
    CK(run_sort_bits(k + 4 * words, temp, kin, kout, vin, vout, n, bits, ctx->stream));
    launch_accum_runs(out, ctx->out_stride, kout, vout, n, npix, A.channels, dst, A.smoke.as<uint8_t>(), ctx->sm_count,
                      ctx->stream);
    ctx->launches += 3;
  }
  CK(cudaGetLastError());
  ctx->out_state = gvpm_ctx::OUT_ADDED;
  return GVPM_OK;
}

int gvpm_accum_fold(gvpm_ctx *ctx, int it, uint64_t n_paths) {
  if (!ctx) return GVPM_ERR_INVALID;
  int rc = accum_check(ctx, "gvpm_accum_fold");
  if (rc) return rc;
  if (it < 1 || n_paths < 1) return fail(ctx, GVPM_ERR_INVALID, "gvpm_accum_fold: it and n_paths must be at least 1");
  gvpm_ctx::Accum &A = ctx->accum;
  if (!A.apa) {
    A.total += n_paths;
    return GVPM_OK;
  }
  cudaSetDevice(ctx->device);
  // the two reciprocals and the conversions formed as the mirror forms them (Spectrum's operators multiply by 1 / x)
  const float rnb = 1.0f / (float)n_paths, rit = 1.0f / (float)it, itm1 = (float)(it - 1);
  launch_accum_fold(A.acc.as<float>(), A.pix.as<float>(), (size_t)A.w * A.h * A.channels, itm1, rnb, rit, ctx->sm_count,
                    ctx->stream);
  ctx->launches += 1;
  CK(cudaGetLastError());
  return GVPM_OK;
}

int gvpm_accum_read(gvpm_ctx *ctx, int normalized, float *acc, uint8_t *have_smoke, uint64_t *total_emitted) {
  if (!ctx) return GVPM_ERR_INVALID;
  int rc = accum_check(ctx, "gvpm_accum_read");
  if (rc) return rc;
  cudaSetDevice(ctx->device);
  const gvpm_ctx::Accum &A = ctx->accum;
  const size_t npix = (size_t)A.w * A.h, count = npix * A.channels;
  if (acc) CK(cudaMemcpyAsync(acc, A.acc.p, count * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  if (have_smoke) CK(cudaMemcpyAsync(have_smoke, A.smoke.p, npix, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (acc && normalized && !A.apa && A.total) {
    const float inv = 1.0f / (float)A.total;   // normalizedAccumulators(): a reciprocal multiply
    for (size_t i = 0; i < count; ++i) acc[i] *= inv;
  }
  if (total_emitted) *total_emitted = A.total;
  return GVPM_OK;
}

int gvpm_accum_device(gvpm_ctx *ctx, const float **acc, const uint8_t **have_smoke) {
  if (!ctx) return GVPM_ERR_INVALID;
  int rc = accum_check(ctx, "gvpm_accum_device");
  if (rc) return rc;
  if (acc) *acc = ctx->accum.acc.as<float>();
  if (have_smoke) *have_smoke = ctx->accum.smoke.as<uint8_t>();
  return GVPM_OK;
}

static int accum_image_check(gvpm_ctx *ctx, const char *what) {
  int rc = accum_check(ctx, what);
  if (rc) return rc;
  if (ctx->accum.channels != GVPM_OUT_FLOATS)
    return fail(ctx, GVPM_ERR_INVALID, std::string(what) + ": needs the 27-channel accumulators of gvpm");
  return GVPM_OK;
}

int gvpm_compute_gradient_accum(gvpm_ctx *ctx, int use_abs, int reuse_primal, float inv_emitted, float *throughput,
                                float *gx, float *gy) {
  if (!ctx) return GVPM_ERR_INVALID;
  int rc = accum_image_check(ctx, "gvpm_compute_gradient_accum");
  if (rc) return rc;
  if (reuse_primal && !(inv_emitted > 0.f)) return fail(ctx, GVPM_ERR_INVALID, "inv_emitted must be positive");
  const gvpm_ctx::Accum &A = ctx->accum;
  return compute_gradient_impl(ctx, A.acc.as<float>(), true, A.w, A.h, use_abs, reuse_primal ? 1 : 0,
                               reuse_primal ? inv_emitted : 1.f, throughput, gx, gy);
}

int gvpm_reconstruct_accum(gvpm_ctx *ctx, int use_abs, const float *direct, const gvpm_poisson_params *params,
                           float *throughput, float *gx, float *gy, float *reconstruction) {
  if (!ctx) return GVPM_ERR_INVALID;
  int rc = accum_image_check(ctx, "gvpm_reconstruct_accum");
  if (rc) return rc;
  const gvpm_ctx::Accum &A = ctx->accum;
  return reconstruct_impl(ctx, A.acc.as<float>(), true, A.w, A.h, use_abs, direct, params, throughput, gx, gy,
                          reconstruction);
}

}  // extern "C"
