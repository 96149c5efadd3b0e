// capi_image.cu — image-space steps: gradients, screened-Poisson reconstruction, both in one call.  The accumulators
// come from the host (gvpm_compute_gradient, gvpm_reconstruct) or from the context's own device accumulators
// (gvpm_compute_gradient_accum, gvpm_reconstruct_accum in capi_accum.cu); the two share one body each.
#include "capi_internal.cuh"

int compute_gradient_impl(gvpm_ctx *ctx, const float *acc, bool acc_on_device, int w, int h, int use_abs, int reuse,
                          float inv_emitted, float *throughput, float *gx, float *gy) {
  if (!ctx || !acc || w <= 0 || h <= 0 || !throughput || !gx || !gy) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const size_t np = (size_t)w * h;
  CK(ctx->grad_out.reserve(np * 9 * 4));
  if (!acc_on_device) {
    CK(ctx->grad_in.reserve(np * GVPM_OUT_FLOATS * 4));
    CK(cudaMemcpyAsync(ctx->grad_in.p, acc, np * GVPM_OUT_FLOATS * 4, cudaMemcpyHostToDevice, ctx->stream));
    acc = ctx->grad_in.as<float>();
  }
  float *o = ctx->grad_out.as<float>();
  launch_gradient(acc, w, h, use_abs, o, o + 3 * np, o + 6 * np, ctx->stream, reuse, inv_emitted);
  ctx->launches += 1;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(throughput, o, np * 12, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(gx, o + 3 * np, np * 12, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(gy, o + 6 * np, np * 12, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GVPM_OK;
}

// computeGradient + reconstruction in one call: the three planes never leave the device (gvpm.cpp:554-690)
int reconstruct_impl(gvpm_ctx *ctx, const float *acc, bool acc_on_device, int w, int h, int use_abs, const float *direct,
                     const gvpm_poisson_params *params, float *throughput, float *gx, float *gy, float *reconstruction) {
  if (!ctx || !acc || w <= 0 || h <= 0 || !params || !reconstruction) return GVPM_ERR_INVALID;
  if (params->cg_precond)
    return fail(ctx, GVPM_ERR_UNSUPPORTED, "the preconditioned CG branch (cgPrecond, enabled by no preset) is not built");
  cudaSetDevice(ctx->device);
  const size_t n = (size_t)w * h, plane = 3 * n * sizeof(float);
  CK(ctx->grad_out.reserve(n * 9 * 4));
  CK(ctx->poisson_io.reserve(5 * plane));
  CK(ctx->poisson_ws.reserve(poisson_workspace_floats(n) * sizeof(float)));
  if (!acc_on_device) CK(ctx->grad_in.reserve(n * GVPM_OUT_FLOATS * 4));
  cudaStream_t st = ctx->stream;
  CK(cudaEventRecord(ctx->ev[2], st));
  if (!acc_on_device) {
    CK(cudaMemcpyAsync(ctx->grad_in.p, acc, n * GVPM_OUT_FLOATS * 4, cudaMemcpyHostToDevice, st));
    acc = ctx->grad_in.as<float>();
  }
  float *o = ctx->grad_out.as<float>(), *io = ctx->poisson_io.as<float>();
  float *d_direct = io + 9 * n, *d_rec = io + 12 * n;
  if (direct) CK(cudaMemcpyAsync(d_direct, direct, plane, cudaMemcpyHostToDevice, st));
  launch_gradient(acc, w, h, use_abs, o, o + 3 * n, o + 6 * n, st);
  ctx->launches += 1;
  const long long launched = poisson_solve_device(
      o, o + 3 * n, o + 6 * n, direct ? d_direct : nullptr, w, h, std::max(params->alpha, 0.0f),
      std::max(params->irls_iter_max, 1), std::max(params->irls_reg_init, 0.0f), std::max(params->irls_reg_iter, 0.0f),
      std::max(params->cg_iter_max, 1), std::max(params->cg_iter_check, 1), std::max(params->cg_tolerance, 0.0f),
      ctx->poisson_ws.as<float>(), (float *)ctx->pair_count_host, d_rec, st);
  if (launched < 0) return fail(ctx, GVPM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
  ctx->launches += (uint64_t)launched;
  if (throughput) CK(cudaMemcpyAsync(throughput, o, plane, cudaMemcpyDeviceToHost, st));
  if (gx) CK(cudaMemcpyAsync(gx, o + 3 * n, plane, cudaMemcpyDeviceToHost, st));
  if (gy) CK(cudaMemcpyAsync(gy, o + 6 * n, plane, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(reconstruction, d_rec, plane, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(ctx->ev[3], st));
  CK(cudaStreamSynchronize(st));
  CK(cudaEventElapsedTime(&ctx->poisson_ms, ctx->ev[2], ctx->ev[3]));
  ctx->timed_gather = false;
  return GVPM_OK;
}

extern "C" {

int gvpm_compute_gradient(gvpm_ctx *ctx, const float *acc, int w, int h, int use_abs, float *throughput,
                          float *gx, float *gy) {
  return compute_gradient_impl(ctx, acc, false, w, h, use_abs, 0, 1.f, throughput, gx, gy);
}
int gvpm_compute_gradient_reuse_primal(gvpm_ctx *ctx, const float *acc, int w, int h, int use_abs, float inv_emitted,
                                       float *throughput, float *gx, float *gy) {
  if (!(inv_emitted > 0.f)) return GVPM_ERR_INVALID;
  return compute_gradient_impl(ctx, acc, false, w, h, use_abs, 1, inv_emitted, throughput, gx, gy);
}

// ---- screened-Poisson reconstruction (row f-3): poisson::Solver of the reference, gvpm.cpp:610-690 -------------------
int gvpm_poisson_preset(const char *preset, gvpm_poisson_params *p) {
  if (!preset || !p) return GVPM_ERR_INVALID;
  // Solver::Params::Params + setConfigPreset, Solver.cpp:59-158
  p->alpha = 0.2f;
  p->irls_iter_max = 1; p->irls_reg_init = 0.f; p->irls_reg_iter = 0.f;
  p->cg_iter_max = 1; p->cg_iter_check = 100; p->cg_precond = 0; p->cg_tolerance = 0.f;
  if (!strcmp(preset, "L1D")) { p->irls_iter_max = 20; p->irls_reg_init = 0.05f; p->irls_reg_iter = 0.5f; p->cg_iter_max = 50; }
  else if (!strcmp(preset, "L1Q")) { p->irls_iter_max = 64; p->irls_reg_init = 1.0f; p->irls_reg_iter = 0.7f; p->cg_iter_max = 1000; }
  else if (!strcmp(preset, "L1L")) { p->irls_iter_max = 7; p->irls_reg_init = 1.0e-4f; p->irls_reg_iter = 1.0e-1f; p->cg_iter_max = 20000; p->cg_tolerance = 1.0e-20f; }
  else if (!strcmp(preset, "L2D")) { p->cg_iter_max = 50; }
  else if (!strcmp(preset, "L2Q")) { p->cg_iter_max = 500; }
  else return GVPM_ERR_INVALID;
  return GVPM_OK;
}

int gvpm_poisson_solve(gvpm_ctx *ctx, int w, int h, const float *throughput, const float *dx, const float *dy,
                       const float *direct, const gvpm_poisson_params *params, float *reconstruction) {
  if (!ctx || w <= 0 || h <= 0 || !dx || !dy || !params || !reconstruction) return GVPM_ERR_INVALID;
  if (params->cg_precond)
    return fail(ctx, GVPM_ERR_UNSUPPORTED, "the preconditioned CG branch (cgPrecond, enabled by no preset) is not built");
  cudaSetDevice(ctx->device);
  // Solver::Params::sanitize, Solver.cpp:162-172
  const float alpha = std::max(params->alpha, 0.0f);
  const int irlsIterMax = std::max(params->irls_iter_max, 1), cgIterMax = std::max(params->cg_iter_max, 1),
            cgIterCheck = std::max(params->cg_iter_check, 1);
  const float irlsRegInit = std::max(params->irls_reg_init, 0.0f), irlsRegIter = std::max(params->irls_reg_iter, 0.0f),
              cgTolerance = std::max(params->cg_tolerance, 0.0f);
  const size_t n = (size_t)w * h, plane = 3 * n * sizeof(float);
  CK(ctx->poisson_io.reserve(5 * plane));
  CK(ctx->poisson_ws.reserve(poisson_workspace_floats(n) * sizeof(float)));
  float *io = ctx->poisson_io.as<float>();
  float *d_tp = io, *d_dx = io + 3 * n, *d_dy = io + 6 * n, *d_direct = io + 9 * n, *d_rec = io + 12 * n;
  cudaStream_t st = ctx->stream;
  CK(cudaEventRecord(ctx->ev[2], st));
  if (throughput) CK(cudaMemcpyAsync(d_tp, throughput, plane, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_dx, dx, plane, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_dy, dy, plane, cudaMemcpyHostToDevice, st));
  if (direct) CK(cudaMemcpyAsync(d_direct, direct, plane, cudaMemcpyHostToDevice, st));
  const long long launched = poisson_solve_device(throughput ? d_tp : nullptr, d_dx, d_dy, direct ? d_direct : nullptr, w, h,
                                                  alpha, irlsIterMax, irlsRegInit, irlsRegIter, cgIterMax, cgIterCheck,
                                                  cgTolerance, ctx->poisson_ws.as<float>(), (float *)ctx->pair_count_host,
                                                  d_rec, st);
  if (launched < 0) return fail(ctx, GVPM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
  ctx->launches += (uint64_t)launched;
  CK(cudaMemcpyAsync(reconstruction, d_rec, plane, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(ctx->ev[3], st));
  CK(cudaStreamSynchronize(st));
  CK(cudaEventElapsedTime(&ctx->poisson_ms, ctx->ev[2], ctx->ev[3]));
  ctx->timed_gather = false;
  return GVPM_OK;
}

int gvpm_reconstruct(gvpm_ctx *ctx, const float *acc, int w, int h, int use_abs, const float *direct,
                     const gvpm_poisson_params *params, float *throughput, float *gx, float *gy, float *reconstruction) {
  return reconstruct_impl(ctx, acc, false, w, h, use_abs, direct, params, throughput, gx, gy, reconstruction);
}

}  // extern "C"
