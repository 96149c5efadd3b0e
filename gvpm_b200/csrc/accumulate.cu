// accumulate.cu — the per-pixel accumulators of a progressive render (gvpm_accum_*, capi_accum.cu): the per-ray results
// of a gather summed per pixel, then the APA running mean of GPMIntegrator (gvpm.cpp:1054-1069) / SPPMIntegrator
// (sppm.cpp:866-871).  The reference is the host mirror's foldIteration (host/gvpm_host.hpp), built without FMA: every
// add and multiply here is an explicitly rounded intrinsic, so nvcc cannot contract them, and every pixel's rays are
// added in ray order.  Memory-bound streaming passes.
#include "gvpm_device.cuh"
#include "launch_sizing.cuh"

namespace gvpm {

// Rays that are one per pixel (gvpm_generate_rays): thread (r, j) adds channel j of ray r onto its pixel.  No two rays
// of one call share a pixel, so there is no race and the order per pixel is the call order.
__global__ void k_accum_scatter(const float *__restrict__ out, uint32_t stride, const int32_t *__restrict__ px,
                                const int32_t *__restrict__ py, uint32_t n, int w, int h, int C, float *__restrict__ dst,
                                uint8_t *__restrict__ smoke) {
  const size_t items = (size_t)n * C;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < items; t += (size_t)gridDim.x * blockDim.x) {
    const uint32_t r = (uint32_t)(t / C);
    const int j = (int)(t - (size_t)r * C);
    const int x = px[r], y = py[r];
    if (x < 0 || y < 0 || x >= w || y >= h) continue;
    const size_t p = (size_t)y * w + x;
    dst[p * C + j] = __fadd_rn(dst[p * C + j], out[(size_t)r * stride + j]);
    if (j == 0) smoke[p] = 1;
  }
}

// Sort keys of uploaded rays: the pixel index, or npix for a ray outside the film (sorted last, skipped).
__global__ void k_accum_keys(const int32_t *__restrict__ px, const int32_t *__restrict__ py, uint32_t n, int w, int h,
                             uint32_t *__restrict__ keys, uint32_t *__restrict__ vals) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int x = px[r], y = py[r];
  keys[r] = (x < 0 || y < 0 || x >= w || y >= h) ? (uint32_t)w * (uint32_t)h : (uint32_t)y * (uint32_t)w + (uint32_t)x;
  vals[r] = r;
}

// Rays sorted by pixel, stable in ray order: thread (i, j) at the head of a pixel's run adds channel j of the run's rays,
// one after the other, onto the pixel.
__global__ void k_accum_runs(const float *__restrict__ out, uint32_t stride, const uint32_t *__restrict__ skeys,
                             const uint32_t *__restrict__ svals, uint32_t n, uint32_t npix, int C, float *__restrict__ dst,
                             uint8_t *__restrict__ smoke) {
  const size_t items = (size_t)n * C;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < items; t += (size_t)gridDim.x * blockDim.x) {
    const uint32_t i = (uint32_t)(t / C);
    const int j = (int)(t - (size_t)i * C);
    const uint32_t k = skeys[i];
    if (k >= npix || (i > 0 && skeys[i - 1] == k)) continue;
    float s = dst[(size_t)k * C + j];
    for (uint32_t m = i; m < n && skeys[m] == k; ++m) s = __fadd_rn(s, out[(size_t)svals[m] * stride + j]);
    dst[(size_t)k * C + j] = s;
    if (j == 0) smoke[k] = 1;
  }
}

// acc = (acc * (it - 1) + pix * rnb) * rit, pix = 0, for every value (float4 body, scalar tail).
__device__ __forceinline__ float apa(float a, float x, float itm1, float rnb, float rit) {
  return __fmul_rn(__fadd_rn(__fmul_rn(a, itm1), __fmul_rn(x, rnb)), rit);
}
__global__ void k_accum_fold(float *__restrict__ acc, float *__restrict__ pix, size_t count, float itm1, float rnb,
                             float rit) {
  const size_t n4 = count / 4, step = (size_t)gridDim.x * blockDim.x;
  float4 *a4 = (float4 *)acc, *p4 = (float4 *)pix;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += step) {
    float4 a = a4[i];
    const float4 x = p4[i];
    a.x = apa(a.x, x.x, itm1, rnb, rit);
    a.y = apa(a.y, x.y, itm1, rnb, rit);
    a.z = apa(a.z, x.z, itm1, rnb, rit);
    a.w = apa(a.w, x.w, itm1, rnb, rit);
    a4[i] = a;
    p4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const size_t tail = 4 * n4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tail < count) {
    acc[tail] = apa(acc[tail], pix[tail], itm1, rnb, rit);
    pix[tail] = 0.f;
  }
}

constexpr int kAccumThreads = 256;

void launch_accum_scatter(const float *out, uint32_t stride, const int32_t *px, const int32_t *py, uint32_t n, int w,
                          int h, int C, float *dst, uint8_t *smoke, int sm_count, cudaStream_t st) {
  if (n == 0) return;
  const unsigned grid = stride_grid<k_accum_scatter>(sm_count, kAccumThreads, (unsigned long long)n * C);
  k_accum_scatter<<<grid, kAccumThreads, 0, st>>>(out, stride, px, py, n, w, h, C, dst, smoke);
}

void launch_accum_keys(const int32_t *px, const int32_t *py, uint32_t n, int w, int h, uint32_t *keys, uint32_t *vals,
                       cudaStream_t st) {
  if (n) k_accum_keys<<<(n + kAccumThreads - 1) / kAccumThreads, kAccumThreads, 0, st>>>(px, py, n, w, h, keys, vals);
}

void launch_accum_runs(const float *out, uint32_t stride, const uint32_t *skeys, const uint32_t *svals, uint32_t n,
                       uint32_t npix, int C, float *dst, uint8_t *smoke, int sm_count, cudaStream_t st) {
  if (n == 0) return;
  const unsigned grid = stride_grid<k_accum_runs>(sm_count, kAccumThreads, (unsigned long long)n * C);
  k_accum_runs<<<grid, kAccumThreads, 0, st>>>(out, stride, skeys, svals, n, npix, C, dst, smoke);
}

void launch_accum_fold(float *acc, float *pix, size_t count, float itm1, float rnb, float rit, int sm_count,
                       cudaStream_t st) {
  if (count == 0) return;
  const unsigned grid = stride_grid<k_accum_fold>(sm_count, kAccumThreads, count / 4 + 4);
  k_accum_fold<<<grid, kAccumThreads, 0, st>>>(acc, pix, count, itm1, rnb, rit);
}

}  // namespace gvpm
