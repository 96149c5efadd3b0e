// poisson.cu — screened-Poisson reconstruction of the gradient-domain image (SURVEY.md §8 row f-3), the step that
// follows computeGradient (gvpm/gvpm.cpp:554-702): x = argmin || W (b - P x) ||, b = [alpha * throughput; dx; dy],
// P = [alpha * I; Dx; Dy], solved by iteratively reweighted least squares around a conjugate-gradient solver on the
// normal equations A = P' W^2 P.  Restates, operation by operation, the reference solver
//   poisson::Solver::setupBackend / solveIndirect / exportImagesMTS      src/integrators/poisson_solver/Solver.cpp:255-578
//   poisson::Backend::calc_Px, calc_PTW2x, calc_Ax_xAx, calc_axpy, calc_xdoty, calc_r_rz, calc_x_p, calc_w2
//                                                                        src/integrators/poisson_solver/Backend.cpp:155-368
// (its CUDA backend, BackendCUDA.cu, targets sm_5x and uses the removed __shfl_xor).  Differences in design:
//   * b is never materialised: the residual kernel forms alpha * throughput, dx, dy on the fly;
//   * the element-wise passes are fused around the three reductions of a CG iteration (3 launches per iteration:
//     Ap + p'Ap | r, r'r | x, p), the scalars alpha = rz2 / pAp and beta = rz / rz2 stay on the device;
//   * every reduction is deterministic: per-CTA partials in a fixed grid, folded in index order by the last CTA to
//     finish (no second launch, no float atomics);
//   * per-element arithmetic uses the explicitly rounded intrinsics in the reference's operation order, so that only
//     the summation order of the reductions differs from the CPU result;
//   * all vectors of a 1080p image (25 MB each) stay resident in the 126 MB L2 across the CG iterations.
#include <cfloat>

#include "gvpm_device.cuh"
#include "warp_ops.cuh"

namespace gvpm {

namespace {

struct f3 { float x, y, z; };
__device__ __forceinline__ f3 ld3(const float *p, size_t i) { return {p[3 * i], p[3 * i + 1], p[3 * i + 2]}; }
__device__ __forceinline__ void st3(float *p, size_t i, f3 v) { p[3 * i] = v.x; p[3 * i + 1] = v.y; p[3 * i + 2] = v.z; }
__device__ __forceinline__ f3 add(f3 a, f3 b) { return {__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z)}; }
__device__ __forceinline__ f3 sub(f3 a, f3 b) { return {__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y), __fsub_rn(a.z, b.z)}; }
__device__ __forceinline__ f3 mul(f3 a, f3 b) { return {__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y), __fmul_rn(a.z, b.z)}; }
__device__ __forceinline__ f3 mul(f3 a, float s) { return {__fmul_rn(a.x, s), __fmul_rn(a.y, s), __fmul_rn(a.z, s)}; }
__device__ __forceinline__ f3 div(f3 a, f3 b) { return {__fdiv_rn(a.x, b.x), __fdiv_rn(a.y, b.y), __fdiv_rn(a.z, b.z)}; }
__device__ __forceinline__ f3 maxc(f3 a, float m) { return {a.x > m ? a.x : m, a.y > m ? a.y : m, a.z > m ? a.z : m}; }
__device__ __forceinline__ f3 zero3() { return {0.f, 0.f, 0.f}; }

constexpr int kThreads = 256;
constexpr int kMaxBlocks = 1024;

// CTA sum of three floats; the last CTA to arrive folds all partials in index order and hands the total to `fin`.
// partial: [gridDim.x * 3]; ticket: zero on entry, zero again on exit.
template <typename Fin>
__device__ __forceinline__ void reduce3_finish(f3 v, float *partial, unsigned *ticket, Fin fin) {
  __shared__ float sh[3][kThreads / 32];
  __shared__ bool last;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float c[3] = {v.x, v.y, v.z};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    c[a] = warp_sum(c[a]);
    if (lane == 0) sh[a][w] = c[a];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int a = 0; a < 3; ++a) {
      float s = 0.f;
      for (int k = 0; k < kThreads / 32; ++k) s += sh[a][k];
      partial[3 * blockIdx.x + a] = s;
    }
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  float t[3] = {0.f, 0.f, 0.f};
  for (unsigned b = threadIdx.x; b < gridDim.x; b += kThreads)
    for (int a = 0; a < 3; ++a) t[a] += ((volatile float *)partial)[3 * b + a];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    t[a] = warp_sum(t[a]);
    if (lane == 0) sh[a][w] = t[a];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    f3 tot = zero3();
    for (int k = 0; k < kThreads / 32; ++k) { tot.x += sh[0][k]; tot.y += sh[1][k]; tot.z += sh[2][k]; }
    fin(tot);
    *ticket = 0u;
  }
}

// x = throughput (or 0), Solver::setupBackend (:338-343)
__global__ void k_poisson_init(const float *__restrict__ tp, float *__restrict__ x, size_t n3) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += (size_t)gridDim.x * blockDim.x)
    x[i] = tp ? tp[i] : 0.f;
}

// e = b - P*x: calc_Px (:155-176) followed by calc_axpy(e, -1, e, b) (:243-259); b = [tp * alpha, dx, dy] (:327-335)
__global__ void k_poisson_residual(const float *__restrict__ tp, const float *__restrict__ dx, const float *__restrict__ dy,
                                   const float *__restrict__ x, int W, int H, float alpha, float *__restrict__ e) {
  const size_t n = (size_t)W * H;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int xx = (int)(i % W), yy = (int)(i / W);
    const f3 xi = ld3(x, i);
    const f3 b0 = tp ? mul(ld3(tp, i), alpha) : zero3();
    const f3 p0 = mul(xi, alpha);
    const f3 p1 = xx != W - 1 ? sub(ld3(x, i + 1), xi) : zero3();
    const f3 p2 = yy != H - 1 ? sub(ld3(x, i + W), xi) : zero3();
    st3(e, i, add(mul(p0, -1.0f), b0));
    st3(e, n + i, add(mul(p1, -1.0f), ld3(dx, i)));
    st3(e, 2 * n + i, add(mul(p2, -1.0f), ld3(dy, i)));
  }
}

__global__ void k_poisson_set(float *__restrict__ v, size_t m, float y) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (size_t)gridDim.x * blockDim.x) v[i] = y;
}

// calc_w2 (:348-368), first loop: w2 = 1 / (length(e) + reg) and its sum; scal[0] = coef = numElems / sum
__global__ void k_poisson_w2(const float *__restrict__ e, size_t m, float reg, float *__restrict__ w2,
                             float *__restrict__ partial, unsigned *__restrict__ ticket, float *__restrict__ coef) {
  float s = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (size_t)gridDim.x * blockDim.x) {
    const f3 ei = ld3(e, i);
    const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ei.x, ei.x), __fmul_rn(ei.y, ei.y)), __fmul_rn(ei.z, ei.z)));
    const float w = __fdiv_rn(1.0f, __fadd_rn(len, reg));
    w2[i] = w;
    s += w;
  }
  reduce3_finish({s, 0.f, 0.f}, partial, ticket, [=](f3 tot) { coef[0] = __fdiv_rn((float)m, tot.x); });
}
__global__ void k_poisson_w2_scale(float *__restrict__ w2, size_t m, const float *__restrict__ coef) {
  const float c = coef[0];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (size_t)gridDim.x * blockDim.x)
    w2[i] = __fmul_rn(w2[i], c);
}

// r = P' diag(w2) e (calc_PTW2x :180-205), rz = r'r (calc_xdoty :263-280), p = r (copy)
__global__ void k_poisson_ptw2x(const float *__restrict__ w2, const float *__restrict__ e, int W, int H, float alpha,
                                float *__restrict__ r, float *__restrict__ p, float *__restrict__ partial,
                                unsigned *__restrict__ ticket, float *__restrict__ rz) {
  const size_t n = (size_t)W * H;
  f3 acc = zero3();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int xx = (int)(i % W), yy = (int)(i / W);
    f3 v = mul(mul(ld3(e, i), w2[i]), alpha);
    if (xx != 0) v = add(v, mul(ld3(e, n + i - 1), w2[n + i - 1]));
    if (xx != W - 1) v = sub(v, mul(ld3(e, n + i), w2[n + i]));
    if (yy != 0) v = add(v, mul(ld3(e, 2 * n + i - W), w2[2 * n + i - W]));
    if (yy != H - 1) v = sub(v, mul(ld3(e, 2 * n + i), w2[2 * n + i]));
    st3(r, i, v);
    st3(p, i, v);
    acc = add(acc, mul(v, v));
  }
  reduce3_finish(acc, partial, ticket, [=](f3 tot) { rz[0] = tot.x; rz[1] = tot.y; rz[2] = tot.z; });
}

// Ap = A*p, pAp = p'*A*p (calc_Ax_xAx :209-239)
__global__ void k_poisson_ax(const float *__restrict__ w2, const float *__restrict__ x, int W, int H, float alpha,
                             float *__restrict__ Ax, float *__restrict__ partial, unsigned *__restrict__ ticket,
                             float *__restrict__ xAx) {
  const size_t n = (size_t)W * H;
  const float alphaSqr = __fmul_rn(alpha, alpha);
  f3 acc = zero3();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int xx = (int)(i % W), yy = (int)(i / W);
    const f3 xi = ld3(x, i);
    f3 a = mul(mul(xi, w2[i]), alphaSqr);
    if (xx != 0) a = add(a, mul(sub(xi, ld3(x, i - 1)), w2[n + i - 1]));
    if (xx != W - 1) a = add(a, mul(sub(xi, ld3(x, i + 1)), w2[n + i]));
    if (yy != 0) a = add(a, mul(sub(xi, ld3(x, i - W)), w2[2 * n + i - W]));
    if (yy != H - 1) a = add(a, mul(sub(xi, ld3(x, i + W)), w2[2 * n + i]));
    st3(Ax, i, a);
    acc = add(acc, mul(xi, a));
  }
  reduce3_finish(acc, partial, ticket, [=](f3 tot) { xAx[0] = tot.x; xAx[1] = tot.y; xAx[2] = tot.z; });
}

// r -= Ap * (rz2 / pAp), rz = r'r (calc_r_rz :284-313)
__global__ void k_poisson_r_rz(float *__restrict__ r, const float *__restrict__ Ap, size_t n, const float *__restrict__ rz2,
                               const float *__restrict__ pAp, float *__restrict__ partial, unsigned *__restrict__ ticket,
                               float *__restrict__ rz) {
  const f3 a = div({rz2[0], rz2[1], rz2[2]}, maxc({pAp[0], pAp[1], pAp[2]}, FLT_MIN));
  f3 acc = zero3();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const f3 ri = sub(ld3(r, i), mul(ld3(Ap, i), a));
    st3(r, i, ri);
    acc = add(acc, mul(ri, ri));
  }
  reduce3_finish(acc, partial, ticket, [=](f3 tot) { rz[0] = tot.x; rz[1] = tot.y; rz[2] = tot.z; });
}

// x += p * (rz2 / pAp), p = r + p * (rz / rz2) (calc_x_p :317-344)
__global__ void k_poisson_x_p(float *__restrict__ x, float *__restrict__ p, const float *__restrict__ r, size_t n,
                              const float *__restrict__ rz, const float *__restrict__ rz2, const float *__restrict__ pAp) {
  const f3 a = div({rz2[0], rz2[1], rz2[2]}, maxc({pAp[0], pAp[1], pAp[2]}, FLT_MIN));
  const f3 b = div({rz[0], rz[1], rz[2]}, maxc({rz2[0], rz2[1], rz2[2]}, FLT_MIN));
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const f3 pi = ld3(p, i);
    st3(x, i, add(ld3(x, i), mul(pi, a)));
    st3(p, i, add(ld3(r, i), mul(pi, b)));
  }
}

// exportImagesMTS "Final" (:559-578): rec = direct + x, or x
__global__ void k_poisson_final(const float *__restrict__ x, const float *__restrict__ direct, size_t n3,
                                float *__restrict__ rec) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += (size_t)gridDim.x * blockDim.x)
    rec[i] = direct ? __fadd_rn(__fmul_rn(1.0f, direct[i]), x[i]) : x[i];
}

inline int grid_for(size_t m) {
  size_t b = (m + kThreads - 1) / kThreads;
  return (int)(b < 1 ? 1 : (b > (size_t)kMaxBlocks ? kMaxBlocks : b));
}

}  // namespace

size_t poisson_workspace_floats(size_t n) {
  // e [9n] + w2 [3n] + x, r, p, Ap [3n each] + partials [3 * kMaxBlocks] + scalars (rz, rz2, pAp, coef: 16) + ticket
  return 9 * n + 3 * n + 4 * 3 * n + 3 * (size_t)kMaxBlocks + 32;
}

// Solver::solveIndirect (:376-504) without the preconditioned branch (no preset enables it).  tp / direct may be null.
// ws: poisson_workspace_floats(n) floats; host_rz: pinned 3 floats; returns the number of kernel launches, < 0 on error.
long long poisson_solve_device(const float *tp, const float *dx, const float *dy, const float *direct, int W, int H,
                               float alpha, int irlsIterMax, float irlsRegInit, float irlsRegIter, int cgIterMax,
                               int cgIterCheck, float cgTolerance, float *ws, float *host_rz, float *rec,
                               cudaStream_t st) {
  const size_t n = (size_t)W * H;
  float *e = ws, *w2 = e + 9 * n, *x = w2 + 3 * n, *r = x + 3 * n, *p = r + 3 * n, *Ap = p + 3 * n;
  float *partial = Ap + 3 * n, *scal = partial + 3 * kMaxBlocks;
  float *rz = scal, *rz2 = scal + 4, *pAp = scal + 8, *coef = scal + 12;
  unsigned *ticket = (unsigned *)(scal + 16);
  long long launches = 0;
  if (cudaMemsetAsync(scal, 0, 32 * sizeof(float), st) != cudaSuccess) return -1;
  const float a = tp ? alpha : 0.0f;   // m_P.alpha (:323)
  const int gn = grid_for(n), g3 = grid_for(3 * n);
  k_poisson_init<<<g3, kThreads, 0, st>>>(tp, x, 3 * n);
  ++launches;
  for (int irlsIter = 0; irlsIter < irlsIterMax; ++irlsIter) {
    k_poisson_residual<<<gn, kThreads, 0, st>>>(tp, dx, dy, x, W, H, a, e);
    if (irlsIter == 0) {
      k_poisson_set<<<g3, kThreads, 0, st>>>(w2, 3 * n, 1.0f);
      launches += 2;
    } else {
      const float reg = irlsRegInit * powf(irlsRegIter, (float)(irlsIter - 1));
      k_poisson_w2<<<g3, kThreads, 0, st>>>(e, 3 * n, reg, w2, partial, ticket, coef);
      k_poisson_w2_scale<<<g3, kThreads, 0, st>>>(w2, 3 * n, coef);
      launches += 3;
    }
    k_poisson_ptw2x<<<gn, kThreads, 0, st>>>(w2, e, W, H, a, r, p, partial, ticket, rz);
    ++launches;
    for (int cgIter = 0;; ++cgIter) {
      if (cgIter % cgIterCheck == 0 || cgIter == cgIterMax) {
        if (cudaMemcpyAsync(host_rz, rz, 3 * sizeof(float), cudaMemcpyDeviceToHost, st) != cudaSuccess) return -1;
        if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
        const float errL2W = host_rz[0] + host_rz[1] + host_rz[2];
        if (cgIter == cgIterMax || errL2W <= cgTolerance) break;
      }
      float *t = rz; rz = rz2; rz2 = t;   // swap(rz, rz2)
      k_poisson_ax<<<gn, kThreads, 0, st>>>(w2, p, W, H, a, Ap, partial, ticket, pAp);
      k_poisson_r_rz<<<gn, kThreads, 0, st>>>(r, Ap, n, rz2, pAp, partial, ticket, rz);
      k_poisson_x_p<<<gn, kThreads, 0, st>>>(x, p, r, n, rz, rz2, pAp);
      launches += 3;
    }
  }
  k_poisson_final<<<g3, kThreads, 0, st>>>(x, direct, 3 * n, rec);
  ++launches;
  return cudaGetLastError() == cudaSuccess ? launches : -1;
}

}  // namespace gvpm
