// warp_ops.cuh — warp and CTA primitives shared by the kernel units: reductions, integer scans, the block total /
// in-block offset of the count -> scan -> emit passes, the segmented per-ray run sum of the shade kernels, and the
// single-CTA exclusive scan between a count pass and its emit pass.  Every helper is collective: all lanes of the warp
// (or all threads of the CTA) must call it, and the float helpers keep the summation order their comments state.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace gvpm {

// Sum over the full warp by the xor butterfly (offsets 16, 8, 4, 2, 1, in that order); every lane holds the result.
template <class T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// fmaxf / fminf over the full warp, same butterfly; every lane holds the result.
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Box of the warp: per axis, l = fminf and h = fmaxf over the full warp by the same butterfly; every lane holds it.
__device__ __forceinline__ void warp_box(float l[3], float h[3]) {
#pragma unroll
  for (int a = 0; a < 3; ++a)
    for (int o = 16; o > 0; o >>= 1) {
      l[a] = fminf(l[a], __shfl_xor_sync(0xffffffffu, l[a], o));
      h[a] = fmaxf(h[a], __shfl_xor_sync(0xffffffffu, h[a], o));
    }
}

// Integer inclusive scan over the full warp (shuffle-up, offsets 1 .. 16): lane i gets the sum of lanes 0 .. i.
template <class T>
__device__ __forceinline__ T warp_inclusive_scan(T v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

// ---- count form: integer values per thread, CTA of kWarps full warps (one __syncthreads each) ----
// The CTA's sum of v, valid in thread 0 only.
template <int kWarps, class T>
__device__ __forceinline__ T block_total(T v) {
  __shared__ T ws[kWarps];
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = v;
  __syncthreads();
  T t = 0;
  if (threadIdx.x == 0)
#pragma unroll
    for (int k = 0; k < kWarps; ++k) t += ws[k];
  return t;
}
// The sum of v over the threads in front of this one (thread order), in every thread.
template <int kWarps, class T>
__device__ __forceinline__ T block_exclusive(T v) {
  __shared__ T ws[kWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const T inc = warp_inclusive_scan(v, lane);
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  T off = inc - v;
#pragma unroll 1
  for (int k = 0; k < w; ++k) off += ws[k];
  return off;
}

// ---- predicate form: per-warp ballot counts of kCols predicates (one per receiver in the photon dispatch) ----
// put() from every warp (lane 0 stores), then the caller's __syncthreads, then total() / before() in any thread.
template <int kWarps, int kCols = 1>
struct BallotCounts {
  uint32_t n[kWarps][kCols];
  // m: the warp's ballot of predicate c
  __device__ __forceinline__ void put(uint32_t m, int c = 0) {
    if ((threadIdx.x & 31) == 0) n[threadIdx.x >> 5][c] = __popc(m);
  }
  // the CTA's count of predicate c
  __device__ __forceinline__ uint32_t total(int c = 0) const {
    uint32_t t = 0;
#pragma unroll
    for (int k = 0; k < kWarps; ++k) t += n[k][c];
    return t;
  }
  // the count of predicate c in the warps in front of this thread's warp
  __device__ __forceinline__ uint32_t before(int c = 0) const {
    uint32_t r = 0;
#pragma unroll 1   // rolled, like the loops it replaces: unrolled, it loads the counts 4-wide and costs registers
    for (int k = 0; k < (int)(threadIdx.x >> 5); ++k) r += n[k][c];
    return r;
  }
};

// Segmented sum over runs of equal `key` in lane order, then out[key * N + j] += the run's a[j] by float atomics from the
// last lane of the run (lanes with !valid take part in the scan but add nothing).  Inclusive shuffle-up scan, offsets
// 1 .. 16, each lane adding the value `off` lanes below while that lane is in its run.  SKIP_ZERO: a run sum that
// compares equal to 0 is not added (an atomic add of +0 would turn a -0 in `out` into +0).
// Offsets at or above the warp's longest run are skipped (warp-uniform): no lane is `off` lanes into its run there, so
// those levels add nothing and the sums are the same bits.  The caller must be converged in a way ptxas can see (a
// warp-uniform loop around the call), or it emits a second, WARPSYNC-wrapped copy of the N x 5 shuffles.
template <int N, bool SKIP_ZERO = false>
__device__ __forceinline__ void warp_run_sum(uint32_t key, float (&a)[N], bool valid, float *out, int lane) {
  const uint32_t kprev = __shfl_up_sync(0xffffffffu, key, 1);
  const uint32_t heads = __ballot_sync(0xffffffffu, lane == 0 || kprev != key);
  const int start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));  // first lane of my run
  const int runMax = (int)__reduce_max_sync(0xffffffffu, (uint32_t)(lane - start)) + 1;  // longest run, in lanes
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    if (off >= runMax) break;
    const bool same = lane - off >= start;
#pragma unroll
    for (int j = 0; j < N; ++j) {
      const float vu = __shfl_up_sync(0xffffffffu, a[j], off);
      if (same) a[j] += vu;
    }
  }
  if (valid && (lane == 31 || (heads >> (lane + 1) & 1u))) {
    float *o = out + (size_t)key * N;
#pragma unroll
    for (int j = 0; j < N; ++j)
      if (!SKIP_ZERO || a[j] != 0.f) atomicAdd(o + j, a[j]);
  }
}

// Exclusive scan in place of v[0 .. n) by one CTA of 1024 threads (kPer consecutive items per thread, 1024 * kPer per
// round); the sum of all n goes to *total.  CTA b works on v + b * stride and writes total + b * stride (one CTA per
// receiver in the photon dispatch, each with its own array).
template <class T, int kPer>
__global__ void __launch_bounds__(1024) k_scan_exclusive(T *v, uint32_t n, T *total, size_t stride) {
  __shared__ T ws[32];
  __shared__ T carry;
  v += blockIdx.x * stride;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (uint32_t base = 0; base < n; base += 1024 * kPer) {
    const uint32_t i0 = base + threadIdx.x * kPer;
    T x[kPer], sum = 0;
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      x[k] = i0 + k < n ? v[i0 + k] : T(0);
      sum += x[k];
    }
    const T inc = warp_inclusive_scan(sum, lane);
    if (lane == 31) ws[w] = inc;
    __syncthreads();
    if (w == 0) {
      const T t = ws[lane];
      ws[lane] = warp_inclusive_scan(t, lane) - t;   // exclusive prefix of the warp totals
    }
    __syncthreads();
    T excl = carry + ws[w] + (inc - sum);
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      if (i0 + k < n) v[i0 + k] = excl;
      excl += x[k];
    }
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl;
    __syncthreads();
  }
  if (threadIdx.x == 0) total[blockIdx.x * stride] = carry;
}

}  // namespace gvpm
