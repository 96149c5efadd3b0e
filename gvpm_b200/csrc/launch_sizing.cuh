// launch_sizing.cuh — grid sizes of the gather kernels, from each kernel instantiation's own occupancy.
#pragma once

#include <cuda_runtime.h>

namespace gvpm {

// Resident CTAs per SM of kernel K at `threads` threads and `smem` bytes of dynamic shared memory, queried on the first
// call and cached per instantiation (at least 1).  A kernel with dynamic shared memory first gets the attribute that
// allows that much; if setting it fails, nothing is cached and 0 is returned (the error is left for cudaGetLastError).
template <auto K>
int resident_ctas(int threads, size_t smem) {
  static int ctas = 0;
  if (ctas == 0) {
    if (smem > 0 && cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, K, threads, smem);
    if (ctas < 1) ctas = 1;
  }
  return ctas;
}

// Persistent grid: every resident CTA slot of the device, but no more CTAs than work units (the CTAs pull work from a
// counter).
template <auto K>
unsigned persistent_grid(int sm_count, int threads, unsigned long long units, size_t smem = 0) {
  const unsigned long long grid = (unsigned long long)sm_count * resident_ctas<K>(threads, smem);
  return (unsigned)(grid < units ? grid : units);
}

// Grid-stride grid: 4 waves of resident CTAs, but no more CTAs than it takes to give every item a thread (at least 1).
template <auto K>
unsigned stride_grid(int sm_count, int threads, unsigned long long items) {
  unsigned long long need = (items + threads - 1) / threads;
  if (need == 0) need = 1;
  const unsigned long long grid = (unsigned long long)sm_count * resident_ctas<K>(threads, 0) * 4;
  return (unsigned)(grid < need ? grid : need);
}

}  // namespace gvpm
