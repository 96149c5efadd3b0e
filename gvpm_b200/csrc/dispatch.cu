// dispatch.cu — photon dispatch between GPUs (SURVEY.md §8 row e): the sending half of the sharded G-BRE iteration.
//
// The image is sharded over the ranks (one process per GPU); every rank holds 1/N of the iteration's photons in its
// staging buffer (traced there, or uploaded over its own PCIe link).  A rank only ever needs the photons its own camera
// rays can reach - for a pinhole's primary rays 10-20 % of the set - so instead of all-gathering the whole set
// (N-1)/N * 102 B per photon in and out of every GPU) each rank CLASSIFIES its own photons against every receiver's
// frustum grid and ray-occupancy mask (frustum_key, the function the receiver's build evaluates) and writes the
// 128-byte gather records of the photons a receiver keeps straight into that receiver's inbox over NVLink
// (peer-mapped stores): packing and exchange are one kernel, a photon crosses the link once per rank that needs it
// (~1.1 times), and a receiver builds its grid over the records it was sent, nothing else.
//
//   k_dispatch_classify   thread per photon: one keep bit per receiver, per-CTA counts per receiver
//   k_scan_exclusive      one CTA per receiver: exclusive scan of the CTA counts (slot of a CTA's first record)
//   k_dispatch_emit       warp per 32 photons: records staged in shared memory (as k_pack_aos), then for every receiver
//                         the warp's kept records go out as ONE contiguous run of 16-byte stores (slots follow the photon
//                         order: deterministic, independent of scheduling)
//   k_dispatch_signal     counts, then a generation flag, written into every receiver's control block
//   k_flag_wait           the receiving side: spins (with a time-out) on its local flags until every sender has signalled
#include <cuda_runtime.h>

#include <cstdint>

#include "frustum_device.cuh"
#include "warp_ops.cuh"

namespace gvpm {

__global__ void __launch_bounds__(256) k_dispatch_classify(const __grid_constant__ DispatchParams P) {
  // a CTA takes chunks blk, blk + gridDim.x, ... of 256 photons: the launch may be a small persistent grid (a side
  // stream next to the gather kernels gets few CTA slots, and keeps them)
  for (uint32_t blk = blockIdx.x; blk < P.nb; blk += gridDim.x) {
  const uint32_t i = blk * blockDim.x + threadIdx.x;
  uint32_t bits = 0u;
  if (i < P.count) {
    const size_t g = (size_t)P.begin + i;
    const float px = __ldg(P.S.pos + 3 * g), py = __ldg(P.S.pos + 3 * g + 1), pz = __ldg(P.S.pos + 3 * g + 2);
    if (P.owner_map) {
      // every receiver projects on the plane of grids[0]: footprint once (frustum_key's arithmetic with the largest
      // pad), then the receivers under the footprint box from the owner map.  A superset of what each receiver's own
      // key keeps (the receiver drops the rest when it builds).
      const FrustumGrid &G = P.grids[0];
      const uint32_t all = (1u << P.n_dst) - 1u;
      const float qx = px - G.C[0], qy = py - G.C[1], qz = pz - G.C[2];
      const float rho = sqrtf(qx * qx + qy * qy + qz * qz);
      float x, y, z;
      frustum_project(G.m, G.u, G.v, qx, qy, qz, x, y, z);
      const float pr = P.pad_r_max * 1.001f + 1e-6f * rho;
      if (rho <= 2.f * pr) {
        bits = all;
      } else if (z < 0.1f * rho) {
        bits = rho <= 6.f * pr ? all : 0u;
      } else {
        const float tanT = sqrtf(x * x + y * y);
        const float sA = pr / rho;
        const float tanA = sA * rsqrtf(1.f - sA * sA) * 1.001f + 1e-6f;
        const float den = 1.f - tanT * tanA;
        const float tanS = den > 1e-3f ? (tanT + tanA) / den : 1e30f;
        if (tanS >= 8.24f) {
          bits = all;
        } else {
          const float wfoot = (tanS - tanT) * 1.01f + 1e-6f * (1.f + tanT) + 1e-5f * (1.f + tanT * tanT);
          // too wide for a receiver's coarsest class: its NEAR bucket, whatever its rays
          for (int d = 0; d < P.n_dst; ++d)
            if (wfoot > P.grids[d].csize[P.grids[d].classes - 1]) bits |= 1u << d;
          if (!(x + wfoot < P.ux0 || x - wfoot > P.ux1 || y + wfoot < P.uy0 || y - wfoot > P.uy1)) {
            const int i0 = occ_cell(x - wfoot, P.ux0, P.uix), i1 = occ_cell(x + wfoot, P.ux0, P.uix);
            const int j0 = occ_cell(y - wfoot, P.uy0, P.uiy), j1 = occ_cell(y + wfoot, P.uy0, P.uiy);
            for (int jj = j0; jj <= j1 && bits != all; ++jj)
              for (int ii = i0; ii <= i1; ++ii) bits |= __ldg(P.owner_map + jj * kOccRes + ii);
          }
        }
      }
    } else {
      for (int d = 0; d < P.n_dst; ++d) {
        const FrustumGrid &G = P.grids[d];
        const uint32_t DROP = (G.parity_split ? 2u : 1u) * G.n_cells + 1u;
        const uint32_t key = frustum_key(G, P.occ[d], px, py, pz, [&]() { return __ldg(P.S.path_id + g) & 1u; });
        if (key != DROP) bits |= 1u << d;
      }
    }
    P.keepbits[i] = (uint8_t)bits;
  }
  __shared__ BallotCounts<8, GVPM_MAX_PEERS> kept;
  for (int d = 0; d < P.n_dst; ++d) kept.put(__ballot_sync(0xffffffffu, (bits >> d) & 1u), d);
  __syncthreads();
  if (threadIdx.x < (unsigned)P.n_dst) P.block_cnt[(size_t)threadIdx.x * (P.nb + 1) + blk] = kept.total(threadIdx.x);
  __syncthreads();
  }
}

__global__ void __launch_bounds__(256) k_dispatch_emit(const __grid_constant__ DispatchParams P) {
  __shared__ float4 tile[8][32 * 9];   // per warp: 32 records x 8 float4, row stride 9 float4 (as k_pack_aos)
  __shared__ BallotCounts<8, GVPM_MAX_PEERS> kept;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (uint32_t blk = blockIdx.x; blk < P.nb; blk += gridDim.x) {
  const uint32_t i = blk * blockDim.x + threadIdx.x;
  const uint32_t bits = i < P.count ? P.keepbits[i] : 0u;
  for (int d = 0; d < P.n_dst; ++d) kept.put(__ballot_sync(0xffffffffu, (bits >> d) & 1u), d);
  float4 *t = tile[w];
  if (bits) {
    const size_t s = (size_t)P.begin + i;
    photon_record(t + lane * 9, P.S, s, (uint32_t)s);   // A7.x: the photon's index in the whole set (parity dumps)
  }
  __syncthreads();
  for (int d = 0; d < P.n_dst; ++d) {
    const uint32_t m = __ballot_sync(0xffffffffu, (bits >> d) & 1u);
    if (m == 0u) continue;
    const uint32_t slot = P.block_cnt[(size_t)d * (P.nb + 1) + blk] + kept.before(d);
    const uint32_t cnt = __popc(m);
    if (slot + cnt > P.region_cap) {
      if (lane == 0) atomicOr(P.overflow, 1u);
      continue;
    }
    float4 *dst = P.inbox[d] + (size_t)slot * 8;
    // the warp's kept records are consecutive slots: cnt * 8 float4, written 32 at a time
    for (uint32_t q = lane; q < cnt * 8u; q += 32u) {
      const int src = __fns(m, 0, (q >> 3) + 1);   // lane holding the (q >> 3)-th kept record
      dst[q] = t[src * 9 + (q & 7u)];
    }
  }
  __syncthreads();
  }
}

__global__ void k_dispatch_signal(const __grid_constant__ SignalParams P) {
  const int d = threadIdx.x;
  if (d >= P.n_dst) return;
  *(volatile uint32_t *)P.count_dst[d] = P.block_cnt[(size_t)d * (P.nb + 1) + P.nb];
  __threadfence_system();
  *(volatile uint32_t *)P.flag_dst[d] = P.gen;
}

// n flags (local memory, written by the peers) must all reach `target`.  One thread polls; gives up after ~4 s
// (a peer that died must not hang the GPU) and raises *timeout.
__global__ void k_flag_wait(const uint32_t *flags, int n, uint32_t target, unsigned *timeout) {
  const long long t0 = clock64();
  for (int i = 0; i < n; ++i) {
    while ((int)(*(volatile const uint32_t *)(flags + i) - target) < 0) {
      if (clock64() - t0 > 8000000000ll) { atomicOr(timeout, 1u); return; }
      __nanosleep(200);
    }
  }
  __threadfence_system();
}
// dst |= src: a protocol failure seen by k_flag_wait (a peer that never signalled) makes the grid built over that inbox
// "incomplete", which the gather reports instead of returning a partial result
__global__ void k_or_flag(uint32_t *dst, const uint32_t *src) {
  if (*src) *dst = 1u;
}
// the same value into one word of every peer (e.g. "my inbox b is free again")
__global__ void k_flag_set(const __grid_constant__ FlagSetParams P) {
  if ((int)threadIdx.x < P.n) {
    __threadfence_system();
    *(volatile uint32_t *)P.dst[threadIdx.x] = P.value;
  }
}

// neighbour dumps of a dispatched photon set: inbox index -> the photon's index in the whole set (word 28 of its record)
__global__ void k_translate_idx(uint32_t *__restrict__ idx, unsigned long long n, const float4 *__restrict__ aos) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = idx[i];
  idx[i] = __float_as_uint(__ldg(&aos[(size_t)(v & 0x7fffffffu) * 8 + 7].x)) | (v & 0x80000000u);
}

// ---- launchers ------------------------------------------------------------------------------------------------------
// ctas > 0: persistent grids of that many CTAs (a side stream: few slots, held to the end); 0: one CTA per chunk
void launch_dispatch(const DispatchParams &P, cudaStream_t st, int ctas) {
  if (P.count == 0) {
    cudaMemsetAsync(P.block_cnt, 0, (size_t)P.n_dst * (P.nb + 1) * 4, st);
    return;
  }
  const uint32_t grid = ctas > 0 ? (uint32_t)ctas < P.nb ? (uint32_t)ctas : P.nb : P.nb;
  k_dispatch_classify<<<grid, 256, 0, st>>>(P);
  k_scan_exclusive<uint32_t, 1><<<P.n_dst, 1024, 0, st>>>(P.block_cnt, P.nb, P.block_cnt + P.nb, P.nb + 1);
  k_dispatch_emit<<<grid, 256, 0, st>>>(P);
}
void launch_dispatch_signal(const SignalParams &P, cudaStream_t st) { k_dispatch_signal<<<1, 32, 0, st>>>(P); }
void launch_flag_wait(const uint32_t *flags, int n, uint32_t target, unsigned *timeout, cudaStream_t st) {
  k_flag_wait<<<1, 1, 0, st>>>(flags, n, target, timeout);
}
void launch_flag_set(const FlagSetParams &P, cudaStream_t st) { k_flag_set<<<1, 32, 0, st>>>(P); }
void launch_or_flag(uint32_t *dst, const uint32_t *src, cudaStream_t st) { k_or_flag<<<1, 1, 0, st>>>(dst, src); }
void launch_translate_idx(uint32_t *idx, unsigned long long n, const float4 *aos, cudaStream_t st) {
  if (n) k_translate_idx<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(idx, n, aos);
}

}  // namespace gvpm
