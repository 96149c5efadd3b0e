// tree_build.cu — GPU build of the photon-point hierarchy.  Replaces PointKDTree::build
// (include/mitsuba/core/kdtree.h:326-378,921-1037; single-threaded sliding-midpoint recursion) and
// GradientBeamRadianceEstimator's constructor + buildHierarchy (gvpm/gvpm_accel.cpp:10-55;
// single-threaded bottom-up AABB recursion) with: bounds reduction -> 30-bit Morton keys (1024^3 cells:
// far finer than a leaf of 32 photons, and half the radix passes of a 63-bit key) -> radix sort -> raw SoA
// packed into 128-byte records (streaming) -> records gathered into Morton-ordered 128-bit planes (every
// random read is one aligned 128-byte record) -> bottom-up 32-ary box levels (one warp per node, shuffle
// reductions).
#include <algorithm>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "gvpm_device.cuh"
#include "frustum_device.cuh"
#include "warp_ops.cuh"

namespace gvpm {

// ---- bounds: per-block partial min/max of n points, then one block folds the partials -----
__global__ void k_bounds_partial(const float *__restrict__ pos, uint32_t stride, uint32_t n, float *__restrict__ partial) {
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      float v = pos[(size_t)stride * i + a];
      lo[a] = fminf(lo[a], v);
      hi[a] = fmaxf(hi[a], v);
    }
  }
  __shared__ float s[6][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  warp_box(lo, hi);
  if (lane == 0)
#pragma unroll
    for (int a = 0; a < 3; ++a) { s[a][w] = lo[a]; s[3 + a][w] = hi[a]; }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = lane < nw ? s[a][lane] : INFINITY;
      hi[a] = lane < nw ? s[3 + a][lane] : -INFINITY;
    }
    warp_box(lo, hi);
    if (lane == 0)
#pragma unroll
      for (int a = 0; a < 3; ++a) { partial[6 * blockIdx.x + a] = lo[a]; partial[6 * blockIdx.x + 3 + a] = hi[a]; }
  }
}
// bounds[0..2] = min, [3..5] = max, [6] = max |coordinate|
__global__ void k_bounds_final(const float *__restrict__ partial, int nblocks, float *__restrict__ bounds) {
  const int lane = threadIdx.x;
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int b = lane; b < nblocks; b += 32)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = fminf(lo[a], partial[6 * b + a]);
      hi[a] = fmaxf(hi[a], partial[6 * b + 3 + a]);
    }
  warp_box(lo, hi);
  float mag = 0.f;
#pragma unroll
  for (int a = 0; a < 3; ++a) mag = fmaxf(mag, fmaxf(fabsf(lo[a]), fabsf(hi[a])));
  if (lane == 0) {
    for (int a = 0; a < 3; ++a) { bounds[a] = lo[a]; bounds[3 + a] = hi[a]; }
    bounds[6] = mag;
  }
}

__device__ __forceinline__ uint32_t spread10(uint32_t v) {  // 10 bits -> every third bit
  uint32_t x = v & 0x3ffu;
  x = (x | x << 16) & 0x030000ffu;
  x = (x | x << 8) & 0x0300f00fu;
  x = (x | x << 4) & 0x030c30c3u;
  x = (x | x << 2) & 0x09249249u;
  return x;
}

// 30-bit 3-D Hilbert index of a 1024^3 cell (Skilling, "Programming the Hilbert curve", 2004: axes -> transpose, then
// the bits are interleaved).  Unlike the Z-order curve the Hilbert curve never jumps: ANY run of consecutive keys is a
// connected blob, so the boxes of 32 consecutive photons (and of 32 consecutive boxes, ...) have no outliers that
// straddle a Z-curve discontinuity, and fewer of them are hit per ray.
__device__ __forceinline__ uint32_t hilbert30(uint32_t x0, uint32_t x1, uint32_t x2) {
  uint32_t X[3] = {x0, x1, x2};
  const uint32_t M = 1u << 9;
#pragma unroll
  for (uint32_t Q = M; Q > 1u; Q >>= 1) {   // inverse undo
    const uint32_t Pm = Q - 1u;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (X[i] & Q) {
        X[0] ^= Pm;
      } else {
        const uint32_t t = (X[0] ^ X[i]) & Pm;
        X[0] ^= t;
        X[i] ^= t;
      }
    }
  }
  X[1] ^= X[0];                              // Gray encode
  X[2] ^= X[1];
  uint32_t t = 0u;
#pragma unroll
  for (uint32_t Q = M; Q > 1u; Q >>= 1)
    if (X[2] & Q) t ^= Q - 1u;
  X[0] ^= t; X[1] ^= t; X[2] ^= t;
  // transpose -> index: bit b of X[0] is the most significant of the triple
  return (spread10(X[0]) << 2) | (spread10(X[1]) << 1) | spread10(X[2]);
}

__global__ void k_morton(const float *__restrict__ pos, uint32_t stride, uint32_t n, const float *__restrict__ bounds,
                         uint32_t *__restrict__ keys, uint32_t *__restrict__ vals) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t q[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float lo = bounds[a], ext = bounds[3 + a] - lo;
    float u = ext > 0.f ? (pos[(size_t)stride * i + a] - lo) / ext : 0.f;
    u = fminf(fmaxf(u, 0.f), 1.f);
    q[a] = min((uint32_t)(u * 1024.f), 1023u);
  }
  keys[i] = hilbert30(q[0], q[1], q[2]);
  vals[i] = i;
}

// raw SoA -> 128-byte records in the caller's order (streaming reads, each thread writes its own record; layout and
// derived terms: gvpm_device.cuh photon_record)
#define GVPM_AOS_FLOAT4 8
// Each thread assembles its photon's record in registers; the warp then transposes through a padded shared tile so
// that every store instruction writes 512 contiguous bytes (4 whole records) instead of 32 scattered 16-byte pieces.
__global__ void __launch_bounds__(256) k_pack_aos(const PhotonStaging S, uint32_t n, float4 *__restrict__ aos) {
  __shared__ float4 tile[8][32 * 9];   // per warp: 32 records x 8 float4, row stride 9 float4 (conflict-free both ways)
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const uint32_t warpBase = blockIdx.x * blockDim.x + (w << 5);
  const uint32_t s = warpBase + lane;
  float4 *t = tile[w];
  if (s < n) photon_record(t + lane * 9, S, s, 0u);
  __syncwarp();
  if (warpBase >= n) return;
  const uint32_t nRec = min(32u, n - warpBase);
  float4 *dst = aos + (size_t)warpBase * GVPM_AOS_FLOAT4;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t q = 32u * j + lane;          // float4 index inside the warp's 4 KB of records
    if ((q >> 3) < nRec) dst[q] = t[(q >> 3) * 9 + (q & 7u)];
  }
}
// sorted position plane P0 (pos.xyz, meta) + original index: the only sorted copies the gather needs
__global__ void k_gather_sorted(const float4 *__restrict__ aos, const uint32_t *__restrict__ sorted, uint32_t n,
                                float4 *__restrict__ planes, uint32_t *__restrict__ orig) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = sorted[i];
  planes[i] = __ldg(aos + (size_t)s * GVPM_AOS_FLOAT4);
  orig[i] = s;
}

// level 0: one warp per leaf of 32 photons; box = AABB(centres) inflated by the radius.
// (the reference's per-photon cube [p-r, p+r], gvpm_accel.cpp:38-42, unioned over the leaf)
__global__ void k_leaf_boxes(const float4 *__restrict__ p0, uint32_t n, uint32_t nLeaves, float radius,
                             float4 *__restrict__ lo, float4 *__restrict__ hi) {
  const uint32_t leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (leaf >= nLeaves) return;
  const uint32_t i = leaf * 32 + lane;
  float l[3] = {INFINITY, INFINITY, INFINITY}, h[3] = {-INFINITY, -INFINITY, -INFINITY};
  if (i < n) {
    const float4 p = p0[i];
    l[0] = h[0] = p.x; l[1] = h[1] = p.y; l[2] = h[2] = p.z;
  }
  warp_box(l, h);
  if (lane == 0) {
    lo[leaf] = make_float4(l[0] - radius, l[1] - radius, l[2] - radius, 0.f);
    hi[leaf] = make_float4(h[0] + radius, h[1] + radius, h[2] + radius, 0.f);
  }
}

// level l+1 from level l: one warp per parent node
__global__ void k_level_boxes(const float4 *__restrict__ clo, const float4 *__restrict__ chi, uint32_t nChild,
                              uint32_t nParent, float4 *__restrict__ plo, float4 *__restrict__ phi) {
  const uint32_t node = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (node >= nParent) return;
  const uint32_t i = node * 32 + lane;
  float l[3] = {INFINITY, INFINITY, INFINITY}, h[3] = {-INFINITY, -INFINITY, -INFINITY};
  if (i < nChild) {
    const float4 a = clo[i], b = chi[i];
    l[0] = a.x; l[1] = a.y; l[2] = a.z; h[0] = b.x; h[1] = b.y; h[2] = b.z;
  }
  warp_box(l, h);
  if (lane == 0) {
    plo[node] = make_float4(l[0], l[1], l[2], 0.f);
    phi[node] = make_float4(h[0], h[1], h[2], 0.f);
  }
}

// ---- ray-region pruning (gvpm_build_points_for_rays) ---------------------------------------------------------------
// When the image is sharded over GPUs a rank gathers only its own camera rays, which cross only a part of the
// scene; photons that no uploaded ray can reach need neither be sorted nor boxed.  The ray segments, dilated by the
// search radius, mark the cells of a 64^3 occupancy grid over their own bounding box; the key pass drops every photon
// whose cell is unmarked.  Conservative by construction (see k_ray_mask), so the gather is unchanged: a dropped
// photon fails the neighbour predicate (gvpm_accel.h:297-301) for every uploaded ray.
constexpr int kGridRes = 64;                                  // cells per axis
constexpr int kGridWords = kGridRes * kGridRes * kGridRes / 32;  // 8192 words = 32 KB: fits a CTA's shared memory
struct RayGrid {       // device-resident, written by k_ray_box_final
  float lo[3], hi[3];  // grid box = AABB of the dilated ray segments
  float inv[3];        // cells per unit length
  float cmin, cmax;    // smallest / largest cell edge
  float mag;           // largest |coordinate| of the box (rounding slack)
  int valid;           // 0: no ray
};

__device__ __forceinline__ void atomic_min_float(float *a, float v) {
  if (v >= 0.f) atomicMin((int *)a, __float_as_int(v)); else atomicMax((unsigned *)a, __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_float(float *a, float v) {
  if (v >= 0.f) atomicMax((int *)a, __float_as_int(v)); else atomicMin((unsigned *)a, __float_as_uint(v));
}
// the part of ray i's supporting line that can hold the projection of a neighbour: t in [-r, edge_len + r]
// (the 3-D kernel samples t' in [disk - r, disk + r] and needs mint <= t' <= edge_len, shift_volume_photon.cpp:707-721)
__device__ __forceinline__ bool ray_segment(const float4 *__restrict__ rays, uint32_t i, float r, float p0[3], float p1[3]) {
  const float4 q0 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4), q1 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4 + 1),
               q2 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4 + 2);
  // sppm's primal query is bounded by maxt (q1.w), gvpm's by edge_len >= maxt: the larger of the two covers both
  const float tEnd = fmaxf(q2.w, q1.w);
  const float t0 = -r, t1 = tEnd + r;
  p0[0] = q0.x + q1.x * t0; p0[1] = q0.y + q1.y * t0; p0[2] = q0.z + q1.z * t0;
  p1[0] = q0.x + q1.x * t1; p1[1] = q0.y + q1.y * t1; p1[2] = q0.z + q1.z * t1;
  return tEnd >= q0.w;   // edge_len >= mint: the gather skips the others
}
__global__ void k_ray_box(const float4 *__restrict__ rays, uint32_t n, float r, float *__restrict__ box) {
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float p0[3], p1[3];
    if (!ray_segment(rays, i, r, p0, p1)) continue;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = fminf(lo[a], fminf(p0[a], p1[a]));
      hi[a] = fmaxf(hi[a], fmaxf(p0[a], p1[a]));
    }
  }
  warp_box(lo, hi);
  if ((threadIdx.x & 31) == 0)
#pragma unroll
    for (int a = 0; a < 3; ++a)
      if (lo[a] <= hi[a]) { atomic_min_float(box + a, lo[a]); atomic_max_float(box + 3 + a, hi[a]); }
}
// box[0..5] -> grid parameters + the 7-float bounds block the traversal reads (min, max, max |coordinate|)
__global__ void k_ray_box_final(const float *__restrict__ box, float r, RayGrid *__restrict__ g, float *__restrict__ bounds) {
  RayGrid G;
  G.valid = box[0] <= box[3] && box[1] <= box[4] && box[2] <= box[5];
  float mag = 0.f, cmin = INFINITY, cmax = 0.f;
  for (int a = 0; a < 3; ++a) {
    float lo = G.valid ? box[a] : 0.f, hi = G.valid ? box[3 + a] : 0.f;
    const float pad = 1.01f * r + 1e-5f * (fabsf(lo) + fabsf(hi) + (hi - lo)) + 1e-30f;
    lo -= pad; hi += pad;
    G.lo[a] = lo; G.hi[a] = hi;
    const float c = (hi - lo) / kGridRes;
    G.inv[a] = 1.f / c;
    cmin = fminf(cmin, c);
    cmax = fmaxf(cmax, c);
    mag = fmaxf(mag, fmaxf(fabsf(lo), fabsf(hi)));
  }
  G.cmin = cmin; G.cmax = cmax; G.mag = mag;
  *g = G;
  for (int a = 0; a < 3; ++a) { bounds[a] = G.lo[a]; bounds[3 + a] = G.hi[a]; }
  bounds[6] = mag;
}
__device__ __forceinline__ int grid_cell(const RayGrid &G, int a, float x) {
  const int c = (int)floorf((x - G.lo[a]) * G.inv[a]);
  return min(max(c, 0), kGridRes - 1);
}
// mark every cell that meets the cube [p - h, p + h] in the CTA's shared mask
__device__ __forceinline__ void mark_cube(uint32_t *mask, const RayGrid &G, const float p[3], float h) {
  const int x0 = grid_cell(G, 0, p[0] - h), x1 = grid_cell(G, 0, p[0] + h);
  const int y0 = grid_cell(G, 1, p[1] - h), y1 = grid_cell(G, 1, p[1] + h);
  const int z0 = grid_cell(G, 2, p[2] - h), z1 = grid_cell(G, 2, p[2] + h);
  for (int z = z0; z <= z1; ++z)
    for (int y = y0; y <= y1; ++y) {
      const int row = (z * kGridRes + y) * (kGridRes / 32);
      for (int w = x0 >> 5; w <= (x1 >> 5); ++w) {
        const int b0 = max(x0 - 32 * w, 0), b1 = min(x1 - 32 * w, 31);
        const uint32_t bits = (0xffffffffu >> (31 - b1)) & (0xffffffffu << b0);
        if ((mask[row + w] & bits) != bits) atomicOr(mask + row + w, bits);
      }
    }
}
// One warp per 32 consecutive rays (neighbouring pixels: gvpm_upload_rays keeps the caller's block order).  Any point
// within r of a segment lies within r + s/2 of one of its samples spaced s apart, hence inside the sample's cube of
// half-width h >= r + s/2; cell indices are monotone in the coordinate, so a photon inside the cube falls in a marked
// cell.  Coherent warps mark only the first ray's segment, dilated by the largest end-point distance to the other
// segments (points at equal fractions of two segments are never farther apart than the farther pair of end points).
__global__ void __launch_bounds__(256) k_ray_mask(const float4 *__restrict__ rays, uint32_t n, float r,
                                                   const RayGrid *__restrict__ gp, uint32_t *__restrict__ gmask) {
  __shared__ uint32_t mask[kGridWords];
  for (int w = threadIdx.x; w < kGridWords; w += blockDim.x) mask[w] = 0u;
  __syncthreads();
  const RayGrid G = *gp;
  const int lane = threadIdx.x & 31;
  const uint32_t nWarpJobs = (n + 31) / 32, warpsPerGrid = gridDim.x * (blockDim.x >> 5);
  for (uint32_t job = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); G.valid && job < nWarpJobs; job += warpsPerGrid) {
    const uint32_t i = job * 32 + lane;
    float p0[3] = {0.f, 0.f, 0.f}, p1[3] = {0.f, 0.f, 0.f};
    const bool act = i < n && ray_segment(rays, i, r, p0, p1);
    const uint32_t am = __ballot_sync(0xffffffffu, act);
    if (am == 0u) continue;
    const int c = __ffs(am) - 1;
    float c0[3], c1[3], spread = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) { c0[a] = __shfl_sync(0xffffffffu, p0[a], c); c1[a] = __shfl_sync(0xffffffffu, p1[a], c); }
    if (act) {
      const float ax = p0[0] - c0[0], ay = p0[1] - c0[1], az = p0[2] - c0[2];
      const float bx = p1[0] - c1[0], by = p1[1] - c1[1], bz = p1[2] - c1[2];
      spread = fmaxf(sqrtf(ax * ax + ay * ay + az * az), sqrtf(bx * bx + by * by + bz * bz));
    }
    spread = warp_max(spread);
    // (a bundle a few cells wide: the rays of a pixel patch fill the dilated region anyway, so nothing is over-marked)
    const bool coherent = spread <= 4.f * G.cmax;
    if (coherent) {  // all lanes work on the first segment
#pragma unroll
      for (int a = 0; a < 3; ++a) { p0[a] = c0[a]; p1[a] = c1[a]; }
    }
    if (!coherent && !act) continue;
    const float dx = p1[0] - p0[0], dy = p1[1] - p0[1], dz = p1[2] - p0[2];
    const float len = sqrtf(dx * dx + dy * dy + dz * dz);
    const int nS = min(128, (int)ceilf(len / G.cmin) + 2);
    const float s = len / (float)(nS - 1);
    const float h = (r + (coherent ? spread * 1.001f : 0.f) + 0.5f * s) * 1.002f + 4e-6f * (G.mag + len);
    for (int k = coherent ? lane : 0; k < nS; k += coherent ? 32 : 1) {
      const float u = (float)k / (float)(nS - 1);
      const float p[3] = {p0[0] + dx * u, p0[1] + dy * u, p0[2] + dz * u};
      mark_cube(mask, G, p, h);
    }
  }
  __syncthreads();
  for (int w = threadIdx.x; w < kGridWords; w += blockDim.x)
    if (mask[w]) atomicOr(gmask + w, mask[w]);
}
// Pass 1 over all photons: keep test (cell of the photon marked?); keepmask gets one bit per photon (word = 32 consecutive
// photons) and block_kept the CTA's number of kept photons.  The kept indices are then compacted in photon order
// (exclusive scan of block_kept + k_compact_kept): the order of the sorted set - hence the pair order and every float
// accumulation order of the gather - does not depend on how the CTAs were scheduled.  Memory-bound: the Hilbert keys are
// computed afterwards, for the kept photons only (k_keys_kept).
__global__ void __launch_bounds__(256) k_keep_pruned(const float *__restrict__ pos, uint32_t n, const RayGrid *__restrict__ gp,
                              const uint32_t *__restrict__ gmask, uint32_t *__restrict__ keepmask,
                              uint32_t *__restrict__ block_kept) {
  __shared__ BallotCounts<8> kept;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  bool keep = false;
  if (i < n) {
    const RayGrid &G = *gp;
    const float x = pos[3 * (size_t)i], y = pos[3 * (size_t)i + 1], z = pos[3 * (size_t)i + 2];
    if (G.valid && x >= G.lo[0] && x <= G.hi[0] && y >= G.lo[1] && y <= G.hi[1] && z >= G.lo[2] && z <= G.hi[2]) {
      const int cx = grid_cell(G, 0, x), cy = grid_cell(G, 1, y), cz = grid_cell(G, 2, z);
      const uint32_t bit = (uint32_t)((cz * kGridRes + cy) * kGridRes + cx);
      keep = (__ldg(gmask + (bit >> 5)) >> (bit & 31u)) & 1u;
    }
  }
  const uint32_t km = __ballot_sync(0xffffffffu, keep);
  if ((threadIdx.x & 31) == 0 && i < n) keepmask[i >> 5] = km;
  kept.put(km);
  __syncthreads();
  if (threadIdx.x == 0) block_kept[blockIdx.x] = kept.total();
}
// Pass 2 over the m kept photons: 30-bit Hilbert key, quantised in the grid box
__global__ void k_keys_kept(const float *__restrict__ pos, const uint32_t *__restrict__ vals, uint32_t m,
                            const RayGrid *__restrict__ gp, uint32_t *__restrict__ keys) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= m) return;
  const RayGrid &G = *gp;
  const size_t i3 = 3 * (size_t)vals[slot];
  uint32_t q[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float u = (__ldg(pos + i3 + a) - G.lo[a]) / (G.hi[a] - G.lo[a]);
    u = fminf(fmaxf(u, 0.f), 1.f);
    q[a] = min((uint32_t)(u * 1024.f), 1023u);
  }
  keys[slot] = hilbert30(q[0], q[1], q[2]);
}
// k_pack_aos for the kept photons only: same streaming layout (the photon set arrives in the caller's order, so the kept
// ones are scattered evenly), loads and the transposed stores predicated by the keep bits
__global__ void __launch_bounds__(256) k_pack_aos_kept(const PhotonStaging S, uint32_t n, const uint32_t *__restrict__ keepmask,
                                                        float4 *__restrict__ aos) {
  __shared__ float4 tile[8][32 * 9];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const uint32_t warpBase = blockIdx.x * blockDim.x + (w << 5);
  if (warpBase >= n) return;
  const uint32_t km = __ldg(keepmask + (warpBase >> 5));
  if (km == 0u) return;
  const uint32_t s = warpBase + lane;
  float4 *t = tile[w];
  if (km >> lane & 1u) photon_record(t + lane * 9, S, s, 0u);
  __syncwarp();
  float4 *dst = aos + (size_t)warpBase * GVPM_AOS_FLOAT4;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t q = 32u * j + lane;          // float4 index inside the warp's 4 KB of records
    if (km >> (q >> 3) & 1u) dst[q] = t[(q >> 3) * 9 + (q & 7u)];
  }
}


// ---- perspective (frustum) grid: build side (gvpm_device.cuh FrustumGrid) ---------------------------------------------
// Pass 1 over the active rays: normal equations of "the point closest to all lines" (A = sum(I - d d^T),
// b = sum((I - d d^T) o)) and the direction sum, in double, one partial per block, folded in block order by
// k_pinhole_solve (deterministic).  partial: [nb][16] doubles = A(6: xx xy xz yy yz zz), b(3), dsum(3), count.
__device__ __forceinline__ bool ray_active(const float4 q0, const float4 q1, const float4 q2) {
  return fmaxf(q2.w, q1.w) >= q0.w;
}
__global__ void __launch_bounds__(256) k_pinhole_accum(const float4 *__restrict__ rays, uint32_t n, double *__restrict__ partial) {
  double acc[13];
#pragma unroll
  for (int k = 0; k < 13; ++k) acc[k] = 0.0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 q0 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4), q1 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4 + 1),
                 q2 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4 + 2);
    if (!ray_active(q0, q1, q2)) continue;
    const double dx = q1.x, dy = q1.y, dz = q1.z, ox = q0.x, oy = q0.y, oz = q0.z;
    const double od = ox * dx + oy * dy + oz * dz;
    acc[0] += 1.0 - dx * dx; acc[1] += -dx * dy; acc[2] += -dx * dz;
    acc[3] += 1.0 - dy * dy; acc[4] += -dy * dz; acc[5] += 1.0 - dz * dz;
    acc[6] += ox - od * dx; acc[7] += oy - od * dy; acc[8] += oz - od * dz;
    acc[9] += dx; acc[10] += dy; acc[11] += dz;
    acc[12] += 1.0;
  }
  __shared__ double sh[8][13];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 13; ++k) {
    const double v = warp_sum(acc[k]);
    if (lane == 0) sh[w][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 13) {
    double v = 0.0;
    for (int k = 0; k < 8; ++k) v += sh[k][threadIdx.x];
    partial[(size_t)blockIdx.x * 16 + threadIdx.x] = v;
  }
}
// fit[0..2] = C, [3..5] = m, [6..8] = u, [9..11] = v, [12] = count, [13] = conditioning (det / trace^3; 0 = no point)
__global__ void k_pinhole_solve(const double *__restrict__ partial, int nb, float *__restrict__ fit, int use_dir, float dir_x,
                                float dir_y, float dir_z) {
  double a[13];
  for (int k = 0; k < 13; ++k) {
    double v = 0.0;
    for (int b = 0; b < nb; ++b) v += partial[(size_t)b * 16 + k];
    a[k] = v;
  }
  const double xx = a[0], xy = a[1], xz = a[2], yy = a[3], yz = a[4], zz = a[5];
  const double det = xx * (yy * zz - yz * yz) - xy * (xy * zz - yz * xz) + xz * (xy * yz - yy * xz);
  const double tr = xx + yy + zz;
  double cond = tr > 0.0 ? det / (tr * tr * tr) : 0.0;
  double C[3] = {0, 0, 0};
  if (cond > 1e-12) {
    const double bx = a[6], by = a[7], bz = a[8];
    C[0] = (bx * (yy * zz - yz * yz) - xy * (by * zz - yz * bz) + xz * (by * yz - yy * bz)) / det;
    C[1] = (xx * (by * zz - yz * bz) - bx * (xy * zz - yz * xz) + xz * (xy * bz - by * xz)) / det;
    C[2] = (xx * (yy * bz - by * yz) - xy * (xy * bz - by * xz) + bx * (xy * yz - yy * xz)) / det;
  } else {
    cond = 0.0;
  }
  double ml = sqrt(a[9] * a[9] + a[10] * a[10] + a[11] * a[11]);
  double m[3] = {0, 0, 1};
  if (ml > 0.0) { m[0] = a[9] / ml; m[1] = a[10] / ml; m[2] = a[11] / ml; } else cond = 0.0;
  if (use_dir) {   // the caller's view direction (gvpm_set_view_direction): every rank of a sharded image then projects
                   // on the same plane, whatever part of the image its own rays cover
    const double dl = sqrt((double)dir_x * dir_x + (double)dir_y * dir_y + (double)dir_z * dir_z);
    m[0] = dir_x / dl; m[1] = dir_y / dl; m[2] = dir_z / dl;
  }
  // any orthonormal basis of the plane orthogonal to m
  double t[3] = {0, 0, 0};
  if (fabs(m[0]) <= fabs(m[1]) && fabs(m[0]) <= fabs(m[2])) t[0] = 1; else if (fabs(m[1]) <= fabs(m[2])) t[1] = 1; else t[2] = 1;
  double u[3] = {t[1] * m[2] - t[2] * m[1], t[2] * m[0] - t[0] * m[2], t[0] * m[1] - t[1] * m[0]};
  const double ul = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
  for (int k = 0; k < 3; ++k) u[k] /= ul;
  const double v[3] = {m[1] * u[2] - m[2] * u[1], m[2] * u[0] - m[0] * u[2], m[0] * u[1] - m[1] * u[0]};
  for (int k = 0; k < 3; ++k) { fit[k] = (float)C[k]; fit[3 + k] = (float)m[k]; fit[6 + k] = (float)u[k]; fit[9 + k] = (float)v[k]; }
  fit[12] = (float)a[12];
  fit[13] = (float)cond;
}
// Pass 2 over the active rays: largest distance of C to a ray's line, smallest cos(d, m), bounds of the projected
// directions.  stats: [0] delta max, [1] -cos min (as max), [2] -xmin, [3] xmax, [4] -ymin, [5] ymax  (all folded with
// atomicMax on non-negative-biased float bits: values are stored + 4 to keep them positive)
__global__ void __launch_bounds__(256) k_pinhole_check(const float4 *__restrict__ rays, uint32_t n, const float *__restrict__ fit,
                                                        unsigned *__restrict__ stats) {
  float mx[6] = {0.f, -2.f, -1e30f, -1e30f, -1e30f, -1e30f};
  const float C[3] = {fit[0], fit[1], fit[2]}, m[3] = {fit[3], fit[4], fit[5]}, u[3] = {fit[6], fit[7], fit[8]}, v[3] = {fit[9], fit[10], fit[11]};
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 q0 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4), q1 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4 + 1),
                 q2 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4 + 2);
    if (!ray_active(q0, q1, q2)) continue;
    const float cx = C[0] - q0.x, cy = C[1] - q0.y, cz = C[2] - q0.z;
    const float t = cx * q1.x + cy * q1.y + cz * q1.z;
    const float ex = cx - t * q1.x, ey = cy - t * q1.y, ez = cz - t * q1.z;
    mx[0] = fmaxf(mx[0], sqrtf(ex * ex + ey * ey + ez * ez));
    float x, y, z;
    frustum_project(m, u, v, q1.x, q1.y, q1.z, x, y, z);
    mx[1] = fmaxf(mx[1], -z);
    if (z > 0.f) { mx[2] = fmaxf(mx[2], -x); mx[3] = fmaxf(mx[3], x); mx[4] = fmaxf(mx[4], -y); mx[5] = fmaxf(mx[5], y); }
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const float vv = warp_max(mx[k]);
    // monotone map float -> unsigned (handles negatives)
    const unsigned b = __float_as_uint(vv);
    const unsigned key = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
    if ((threadIdx.x & 31) == 0) atomicMax(stats + k, key);
  }
}

// Coarse occupancy of the rays' projected directions: kOccRes x kOccRes bits over [xmin, xmax] x [ymin, ymax], built in
// shared memory per CTA and OR-ed into global memory.  k_frustum_keys drops a photon when no bit under its footprint
// box is set (no ray can reach it): this is what leaves most of the photon set out of a rank's sort when the image is
// sharded over GPUs.
__global__ void __launch_bounds__(256) k_frustum_mark(const float4 *__restrict__ rays, uint32_t n, const FrustumGrid G,
                                                       uint32_t *__restrict__ occ) {
  __shared__ uint32_t mask[kOccWords];
  for (int w = threadIdx.x; w < kOccWords; w += blockDim.x) mask[w] = 0u;
  __syncthreads();
  const float ix = kOccRes / fmaxf(G.xmax - G.xmin, 1e-20f), iy = kOccRes / fmaxf(G.ymax - G.ymin, 1e-20f);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 q0 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4), q1 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4 + 1),
                 q2 = __ldg(rays + (size_t)i * GVPM_RAY_FLOAT4 + 2);
    if (!ray_active(q0, q1, q2)) continue;
    float x, y, z;
    frustum_project(G.m, G.u, G.v, q1.x, q1.y, q1.z, x, y, z);
    const int bit = occ_cell(y, G.ymin, iy) * kOccRes + occ_cell(x, G.xmin, ix);
    const uint32_t b = 1u << (bit & 31);
    if (!(mask[bit >> 5] & b)) atomicOr(&mask[bit >> 5], b);
  }
  __syncthreads();
  for (int w = threadIdx.x; w < kOccWords; w += blockDim.x)
    if (mask[w]) atomicOr(occ + w, mask[w]);
}
// per photon: footprint class, cell, key (see FrustumGrid).  vals = the photon's rank inside its cell (one atomic on the
// cell's counter): cell_start is the exclusive scan of the counters, and k_scatter_index puts the photon's index at
// cell_start[key] + rank.  coord_mag: atomicMax of the largest |coordinate| (float bits; the traversal's rounding pad).
__global__ void __launch_bounds__(256) k_frustum_keys(const float *__restrict__ pos, uint32_t stride,
                                                       const uint32_t *__restrict__ par_src, uint32_t par_stride, uint32_t par_shift,
                                                       uint32_t n, const FrustumGrid G, const uint32_t *__restrict__ occ,
                                                       uint32_t *__restrict__ keys, uint32_t *__restrict__ vals,
                                                       unsigned *__restrict__ coord_mag, uint32_t *__restrict__ keepmask,
                                                       uint32_t *__restrict__ cell_count, uint32_t region_cap,
                                                       const uint32_t *__restrict__ region_count) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  float mag = 0.f;
  bool keep = false;
  // dispatched photon sets (dispatch.cu): the index space is one region of region_cap records per sending rank, of which
  // the first region_count[sender] are filled
  const bool filled = i < n && (region_cap == 0u || (i % region_cap) < __ldg(region_count + i / region_cap));
  if (i < n && !filled) keys[i] = (G.parity_split ? 2u : 1u) * G.n_cells + 1u;
  if (filled) {
    const float px = pos[(size_t)stride * i], py = pos[(size_t)stride * i + 1], pz = pos[(size_t)stride * i + 2];
    mag = fmaxf(fmaxf(fabsf(px), fabsf(py)), fabsf(pz));
    const uint32_t key = frustum_key(G, occ, px, py, pz, [&]() { return (__ldg(par_src + (size_t)par_stride * i) >> par_shift) & 1u; });
    const uint32_t DROP = (G.parity_split ? 2u : 1u) * G.n_cells + 1u;
    keys[i] = key;
    keep = key != DROP;
    if (keep) vals[i] = atomicAdd(cell_count + key, 1u);
  }
  // one keep bit per photon (word = 32 consecutive photons): the record packing and the index scatter read them
  const uint32_t km = __ballot_sync(0xffffffffu, keep);
  if ((threadIdx.x & 31) == 0 && i < n) keepmask[i >> 5] = km;
  // one atomic per CTA, and only while the CTA's maximum beats what is already there (a single hot address otherwise
  // serialises hundreds of thousands of atomics)
  __shared__ float wmag[8];
  mag = warp_max(mag);
  if ((threadIdx.x & 31) == 0) wmag[threadIdx.x >> 5] = mag;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = 0.f;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) m = fmaxf(m, wmag[k]);
    if (m > __uint_as_float(*(volatile unsigned *)coord_mag)) atomicMax(coord_mag, __float_as_uint(m));
  }
}
// counting sort: the index map alone (orig[cell_start[key] + rank] = photon).  4-byte random writes into an array that
// stays in L2 (40 MB for 10 M photons); the position plane is then gathered with coalesced writes (k_gather_sorted).
// Scattering the 16-byte plane entries directly costs more than both passes together: random partial-sector writes into
// 160 MB are read-modify-write cycles in DRAM (measured: 0.40 ms against 0.06 + 0.24 ms).
__global__ void __launch_bounds__(256) k_scatter_index(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ rank,
                                                        const uint32_t *__restrict__ keepmask, const uint32_t *__restrict__ cell_start,
                                                        uint32_t n, uint32_t *__restrict__ orig) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !(__ldg(keepmask + (i >> 5)) >> (i & 31u) & 1u)) return;
  orig[__ldg(cell_start + keys[i]) + rank[i]] = i;
}
// position plane from the index map; m = number of sorted slots, read from the device (cell_start[n_keys - 1] = kept photons)
__global__ void k_gather_by_index(const float4 *__restrict__ aos, const uint32_t *__restrict__ orig, const uint32_t *__restrict__ m_dev,
                                  float4 *__restrict__ planes) {
  const uint32_t m = __ldg(m_dev);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x)
    planes[i] = __ldg(aos + (size_t)__ldg(orig + i) * GVPM_AOS_FLOAT4);
}
// indices of the kept photons, in index order, packed to the front: block_off = exclusive scan of block_kept
__global__ void __launch_bounds__(256) k_compact_kept(const uint32_t *__restrict__ keepmask, const uint32_t *__restrict__ block_off,
                                                       uint32_t n, uint32_t *__restrict__ vals_c) {
  __shared__ BallotCounts<8> kept;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t km = i < n ? __ldg(keepmask + (i >> 5)) : 0u;   // i and its warp share the word (blockDim = 256, aligned)
  kept.put(km);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  if (!(km >> lane & 1u)) return;
  vals_c[block_off[blockIdx.x] + kept.before() + __popc(km & ((1u << lane) - 1u))] = i;
}

// raw ray SoA -> 5 x 64 B records per ray
__global__ void k_pack_rays(const RayStaging S, uint32_t r0, uint32_t n, float4 *__restrict__ rays) {
  const uint32_t i = r0 + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 *r = rays + (size_t)i * GVPM_RAY_FLOAT4;
  const size_t i3 = 3 * (size_t)i;
  r[0] = make_float4(S.o[i3], S.o[i3 + 1], S.o[i3 + 2], S.mint[i]);
  r[1] = make_float4(S.d[i3], S.d[i3 + 1], S.d[i3 + 2], S.maxt[i]);
  r[2] = make_float4(S.eye_contrib[i3], S.eye_contrib[i3 + 1], S.eye_contrib[i3 + 2], S.edge_len[i]);
  r[3] = make_float4(S.xi[i], __uint_as_float((uint32_t)S.px[i]), __uint_as_float((uint32_t)S.py[i]),
                     __uint_as_float((uint32_t)S.edge_id[i]));
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const size_t j = 4 * (size_t)i + k, j3 = 3 * j;
    r[4 * (k + 1)] = make_float4(S.off_o[j3], S.off_o[j3 + 1], S.off_o[j3 + 2], S.off_len[j]);
    r[4 * (k + 1) + 1] = make_float4(S.off_d[j3], S.off_d[j3 + 1], S.off_d[j3 + 2], S.off_sensor[j]);
    r[4 * (k + 1) + 2] = make_float4(S.off_eye[j3], S.off_eye[j3 + 1], S.off_eye[j3 + 2],
                                     __uint_as_float(S.off_valid[j] ? 1u : 0u));
    r[4 * (k + 1) + 3] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// ---- host-side drivers ---------------------------------------------------------------------
size_t sort_temp_bytes(uint32_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint32_t *)nullptr, (uint32_t *)nullptr,
                                  (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)n, 0, 30);
  return bytes;
}

cudaError_t run_sort_bits(void *temp, size_t temp_bytes, const uint32_t *kin, uint32_t *kout, const uint32_t *vin,
                          uint32_t *vout, uint32_t n, int bits, cudaStream_t st) {
  return cub::DeviceRadixSort::SortPairs(temp, temp_bytes, kin, kout, vin, vout, (int)n, 0, bits, st);
}

int bounds_blocks(uint32_t n) {
  int b = (int)((n + 255) / 256);
  return b < 1 ? 1 : (b > 1024 ? 1024 : b);
}

void launch_bounds(const float *pos, uint32_t n, float *partial, float *bounds, cudaStream_t st, uint32_t stride) {
  const int nb = bounds_blocks(n);
  k_bounds_partial<<<nb, 256, 0, st>>>(pos, stride, n, partial);
  k_bounds_final<<<1, 32, 0, st>>>(partial, nb, bounds);
}
void launch_morton(const float *pos, uint32_t n, const float *bounds, uint32_t *keys, uint32_t *vals,
                   cudaStream_t st, uint32_t stride) {
  k_morton<<<(n + 255) / 256, 256, 0, st>>>(pos, stride, n, bounds, keys, vals);
}
void launch_pack_sorted(const PhotonStaging &S, float4 *aos, const uint32_t *sorted, uint32_t n, float4 *planes,
                        uint32_t *orig, cudaStream_t st, bool records_ready) {
  if (!records_ready) k_pack_aos<<<(n + 255) / 256, 256, 0, st>>>(S, n, aos);
  k_gather_sorted<<<(n + 255) / 256, 256, 0, st>>>(aos, sorted, n, planes, orig);
}
size_t ray_grid_bytes() { return sizeof(RayGrid); }
size_t ray_mask_bytes() { return (size_t)kGridWords * 4; }
// box: 6 floats (+inf x3, -inf x3 on entry); grid: RayGrid; mask: zeroed kGridWords words
void launch_ray_region(const float4 *rays, uint32_t nRays, float radius, float *box, void *grid, uint32_t *mask,
                       float *bounds, int sm_count, cudaStream_t st) {
  if (nRays) k_ray_box<<<std::min<uint32_t>((nRays + 255) / 256, 1024u), 256, 0, st>>>(rays, nRays, radius, box);
  k_ray_box_final<<<1, 1, 0, st>>>(box, radius, (RayGrid *)grid, bounds);
  if (nRays) {
    const uint32_t need = (nRays + 255) / 256;
    k_ray_mask<<<std::min<uint32_t>(need, 2u * (uint32_t)sm_count), 256, 0, st>>>(rays, nRays, radius, (const RayGrid *)grid, mask);
  }
}
void launch_keep_pruned(const float *pos, uint32_t n, const void *grid, const uint32_t *mask, uint32_t *keepmask,
                        uint32_t *block_kept, cudaStream_t st) {
  if (n) k_keep_pruned<<<(n + 255) / 256, 256, 0, st>>>(pos, n, (const RayGrid *)grid, mask, keepmask, block_kept);
}
void launch_keys_kept(const float *pos, const uint32_t *vals, uint32_t m, const void *grid, uint32_t *keys, cudaStream_t st) {
  if (m) k_keys_kept<<<(m + 255) / 256, 256, 0, st>>>(pos, vals, m, (const RayGrid *)grid, keys);
}
// records of the kept photons only (keepmask), then the sorted position plane / index map of the first m sorted slots
void launch_pack_sorted_kept(const PhotonStaging &S, uint32_t n, const uint32_t *keepmask, const uint32_t *sorted, uint32_t m,
                             float4 *aos, float4 *planes, uint32_t *orig, cudaStream_t st) {
  if (n) k_pack_aos_kept<<<(n + 255) / 256, 256, 0, st>>>(S, n, keepmask, aos);
  if (m) k_gather_sorted<<<(m + 255) / 256, 256, 0, st>>>(aos, sorted, m, planes, orig);
}
// in-place exclusive scan of nb words by one CTA (a few thousand entries, 8 per thread); total -> total[0]
void launch_scan_u32(uint32_t *vals, uint32_t nb, uint32_t *total, cudaStream_t st) {
  k_scan_exclusive<uint32_t, 8><<<1, 1024, 0, st>>>(vals, nb, total, 0);
}

// ---- frustum grid launchers ----
int pinhole_blocks(uint32_t n) { int b = (int)((n + 255) / 256); return b < 1 ? 1 : (b > 512 ? 512 : b); }
// partial: [pinhole_blocks * 16] doubles; fit: 16 floats; stats: 8 words (zeroed here)
void launch_pinhole_fit(const float4 *rays, uint32_t n, double *partial, float *fit, unsigned *stats, cudaStream_t st,
                        const float *view_dir) {
  const int nb = pinhole_blocks(n);
  k_pinhole_accum<<<nb, 256, 0, st>>>(rays, n, partial);
  k_pinhole_solve<<<1, 1, 0, st>>>(partial, nb, fit, view_dir ? 1 : 0, view_dir ? view_dir[0] : 0.f, view_dir ? view_dir[1] : 0.f,
                                  view_dir ? view_dir[2] : 1.f);
  cudaMemsetAsync(stats, 0, 32, st);
  k_pinhole_check<<<nb, 256, 0, st>>>(rays, n, fit, stats);
}
size_t frustum_occ_bytes() { return (size_t)kOccWords * 4; }
void launch_compact_kept(const uint32_t *keepmask, const uint32_t *block_off, uint32_t n, uint32_t *vals_c, cudaStream_t st) {
  if (n) k_compact_kept<<<(n + 255) / 256, 256, 0, st>>>(keepmask, block_off, n, vals_c);
}
// occ: frustum_occ_bytes() (zeroed here); coord_mag: one word (zeroed here); cell_count: n_keys + 1 words, zeroed
// pos / stride: photon positions (stride in floats: 3 for the staged SoA plane, 32 for 128-byte records); parity of the
// photon's path id = (par_src[par_stride * i] >> par_shift) & 1
// region_cap / region_count: dispatched photon sets (0 / nullptr: every index up to n holds a photon)
void launch_frustum_keys(const float4 *rays, uint32_t n_rays, const float *pos, uint32_t stride, const uint32_t *par_src,
                         uint32_t par_stride, uint32_t par_shift, uint32_t n,
                         const FrustumGrid &G, uint32_t *occ, uint32_t *keys, uint32_t *vals, unsigned *coord_mag,
                         uint32_t *keepmask, uint32_t *cell_count, uint32_t region_cap, const uint32_t *region_count,
                         int sm_count, cudaStream_t st) {
  cudaMemsetAsync(occ, 0, frustum_occ_bytes(), st);
  cudaMemsetAsync(coord_mag, 0, 4, st);
  if (n_rays) k_frustum_mark<<<std::min<uint32_t>((n_rays + 255) / 256, 2u * (uint32_t)sm_count), 256, 0, st>>>(rays, n_rays, G, occ);
  if (n) k_frustum_keys<<<(n + 255) / 256, 256, 0, st>>>(pos, stride, par_src, par_stride, par_shift, n, G, occ, keys, vals, coord_mag, keepmask, cell_count, region_cap, region_count);
}
// counting sort: cell_start[0 .. n_keys] = exclusive scan of the per-cell counts (cell_count[n_keys] must be 0)
size_t cell_scan_temp_bytes(uint32_t n_keys) {
  size_t bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)n_keys + 1);
  return bytes;
}
cudaError_t launch_cell_scan(void *temp, size_t temp_bytes, const uint32_t *cell_count, uint32_t *cell_start, uint32_t n_keys,
                             cudaStream_t st) {
  return cub::DeviceScan::ExclusiveSum(temp, temp_bytes, cell_count, cell_start, (int)n_keys + 1, st);
}
// records of the kept photons, index map at cell_start[key] + rank, position plane gathered from it (kept_dev: slots in use)
void launch_pack_scatter(const PhotonStaging &S, uint32_t n, const uint32_t *keepmask, const uint32_t *keys, const uint32_t *rank,
                         const uint32_t *cell_start, float4 *aos, float4 *planes, uint32_t *orig, cudaStream_t st,
                         bool records_ready, const uint32_t *kept_dev, int sm_count) {
  if (!n) return;
  if (!records_ready) k_pack_aos_kept<<<(n + 255) / 256, 256, 0, st>>>(S, n, keepmask, aos);
  k_scatter_index<<<(n + 255) / 256, 256, 0, st>>>(keys, rank, keepmask, cell_start, n, orig);
  k_gather_by_index<<<std::min<uint32_t>((n + 255) / 256, 16u * (uint32_t)sm_count), 256, 0, st>>>(aos, orig, kept_dev, planes);
}
// the occupancy mask alone (what a rank publishes to the ranks that send it photons)
void launch_frustum_mark(const float4 *rays, uint32_t n_rays, const FrustumGrid &G, uint32_t *occ, int sm_count, cudaStream_t st) {
  cudaMemsetAsync(occ, 0, frustum_occ_bytes(), st);
  if (n_rays) k_frustum_mark<<<std::min<uint32_t>((n_rays + 255) / 256, 2u * (uint32_t)sm_count), 256, 0, st>>>(rays, n_rays, G, occ);
}
void launch_leaf_boxes(const float4 *p0, uint32_t n, uint32_t nLeaves, float radius, float4 *lo, float4 *hi,
                       cudaStream_t st) {
  k_leaf_boxes<<<(nLeaves + 7) / 8, 256, 0, st>>>(p0, n, nLeaves, radius, lo, hi);
}
void launch_level_boxes(const float4 *clo, const float4 *chi, uint32_t nChild, uint32_t nParent, float4 *plo,
                        float4 *phi, cudaStream_t st) {
  k_level_boxes<<<(nParent + 7) / 8, 256, 0, st>>>(clo, chi, nChild, nParent, plo, phi);
}
void launch_pack_rays(const RayStaging &S, uint32_t n, float4 *rays, cudaStream_t st) {
  k_pack_rays<<<(n + 255) / 256, 256, 0, st>>>(S, 0u, n, rays);
}
void launch_pack_rays_range(const RayStaging &S, uint32_t r0, uint32_t r1, float4 *rays, cudaStream_t st) {
  if (r1 > r0) k_pack_rays<<<(r1 - r0 + 255) / 256, 256, 0, st>>>(S, r0, r1, rays);
}

}  // namespace gvpm
