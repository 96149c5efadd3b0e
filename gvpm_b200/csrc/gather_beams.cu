// gather_beams.cu — G-Beams gather, beam3d and beam1d kernels (SURVEY.md §8 rows a13-a15).  Replaces, per iteration,
//   SubBeamBVH construction + buildHierarchy + query   photonmapper/beams_accel.h:90-243
//   BeamGradRadianceQuery::operator() and its shifts   gvpm/shift/shift_volume_beams.cpp:139-539,748-786
//   the gather loop of computeVolumeGradientBeams      gvpm/gvpm.cpp:880-986
//
// Hierarchy: beams are cut into sub-beams of avgLength/10 like the reference (beams_accel.h:98-124); the
// sub-beam midpoints are Morton-sorted and an implicit 32-ary AABB hierarchy is built over them (box of a
// sub-beam = its two r-cubes, beams_accel.h:222-231).
// k_beam_traverse: one warp per packet of 4 camera rays, same stackless ballot-mask walk as k_bre_traverse;
//   at a leaf lane c holds sub-beam c and keeps it as a candidate for ray j when the two supporting lines
//   pass within r of each other (relaxed, conservative).  Candidates go to the (ray, sub-beam) pair list.
// k_beam_shade: one thread per pair.  The kernel record of the WHOLE beam is evaluated in strictly rounded
//   fp32 / fp64 (cylinder intersection); the pair survives only in the sub-beam that owns tNear (half-open
//   [t1, t2), the reference's ownership rule :214-220 made exact at sub-beam boundaries), so each (ray, beam)
//   is counted once whatever the tree.  Then the functor with its 4 offsets, a segmented warp scan by ray,
//   and 27 float atomics per run.
#include "beam_device.cuh"
#include "launch_sizing.cuh"
#include "warp_ops.cuh"

namespace gvpm {

// raw sub-beam records -> Morton order
__global__ void k_sub_gather(const float4 *__restrict__ raw, const uint32_t *__restrict__ sorted, uint32_t n,
                             float4 *__restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = raw[sorted[i]];
}

// level 0: one warp per leaf of 32 sub-beams
__global__ void k_subbeam_leaf_boxes(const float4 *__restrict__ subs, const float4 *__restrict__ beams, uint32_t n,
                                     uint32_t nLeaves, float radius, float4 *__restrict__ lo,
                                     float4 *__restrict__ hi) {
  const uint32_t leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (leaf >= nLeaves) return;
  const uint32_t i = leaf * 32 + lane;
  float l[3] = {INFINITY, INFINITY, INFINITY}, h[3] = {-INFINITY, -INFINITY, -INFINITY};
  if (i < n) {
    const float4 s = subs[i];
    const uint32_t bi = __float_as_uint(s.z);
    const float4 b0 = beams[(size_t)bi * GVPM_BEAM_FLOAT4], b1 = beams[(size_t)bi * GVPM_BEAM_FLOAT4 + 1];
    const float o[3] = {b0.x, b0.y, b0.z}, d[3] = {b1.x, b1.y, b1.z};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float p1 = o[a] + d[a] * s.x, p2 = o[a] + d[a] * s.y;
      l[a] = fminf(p1, p2);
      h[a] = fmaxf(p1, p2);
    }
  }
  warp_box(l, h);
  if (lane == 0) {
    const float pad = radius * 1.0001f;
    lo[leaf] = make_float4(l[0] - pad, l[1] - pad, l[2] - pad, 0.f);
    hi[leaf] = make_float4(h[0] + pad, h[1] + pad, h[2] + pad, 0.f);
  }
}

constexpr int kBeamWarps = 4;
constexpr int BPK = GVPM_PACKET;

struct BeamTravShared {
  float4 ray[BPK][4];
  uint32_t queue[BPK][64];
  uint32_t mask[GVPM_MAX_LEVELS];
  uint32_t base[GVPM_MAX_LEVELS];
};

// Flush `take` queued candidates of one ray: lane = candidate.  Before a pair is written it passes the CHORD test - with
// all lanes busy here, where the leaf loop runs it for the rare lanes that pass the line test.
// Where can the beam run inside the cylinder around the camera LINE?  Around the beam parameter tc of the lines'
// closest approach, at most r / sin(theta) to either side: the chord [tN, tF].  The kernel record's tNear - the entry
// point, moved to an end cap when the camera SEGMENT starts or ends inside the chord (cylinder_intersection) - lies in
// it, as does the 1-D kernel's closest-approach parameter, and only the sub-beam that holds that parameter keeps the
// pair (ownership rule of k_beam_shade; sppm's per-sub-beam techniques intersect the sub-beam's own piece of the
// chord): a sub-beam the chord misses cannot contribute, nor can a chord that lies entirely in front of or behind the
// camera segment.  Relaxed arithmetic: the half-length is the largest a chord can have and is padded for the rounding
// of tc (amplified by 1 / sin^2); pairs closer to parallel than ~6 degrees are kept as they are.
__device__ __noinline__ uint32_t flush_beam_pairs(const GatherParams &P, const uint32_t *queue, uint32_t ray,
                                                  uint32_t qn, uint32_t take, int lane, const float4 *rayRec, float fpad) {
  qn -= take;
  bool keep = false;
  uint32_t si = 0;
  if ((uint32_t)lane < take) {
    si = queue[qn + lane];
    keep = true;
    const float4 sb = ldg4(P.subs + si);
    const uint32_t bi = __float_as_uint(sb.z), flags = __float_as_uint(sb.w);
    const float4 b0 = ldg4(P.beams + (size_t)bi * GVPM_BEAM_FLOAT4), b1 = ldg4(P.beams + (size_t)bi * GVPM_BEAM_FLOAT4 + 1);
    const float4 r0 = rayRec[0], r1 = rayRec[1], r2 = rayRec[2];
    const float cx = r1.y * b1.z - r1.z * b1.y, cy = r1.z * b1.x - r1.x * b1.z, cz = r1.x * b1.y - r1.y * b1.x;
    const float sin2 = cx * cx + cy * cy + cz * cz;
    if (sin2 >= 1e-2f) {
      const float wx = b0.x - r0.x, wy = b0.y - r0.y, wz = b0.z - r0.z;
      const float a = r1.x * b1.x + r1.y * b1.y + r1.z * b1.z;
      const float wd = wx * r1.x + wy * r1.y + wz * r1.z;
      const float wb = wx * b1.x + wy * b1.y + wz * b1.z;
      const float iA = 1.f / sin2;                      // sin2 = |d x b|^2 = 1 - (d.b)^2 for unit directions
      const float tc = (wd * a - wb) * iA;
      const float wmag = fabsf(wx) + fabsf(wy) + fabsf(wz);
      const float h = (P.radius + 4.f * fpad) * sqrtf(iA) * 1.01f + (1e-5f * iA) * (wmag + 1.f) + 1e-4f * fabsf(tc);
      const float tN = tc - h, tF = tc + h;
      if (!(flags & 2u) && tN > sb.y) keep = false;    // chord entirely behind this sub-beam
      if (!(flags & 1u) && tF < sb.x) keep = false;    // ... or entirely in front of it
      // camera distance of the beam point at the two chord ends (linear in between)
      const float zN = wd + tN * a, zF = wd + tF * a;
      // (+ r: sppm's per-sub-beam techniques put the cylinder around the BEAM; a camera point inside it and the beam
      // point it is closest to project onto the camera line within r of each other)
      const float padZ = 1e-4f * (1.f + fabsf(zN) + fabsf(zF)) + 16.f * fpad + P.radius;
      if (fmaxf(zN, zF) + padZ < r0.w || fminf(zN, zF) - padZ > fmaxf(r2.w, r1.w)) keep = false;
    }
  }
  const uint32_t km = __ballot_sync(0xffffffffu, keep);
  if (km) {
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(P.pair_counter, (unsigned long long)__popc(km));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (keep) {
      const unsigned long long idx = base + __popc(km & ((1u << lane) - 1u));
      if (idx < P.pair_cap) P.pairs[idx] = make_uint2(ray, si);
    }
  }
  __syncwarp();
  return qn;
}

__global__ void __launch_bounds__(kBeamWarps * 32, 6) k_beam_traverse(const __grid_constant__ GatherParams P) {
  __shared__ BeamTravShared sh[kBeamWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  BeamTravShared &S = sh[w];
  const Tree &T = P.tree;
  const int top = T.levels - 1;
  const uint32_t nPackets = (P.ray_end - P.ray_begin + BPK - 1) / BPK;
  const float coordMag = T.n ? __ldg(P.bounds + 6) : 0.f;
  float spreadMax = 16.f * P.radius;
  if (T.n) {
    const float ex = __ldg(P.bounds + 3) - __ldg(P.bounds), ey = __ldg(P.bounds + 4) - __ldg(P.bounds + 1),
                ez = __ldg(P.bounds + 5) - __ldg(P.bounds + 2);
    spreadMax = fmaxf(spreadMax, 0.01f * sqrtf(ex * ex + ey * ey + ez * ez));
  }
  for (;;) {
    uint32_t pk = 0;
    if (lane == 0) pk = atomicAdd(P.work_counter, 1u);
    pk = __shfl_sync(0xffffffffu, pk, 0);
    if (pk >= nPackets) break;
    const uint32_t r0 = P.ray_begin + pk * BPK;
    const int nr = min((uint32_t)BPK, P.ray_end - r0);
    __syncwarp();
    if (lane < 4 * nr) S.ray[lane >> 2][lane & 3] = ldg4(P.rays + (size_t)(r0 + (lane >> 2)) * GVPM_RAY_FLOAT4 + (lane & 3));
    __syncwarp();
    float ox[BPK], oy[BPK], oz[BPK], dx[BPK], dy[BPK], dz[BPK], mint[BPK], elen[BPK];
    int par[BPK], eid[BPK];
    uint32_t qn[BPK];
    uint32_t actMask = 0;
#pragma unroll
    for (int j = 0; j < BPK; ++j) {
      const int jj = j < nr ? j : 0;
      const float4 b0 = S.ray[jj][0], b1 = S.ray[jj][1], b2 = S.ray[jj][2], b3 = S.ray[jj][3];
      ox[j] = b0.x; oy[j] = b0.y; oz[j] = b0.z; mint[j] = b0.w;
      dx[j] = b1.x; dy[j] = b1.y; dz[j] = b1.z; elen[j] = fmaxf(b2.w, b1.w);   // edge length / maxt, whichever is larger
      par[j] = ((int)__float_as_uint(b3.y) + (int)__float_as_uint(b3.z)) % 2;
      eid[j] = (int)__float_as_uint(b3.w);
      qn[j] = 0;
      if (j < nr && T.n > 0 && elen[j] >= mint[j]) actMask |= 1u << j;
    }
    uint32_t groups[BPK];
    int ng = 0;
    float spread = 0.f;
    if (actMask) {
      const int c0 = __ffs(actMask) - 1;
      float cox = 0, coy = 0, coz = 0, cdx = 0, cdy = 0, cdz = 0, tEnd = 0;
#pragma unroll
      for (int j = 0; j < BPK; ++j) {
        if (j == c0) { cox = ox[j]; coy = oy[j]; coz = oz[j]; cdx = dx[j]; cdy = dy[j]; cdz = dz[j]; }
        if (actMask >> j & 1) tEnd = fmaxf(tEnd, elen[j]);
      }
      tEnd += P.radius;
#pragma unroll
      for (int j = 0; j < BPK; ++j)
        if (actMask >> j & 1) {
          const float ax = ox[j] - cox, ay = oy[j] - coy, az = oz[j] - coz;
          const float bx = ax + tEnd * (dx[j] - cdx), by = ay + tEnd * (dy[j] - cdy), bz = az + tEnd * (dz[j] - cdz);
          spread = fmaxf(spread, fmaxf(sqrtf(ax * ax + ay * ay + az * az), sqrtf(bx * bx + by * by + bz * bz)));
        }
      spread *= 1.0001f;
      if (spread <= spreadMax) {
        groups[ng++] = actMask;
      } else {
        spread = 0.f;
#pragma unroll
        for (int j = 0; j < BPK; ++j)
          if (actMask >> j & 1) groups[ng++] = 1u << j;
      }
    }
    // rounding pad of the packet (chord test at the flushes)
    float fpadPacket;
    {
      float om = 0.f, tm = 0.f;
#pragma unroll
      for (int j = 0; j < BPK; ++j)
        if (actMask >> j & 1) {
          om = fmaxf(om, fmaxf(fmaxf(fabsf(ox[j]), fabsf(oy[j])), fabsf(oz[j])));
          tm = fmaxf(tm, fabsf(elen[j]));
        }
      fpadPacket = (om + coordMag + tm + P.radius) * 3.8147e-6f;
    }
    for (int g = 0; g < ng; ++g) {
      const uint32_t gm = groups[g];
      const int c0 = __ffs(gm) - 1;
      float cox = 0, coy = 0, coz = 0, cdx = 1, cdy = 1, cdz = 1, tloG = 3.4e38f, thiG = -3.4e38f, omag = 0.f;
#pragma unroll
      for (int j = 0; j < BPK; ++j) {
        if (j == c0) { cox = ox[j]; coy = oy[j]; coz = oz[j]; cdx = dx[j]; cdy = dy[j]; cdz = dz[j]; }
        if (gm >> j & 1) {
          tloG = fminf(tloG, mint[j]);
          thiG = fmaxf(thiG, elen[j]);
          omag = fmaxf(omag, fmaxf(fmaxf(fabsf(ox[j]), fabsf(oy[j])), fabsf(oz[j])));
        }
      }
      const float fpad = (omag + coordMag + fabsf(thiG) + P.radius) * 3.8147e-6f;
      const float pad = fpad + ((gm & (gm - 1)) ? spread : 0.f);
      const float oxp = cox + pad, oxm = cox - pad, oyp = coy + pad, oym = coy - pad, ozp = coz + pad,
                  ozm = coz - pad;
      const float ix = 1.f / cdx, iy = 1.f / cdy, iz = 1.f / cdz;
      const float tlo = -4.f * fpad - P.radius;
      const float thi = thiG + P.radius + 4.f * fpad;
      const float rpad2 = (P.radius + 4.f * fpad) * (P.radius + 4.f * fpad);
      uint32_t cur, base = 0;
      int l = top;
      cur = __ballot_sync(0xffffffffu, (uint32_t)lane < T.cnt[top] &&
                                           box_hit(T, T.off[top] + lane, oxp, oxm, oyp, oym, ozp, ozm, ix, iy,
                                                   iz, tlo, thi));
      for (;;) {
        if (cur == 0) {
          if (l == top) break;
          ++l;
          cur = S.mask[l];
          base = S.base[l];
          continue;
        }
        const int c = __ffs(cur) - 1;
        cur &= cur - 1;
        const uint32_t node = base + c;
        if (l > 0) {
          S.mask[l] = cur;
          S.base[l] = base;
          --l;
          base = node << 5;
          const uint32_t idx = base + lane;
          cur = __ballot_sync(0xffffffffu, idx < T.cnt[l] && box_hit(T, T.off[l] + idx, oxp, oxm, oyp, oym, ozp,
                                                                       ozm, ix, iy, iz, tlo, thi));
          continue;
        }
        // ---- leaf: lane holds sub-beam (node*32 + lane) ----
        const uint32_t si = (node << 5) + lane;
        uint32_t cand = 0;
        if (si < T.n) {
          const float4 sb = ldg4(P.subs + si);
          const uint32_t bi = __float_as_uint(sb.z);
          const float4 b0 = ldg4(P.beams + (size_t)bi * GVPM_BEAM_FLOAT4), b1 = ldg4(P.beams + (size_t)bi * GVPM_BEAM_FLOAT4 + 1);
          const uint32_t meta = __float_as_uint(b1.w);
          const int type = meta & 3, depth = (meta >> 2) & 255, parity = (meta >> 10) & 1;
          const int m = P.cfg.lighting_mode;
          bool modeOk = true;
          if (!((m & GVPM_SURF2MEDIA) && (m & GVPM_MEDIA2MEDIA))) {
            if (type == GVPM_PARENT_MEDIUM && !(m & GVPM_MEDIA2MEDIA)) modeOk = false;
            if (type != GVPM_PARENT_MEDIUM && !(m & GVPM_SURF2MEDIA)) modeOk = false;
          }
#pragma unroll
          for (int j = 0; j < BPK; ++j) {
            // supporting lines within r of each other (cylinderIntersection's early test, relaxed + padded)
            const float cx = dy[j] * b1.z - dz[j] * b1.y, cy = dz[j] * b1.x - dx[j] * b1.z,
                        cz = dx[j] * b1.y - dy[j] * b1.x;
            const float sin2 = cx * cx + cy * cy + cz * cz;
            const float ad = (b0.x - ox[j]) * cx + (b0.y - oy[j]) * cy + (b0.z - oz[j]) * cz;
            bool ok = (gm >> j & 1) && (sin2 < 1e-6f || ad * ad < rpad2 * sin2 * 1.001f);
            // the filters only drop pairs (they never make one valid): keep them out of the pair list unless
            // the parity dump needs the geometric set
            if (P.beam_prefilter) {
              if (P.cfg.max_depth > 0 && eid[j] + depth > P.cfg.max_depth) ok = false;
              if (!modeOk) ok = false;
              if (P.cfg.path_set && parity != par[j]) ok = false;
            }
            if (ok) cand |= 1u << j;
          }
        }
        const uint32_t anyc = __reduce_or_sync(0xffffffffu, cand);
        if (anyc == 0) continue;
#pragma unroll
        for (int j = 0; j < BPK; ++j) {
          if (!(anyc >> j & 1)) continue;
          const bool c1 = cand >> j & 1;
          const uint32_t cmask = __ballot_sync(0xffffffffu, c1);
          if (c1) S.queue[j][qn[j] + __popc(cmask & ((1u << lane) - 1u))] = si;
          qn[j] += __popc(cmask);
          __syncwarp();
          if (qn[j] >= 32) qn[j] = flush_beam_pairs(P, S.queue[j], r0 + j, qn[j], 32, lane, S.ray[j], fpadPacket);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < BPK; ++j)
      if (qn[j] > 0) qn[j] = flush_beam_pairs(P, S.queue[j], r0 + j, qn[j], qn[j], lane, S.ray[j], fpadPacket);
  }
}

// Only ~40 % of the candidate pairs own a valid kernel record (the traversal tests the supporting LINES), so a kernel
// that runs the functor under `if (valid)` keeps 9 of 32 lanes busy (ncu: profiles/r2_beams.md).  Two phases per warp
// instead: phase 1, lane = candidate pair, evaluates the kernel record (fp64 cylinder island), the ownership rule and
// the filters with full lanes and appends the survivors to a per-warp ring in shared memory, in pair order; whenever
// the ring holds 32 survivors, phase 2 runs the functor (4 offsets, reconnections, shadow rays) for them with all
// lanes, then the segmented warp scan by ray and the float atomics.  Pair order is preserved, so a ray's survivors
// still form runs.
constexpr int kBeamRing = 64;
struct BeamShadeShared {
  uint32_t ray[kBeamRing], beam[kBeamRing];
  float f[9][kBeamRing];   // v, w, pdfKernel, pdfEdgeFailure, weightKernel, u, contrib.xyz
  float t[32][GVPM_OUT_FLOATS + 2];   // a batch's results, transposed reduction (odd row stride: no bank conflicts)
};

template <bool K1D>
__device__ __forceinline__ void beam_shade_batch(const GatherParams &P, BeamShadeShared &Q, uint32_t head, uint32_t cnt,
                                                 int lane) {
  float a[GVPM_OUT_FLOATS];
#pragma unroll
  for (int j = 0; j < GVPM_OUT_FLOATS; ++j) a[j] = 0.f;
  const bool valid = (uint32_t)lane < cnt;
  uint32_t key = 0xffffffffu;
  if (valid) {
    const uint32_t e = (head + lane) & (kBeamRing - 1);
    key = Q.ray[e];
    const float4 *rec = P.rays + (size_t)key * GVPM_RAY_FLOAT4;
    const BaseRay R = load_base_ray(rec);
    const BeamRec beam = load_beam(P, Q.beam[e]);
    BeamKernelRec kRec;
    kRec.v = sf(Q.f[0][e]); kRec.w = sf(Q.f[1][e]); kRec.pdfKernel = sf(Q.f[2][e]); kRec.pdfEdgeFailure = sf(Q.f[3][e]);
    kRec.weightKernel = sf(Q.f[4][e]); kRec.u = sf(Q.f[5][e]);
    kRec.contrib = v3(Q.f[6][e], Q.f[7][e], Q.f[8][e]);
    kRec.valid = true;
    beam_functor<K1D>(P, rec, R, beam, kRec, a);
  }
  // per-ray sums over runs of equal ray id, transposed through shared memory: lane j walks column j of the 32 x 27
  // results in pair order and adds a run's sum with one coalesced atomic instruction (a rolled loop: the 27 x 5
  // shuffle scan the other shade kernels use is 17 KB of code, and this kernel is bound by instruction fetch)
  const uint32_t kprev = __shfl_up_sync(0xffffffffu, key, 1);
  const uint32_t heads = __ballot_sync(0xffffffffu, lane == 0 || kprev != key);
#pragma unroll
  for (int j = 0; j < GVPM_OUT_FLOATS; ++j) Q.t[lane][j] = a[j];
  Q.t[lane][GVPM_OUT_FLOATS] = __uint_as_float(key);
  __syncwarp();
  if (lane < GVPM_OUT_FLOATS) {
    float acc = 0.f;
#pragma unroll 1
    for (uint32_t p = 0; p < cnt; ++p) {
      acc += Q.t[p][lane];
      if (p + 1 == cnt || (heads >> (p + 1) & 1u)) {
        if (acc != 0.f) atomicAdd(P.out + (size_t)__float_as_uint(Q.t[p][GVPM_OUT_FLOATS]) * GVPM_OUT_FLOATS + lane, acc);
        acc = 0.f;
      }
    }
  }
  __syncwarp();
}

template <bool K1D>
__global__ void __launch_bounds__(128, 3) k_beam_shade(const __grid_constant__ GatherParams P) {
  __shared__ BeamShadeShared ring[4];
  const int lane = threadIdx.x & 31;
  BeamShadeShared &Q = ring[threadIdx.x >> 5];
  uint32_t head = 0, qn = 0;
  unsigned long long total = *P.pair_counter;
  if (total > P.pair_cap) total = P.pair_cap;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  // one loop, one copy of each phase (the kernel's code size is what bounds it: instruction-fetch stalls)
  unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31);
  for (;;) {
    const bool more = i0 < total;
    if (!more && qn == 0u) break;
    const unsigned long long i = i0 + lane;
    i0 += stride;
    bool shade = false;
    uint32_t key = 0, bi = 0;
    BeamKernelRec kRec;
    if (more && i < total) {
      const uint2 pr = P.pairs[i];
      key = pr.x;
      const float4 sb = ldg4(P.subs + pr.y);
      bi = __float_as_uint(sb.z);
      const uint32_t flags = __float_as_uint(sb.w);
      const float4 *rec = P.rays + (size_t)key * GVPM_RAY_FLOAT4;
      const BaseRay R = load_base_ray(rec);
      const BeamRec beam = load_beam(P, bi);
      double tNear = 0.0;
      bool owner;
      if (K1D) {
        // 1-D kernel: the sub-beam [t1, t2] accepts v in (t1, t2] (beams_struct.h:299-301); first / last sub-beam
        // take the rest of (0, length)
        kRec = beam_kernel_eval_1d(P, beam, R);
        owner = ((flags & 1u) || kRec.v.v > sb.x) && ((flags & 2u) || kRec.v.v <= sb.y);
      } else {
        kRec = beam_kernel_eval(P, beam, R, bi, tNear);   // beam records keep the caller's order; only sub-beams are sorted
        // sub-beam ownership: half-open [t1, t2), first sub-beam also owns tNear < 0, last one the tail
        owner = ((flags & 1u) || tNear >= (double)sb.x) && ((flags & 2u) || tNear < (double)sb.y);
      }
      if (kRec.valid && owner) {
        const uint32_t meta = __float_as_uint(__ldg(&P.beams[(size_t)bi * GVPM_BEAM_FLOAT4 + 1].w));
        // depth / interaction-mode / pathSet filters of the beam functor (shift_volume_beams.cpp:143-187;
        // no minDepth test here: the driver skips camera edges instead, gvpm.cpp:922)
        bool contributes = true;
        {
          const int type = meta & 3, depth = (meta >> 2) & 255, parity = (meta >> 10) & 1;
          if (P.cfg.max_depth > 0 && R.edgeId + depth > P.cfg.max_depth) contributes = false;
          const int m = P.cfg.lighting_mode;
          if (!((m & GVPM_SURF2MEDIA) && (m & GVPM_MEDIA2MEDIA))) {
            if (type == GVPM_PARENT_MEDIUM && !(m & GVPM_MEDIA2MEDIA)) contributes = false;
            if (type != GVPM_PARENT_MEDIUM && !(m & GVPM_SURF2MEDIA)) contributes = false;
          }
          if (P.cfg.path_set && parity != ((R.px + R.py) % 2)) contributes = false;
        }
        if (P.counts) {
          atomicAdd(P.counts + 2 * (size_t)key, 1u);
          if (contributes) atomicAdd(P.counts + 2 * (size_t)key + 1, 1u);
        }
        if (P.dump_pairs) {
          const unsigned long long slot = atomicAdd(P.dump_counter, 1ull);
          if (slot < P.dump_cap) P.dump_pairs[slot] = make_uint2(key, bi | (contributes ? 0x80000000u : 0u));
        } else {
          shade = contributes;
        }
      }
    }
    if (P.dump_pairs) { if (!more) break; continue; }
    const uint32_t m = __ballot_sync(0xffffffffu, shade);
    if (shade) {
      const uint32_t e = (head + qn + __popc(m & ((1u << lane) - 1u))) & (kBeamRing - 1);
      Q.ray[e] = key; Q.beam[e] = bi;
      Q.f[0][e] = kRec.v.v; Q.f[1][e] = kRec.w.v; Q.f[2][e] = kRec.pdfKernel.v; Q.f[3][e] = kRec.pdfEdgeFailure.v;
      Q.f[4][e] = kRec.weightKernel.v; Q.f[5][e] = kRec.u.v;
      Q.f[6][e] = kRec.contrib.x.v; Q.f[7][e] = kRec.contrib.y.v; Q.f[8][e] = kRec.contrib.z.v;
    }
    qn += __popc(m);
    __syncwarp();
    if (qn >= 32u || (!more && qn > 0u)) {   // a full batch, or what is left once the pair list is exhausted
      const uint32_t take = min(qn, 32u);
      beam_shade_batch<K1D>(P, Q, head, take, lane);
      head = (head + take) & (kBeamRing - 1);
      qn -= take;
      __syncwarp();
    }
  }
}

// sppm primal photon beams (volumePhotonBeamPass, sppm.cpp:823-860): one thread per (camera beam, sub-beam) candidate
// of the same traversal; the functor of technique P.sppm_beam_technique, the depth window of sppm.cpp:853-854,
// Li * beam.weight reduced per ray by a segmented warp scan, 3 float atomics per run.  P.out is [n_rays][3].
__global__ void __launch_bounds__(128, 4) k_beam_shade_sppm(const __grid_constant__ GatherParams P) {
  const int lane = threadIdx.x & 31;
  unsigned long long total = *P.pair_counter;
  if (total > P.pair_cap) total = P.pair_cap;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < total;
       i0 += stride) {
    const unsigned long long i = i0 + lane;
    const bool valid = i < total;
    float a[3] = {0.f, 0.f, 0.f};
    uint32_t key = 0xffffffffu;
    if (valid) {
      const uint2 pr = P.pairs[i];
      key = pr.x;
      const float4 sb = ldg4(P.subs + pr.y);
      const uint32_t bi = __float_as_uint(sb.z);
      const BaseRay R = load_base_ray(P.rays + (size_t)key * GVPM_RAY_FLOAT4);
      // only origin / direction / length / flux / depth of the record are read
      const float4 *b = P.beams + (size_t)bi * GVPM_BEAM_FLOAT4;
      const float4 b0 = ldg4(b), b1 = ldg4(b + 1), b2 = ldg4(b + 2);
      BeamRec beam;
      beam.o = v3(b0.x, b0.y, b0.z); beam.length = sf(b0.w);
      beam.dir = v3(b1.x, b1.y, b1.z);
      beam.flux = v3(b2.x, b2.y, b2.z);
      const int depth = (__float_as_uint(b1.w) >> 2) & 255;
      v3 Li;
      if (sppm_beam_functor(P, R, beam, bi, sb, Li)) {
        const int maxDepthQ = P.cfg.max_depth == -1 ? -1 : P.cfg.max_depth - R.edgeId;
        const int minDepthQ = max(0, P.cfg.min_depth - R.edgeId);
        const bool contributes = !(maxDepthQ != -1 && depth > maxDepthQ) && !(minDepthQ != 0 && depth < minDepthQ);
        if (P.counts) {
          atomicAdd(P.counts + 2 * (size_t)key, 1u);
          if (contributes) atomicAdd(P.counts + 2 * (size_t)key + 1, 1u);
        }
        if (P.dump_pairs) {
          const unsigned long long slot = atomicAdd(P.dump_counter, 1ull);
          if (slot < P.dump_cap) P.dump_pairs[slot] = make_uint2(key, bi | (contributes ? 0x80000000u : 0u));
        } else if (contributes) {
          const v3 c = Li * R.eye;
          a[0] = c.x.v; a[1] = c.y.v; a[2] = c.z.v;
        }
      }
    }
    if (P.dump_pairs) continue;
    warp_run_sum<3, true>(key, a, valid, P.out, lane);
  }
}

// ---- host-side launchers -----------------------------------------------------------------------
void launch_sub_gather(const float4 *raw, const uint32_t *sorted, uint32_t n, float4 *out, cudaStream_t st) {
  if (n) k_sub_gather<<<(n + 255) / 256, 256, 0, st>>>(raw, sorted, n, out);
}
void launch_subbeam_leaf_boxes(const float4 *subs, const float4 *beams, uint32_t n, uint32_t nLeaves, float radius,
                               float4 *lo, float4 *hi, cudaStream_t st) {
  if (nLeaves) k_subbeam_leaf_boxes<<<(nLeaves + 7) / 8, 256, 0, st>>>(subs, beams, n, nLeaves, radius, lo, hi);
}

cudaError_t launch_beam_traverse(const GatherParams &P, int sm_count, cudaStream_t stream) {
  if (P.ray_end <= P.ray_begin) return cudaSuccess;
  const unsigned packets = (P.ray_end - P.ray_begin + BPK - 1) / BPK;
  const unsigned need = (packets + kBeamWarps - 1) / kBeamWarps;   // persistent: warps pull packets from a counter
  k_beam_traverse<<<persistent_grid<k_beam_traverse>(sm_count, kBeamWarps * 32, need), kBeamWarps * 32, 0, stream>>>(P);
  return cudaGetLastError();
}
cudaError_t launch_beam_shade(const GatherParams &P, unsigned long long total, int sm_count, cudaStream_t stream) {
  if (total == 0) return cudaSuccess;
  if (P.cfg.beam_kernel_1d) k_beam_shade<true><<<stride_grid<k_beam_shade<true>>(sm_count, 128, total), 128, 0, stream>>>(P);
  else k_beam_shade<false><<<stride_grid<k_beam_shade<false>>(sm_count, 128, total), 128, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_beam_shade_sppm(const GatherParams &P, unsigned long long total, int sm_count, cudaStream_t stream) {
  if (total == 0) return cudaSuccess;
  k_beam_shade_sppm<<<stride_grid<k_beam_shade_sppm>(sm_count, 128, total), 128, 0, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace gvpm
