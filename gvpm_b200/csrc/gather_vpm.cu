// gather_vpm.cu — G-VPM point gather (SURVEY.md §8 row a12).  Replaces, for every camera distance
// sample of an iteration,
//   GPhotonMap::evaluate -> PointKDTree::executeQuery   gvpm/gvpm_accel.h:111, include/mitsuba/core/kdtree.h:675-731
//   VolumeGradientPositionQuery::operator()            gvpm/shift/shift_volume_photon.cpp:489-655
//   the per-sample accumulation of computeVolumeGradientPhoton   gvpm/gvpm.cpp:1141-1185
//
// k_vpm_traverse: one warp per distance sample.  The query point o + t*d is formed in strictly rounded
//   arithmetic; the warp descends the implicit 32-ary hierarchy (boxes inflated by the build radius,
//   which must be >= every sample radius) with a point-in-box test per lane, and at a leaf lane c tests
//   photon c with the kd-tree's predicate |p - q|^2 < r^2 (kdtree.h:721-723).  `found` (the reference's
//   MVol increment) is counted before the depth / interaction-mode filters; contributing photons go to
//   the (sample, photon) pair list.
// k_vpm_shade: one thread per pair, same structure as k_bre_shade; the per-sample results are scaled by
//   1/nbCameraSamples and folded into the ray's 27 accumulators.
#include "bre_device.cuh"
#include "launch_sizing.cuh"
#include "warp_ops.cuh"

namespace gvpm {

struct VpmShared {
  uint32_t queue[64];
  uint32_t mask[GVPM_MAX_LEVELS];
  uint32_t base[GVPM_MAX_LEVELS];
};

constexpr int kVpmWarps = 4;

template <bool DUMP>
__global__ void __launch_bounds__(kVpmWarps * 32, 8) k_vpm_traverse(const __grid_constant__ GatherParams P) {
  __shared__ VpmShared sh[kVpmWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  VpmShared &S = sh[w];
  const Tree &T = P.tree;
  const int top = T.levels - 1;
  const float coordMag = T.n ? __ldg(P.bounds + 6) : 0.f;

  for (;;) {
    uint32_t si = 0;
    if (lane == 0) si = atomicAdd(P.work_counter, 1u);
    si = __shfl_sync(0xffffffffu, si, 0);
    if (si >= P.n_samples) break;
    const float4 s0 = ldg4(P.samples + 2 * (size_t)si), s1 = ldg4(P.samples + 2 * (size_t)si + 1);
    const uint32_t ray = __float_as_uint(s1.w);
    const float4 *rec = P.rays + (size_t)ray * GVPM_RAY_FLOAT4;
    const float4 b0 = ldg4(rec), b1 = ldg4(rec + 1), b3 = ldg4(rec + 3);
    const sf t(s0.x), r(s0.w);
    const v3 q = v3(b0.x, b0.y, b0.z) + t * v3(b1.x, b1.y, b1.z);  // ray.o + mRec.t * ray.d, gvpm.cpp:1174
    const sf rr2 = r * r;
    const int edgeId = (int)__float_as_uint(b3.w);
    uint32_t found = 0, ncontrib = 0, qn = 0;

    if (T.n > 0) {
      // point-in-box against boxes inflated by the build radius; pad covers the rounding of q
      const float pad = (fabsf(q.x.v) + fabsf(q.y.v) + fabsf(q.z.v) + coordMag) * 3.8147e-6f +
                        fmaxf(r.v - P.radius, 0.f);
      const float qxp = q.x.v + pad, qxm = q.x.v - pad, qyp = q.y.v + pad, qym = q.y.v - pad, qzp = q.z.v + pad,
                  qzm = q.z.v - pad;
      auto inbox = [&](uint32_t i) {
        const float4 lo = ldg4(T.lo + i), hi = ldg4(T.hi + i);
        return lo.x <= qxp && hi.x >= qxm && lo.y <= qyp && hi.y >= qym && lo.z <= qzp && hi.z >= qzm;
      };
      uint32_t cur, base = 0;
      int l = top;
      cur = __ballot_sync(0xffffffffu, (uint32_t)lane < T.cnt[top] && inbox(T.off[top] + lane));
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
          cur = __ballot_sync(0xffffffffu, idx < T.cnt[l] && inbox(T.off[l] + idx));
          continue;
        }
        const uint32_t pi = (node << 5) + lane;
        bool geom = false, contrib = false;
        if (pi < T.n) {
          const float4 q0 = ldg4(P.planes + pi);
          geom = length_sq(v3(q0.x, q0.y, q0.z) - q) < rr2;  // kdtree.h:721-723
          if (geom) {
            const uint32_t meta = __float_as_uint(q0.w);
            const int type = meta & 3, depth = (meta >> 2) & 255;
            contrib = true;
            if (P.cfg.max_depth > 0 && edgeId + depth > P.cfg.max_depth) contrib = false;  // :503-505
            const int m = P.cfg.lighting_mode;
            if (!((m & GVPM_SURF2MEDIA) && (m & GVPM_MEDIA2MEDIA))) {
              if (type == GVPM_PARENT_MEDIUM && !(m & GVPM_MEDIA2MEDIA)) contrib = false;
              if (type != GVPM_PARENT_MEDIUM && !(m & GVPM_SURF2MEDIA)) contrib = false;
            }
          }
        }
        const uint32_t gmask = __ballot_sync(0xffffffffu, geom), cmask = __ballot_sync(0xffffffffu, contrib);
        if (DUMP) {
          if (geom) {
            const uint32_t rank = __popc(gmask & ((1u << lane) - 1u));
            P.nbr_idx[P.nbr_offsets[si] + found + rank] = P.orig[pi] | (contrib ? 0x80000000u : 0u);
          }
        }
        found += __popc(gmask);
        ncontrib += __popc(cmask);
        if (DUMP || cmask == 0) continue;
        if (contrib) S.queue[qn + __popc(cmask & ((1u << lane) - 1u))] = pi;
        qn += __popc(cmask);
        __syncwarp();
        if (qn >= 32) {
          unsigned long long bs = 0;
          if (lane == 0) bs = atomicAdd(P.pair_counter, 32ull);
          bs = __shfl_sync(0xffffffffu, bs, 0);
          qn -= 32;
          if (bs + lane < P.pair_cap) P.pairs[bs + lane] = make_uint2(si, S.queue[qn + lane]);
          __syncwarp();
        }
      }
      if (!DUMP && qn > 0) {
        unsigned long long bs = 0;
        if (lane == 0) bs = atomicAdd(P.pair_counter, (unsigned long long)qn);
        bs = __shfl_sync(0xffffffffu, bs, 0);
        if ((uint32_t)lane < qn && bs + lane < P.pair_cap) P.pairs[bs + lane] = make_uint2(si, S.queue[lane]);
        __syncwarp();
      }
    }
    if (lane == 0) {
      if (P.sample_counts) {
        P.sample_counts[2 * (size_t)si] = found;
        P.sample_counts[2 * (size_t)si + 1] = ncontrib;
      }
      if (!DUMP && P.mvol && found) atomicAdd(P.mvol + ray, found);  // MVol += evaluate(...), gvpm.cpp:1175
    }
  }
}

// VolumeGradientPositionQuery::operator() for one (sample, photon) pair, after the filters.
template <bool BVH>
__device__ __forceinline__ void vpm_photon(const GatherParams &P, const float4 *__restrict__ rec, float4 s0,
                                           float4 s1, uint32_t pi, float *a) {
  const BaseRay R = load_base_ray(rec);
  const PhotonRec ph = load_photon(P, pi);
  const sf t(s0.x), pdfSuccess(s0.y), pdfSel(s0.z), r(s0.w);
  const sf rr2 = r * r;
  const v3 Tbase(s1.x, s1.y, s1.z);
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);
  const v3 q = R.o + t * R.d;
  const v3 wi = ph.wi;
  const v3 photonContrib = (sigS * ph.flux) * phase_eval(P, wi, -R.d);
  const v3 baseContrib = (R.eye * Tbase) * photonContrib;  // :529
  // Float kernelVol = (4.0/3.0) * M_PI * pow(searchRadius, 3) in double (:530)
  const double rd = (double)r.v;
  const sf kernelVol((float)((4.0 / 3.0) * (double)GVPM_PI * (rd * rd * rd)));
  const sf pdfBase = pdfSuccess * pdfSel;
  const sf recip = sf(1.f) / (kernelVol * pdfBase);
  acc_add(a, 0, baseContrib * recip);
  const OccluderNear near = pair_occluders<BVH>(P, ph.parent, ph.lBase);

  float Sx[4], Sy[4], Sz[4], Wk[4];
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    const float4 o0 = ldg4(rec + 4 * (k + 1)), o1 = ldg4(rec + 4 * (k + 1) + 1), o2 = ldg4(rec + 4 * (k + 1) + 2);
    sf weight(1.f);
    v3 S(0.f, 0.f, 0.f);
    const sf lenK(o0.w);
    if (__float_as_uint(o2.w) != 0u && lenK >= t) {  // validVolumeEdge && shiftDistMax >= baseRay.maxt, :543-553
      const v3 ok(o0.x, o0.y, o0.z), dk(o1.x, o1.y, o1.z), eyeK(o2.x, o2.y, o2.z);
      const sf sensor(o1.w);
      // shiftMRec[k]: medium->eval(shiftRay, ., EDistanceAlwaysValid) with mRec.t = t (homogeneous.cpp:468-476)
      const sf st(P.sigma_t[0]);
      const sf maxDist = lenK - sf(P.cfg.epsilon);
      const sf normalization = sf(1.f) - sf(expf(((-st) * maxDist).v));
      sf Tk(expf(((-st) * t).v));
      sf x = (st / normalization) * Tk;
      const sf pdfShift = (((x + x) + x) / sf(3.f)) * pdfSel;
      if (Tk.v < 1e-20f) Tk = sf(0.f);
      const v3 zShift = ok + t * dk;
      if (P.cfg.use_shift_null && length_sq(ph.p - zShift) < rr2) {  // :584-602
        shift_null(P, ph.flux, wi, dk, eyeK, sensor, Tk, pdfBase, pdfShift, S, weight);
      } else {  // :604-639
        const v3 offsetPos = get_shift_pos(P, rr2, ph.p, q, zShift, R.d, dk, false);
        shift_photon_diffuse<BVH>(P, ph, near, offsetPos, dk, eyeK, sensor, Tk, pdfBase, pdfShift, S, weight);
      }
    }
    if ((k == 1 && R.px == P.cfg.film_w - 1) || (k == 2 && R.py == P.cfg.film_h - 1)) weight = sf(1.f);
    Sx[k] = S.x.v; Sy[k] = S.y.v; Sz[k] = S.z.v; Wk[k] = weight.v;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const sf wk(Wk[k]);
    acc_add(a, 1 + k, (v3(Sx[k], Sy[k], Sz[k]) * wk) * recip);
    acc_add(a, 5 + k, (baseContrib * wk) * recip);
  }
}

// BVH: shadow rays walk the occluder BVH (occluder_device.cuh)
template <bool BVH>
__global__ void __launch_bounds__(128, 4) k_vpm_shade(const __grid_constant__ GatherParams P) {
  const int lane = threadIdx.x & 31;
  unsigned long long total = *P.pair_counter;
  if (total > P.pair_cap) total = P.pair_cap;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  const float normalization = P.vpm_normalization;  // 1.f / nbCameraSamples, gvpm.cpp:1132
  for (unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < total;
       i0 += stride) {
    const unsigned long long i = i0 + lane;
    const bool valid = i < total;
    float a[GVPM_OUT_FLOATS];
#pragma unroll
    for (int j = 0; j < GVPM_OUT_FLOATS; ++j) a[j] = 0.f;
    uint32_t key = 0xffffffffu;
    if (valid) {
      const uint2 pr = P.pairs[i];
      const float4 s0 = ldg4(P.samples + 2 * (size_t)pr.x), s1 = ldg4(P.samples + 2 * (size_t)pr.x + 1);
      key = __float_as_uint(s1.w);
      vpm_photon<BVH>(P, P.rays + (size_t)key * GVPM_RAY_FLOAT4, s0, s1, pr.y, a);
#pragma unroll
      for (int j = 0; j < GVPM_OUT_FLOATS; ++j) a[j] *= normalization;
    }
    // per-ray sums over runs of equal ray index (samples of a ray are adjacent)
    warp_run_sum(key, a, valid, P.out, lane);
  }
}

cudaError_t launch_vpm_traverse(const GatherParams &P, bool dump, int sm_count, cudaStream_t stream) {
  if (P.n_samples == 0) return cudaSuccess;
  const unsigned need = (P.n_samples + kVpmWarps - 1) / kVpmWarps;   // persistent: warps pull samples from a counter
  if (dump) k_vpm_traverse<true><<<persistent_grid<k_vpm_traverse<true>>(sm_count, kVpmWarps * 32, need), kVpmWarps * 32, 0, stream>>>(P);
  else k_vpm_traverse<false><<<persistent_grid<k_vpm_traverse<false>>(sm_count, kVpmWarps * 32, need), kVpmWarps * 32, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_vpm_shade(const GatherParams &P, unsigned long long total, int sm_count, cudaStream_t stream) {
  if (total == 0) return cudaSuccess;
  if (P.occ_nodes) k_vpm_shade<true><<<stride_grid<k_vpm_shade<true>>(sm_count, 128, total), 128, 0, stream>>>(P);
  else k_vpm_shade<false><<<stride_grid<k_vpm_shade<false>>(sm_count, 128, total), 128, 0, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace gvpm
