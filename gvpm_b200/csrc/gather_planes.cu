// gather_planes.cu — G-Planes 0D gather (SURVEY.md §8 row a16).  Replaces, per iteration,
//   PhotonPlaneBVH construction + buildHierarchy + query    photonmapper/plane_accel.h:84-211
//   PlaneGradRadianceQuery::operator() / specularShift      gvpm/shift/shift_volume_planes.h:57-101,263-453
//   the gather loop of computeVolumeGradientPlanes          gvpm/gvpm.cpp:782-878
//
// Photon planes are LARGE primitives (both edges are free-flight distances of the medium): a camera ray crosses a
// sizeable fraction of all planes, so the gather is dense (ray x plane) work, not a sparse search, and a pair list
// as the point / beam gathers use would not fit in memory.  Design:
//   build   Morton sort of the plane centres -> sorted SoA records (6 float4 planes) + one AABB per leaf of 32
//           planes (corners of the parallelograms, PhotonPlane::getAABB plane_struct.h:68-74).
//   gather  k_plane_gather: a CTA owns a block of 128 camera rays, ONE RAY PER LANE, 27 accumulators in registers
//           (no atomics, no cross-lane reduction, one coalesced 108-byte store per ray at the end).  The sorted planes
//           stream through shared memory in chunks; leaves whose box misses the (padded) bounds of the CTA's ray
//           block are skipped.  Phase A: every lane tests its ray against the chunk's planes (plane data broadcast
//           from shared memory, relaxed FMA arithmetic with conservative margins) and pushes candidates into its own
//           shared-memory queue.  Phase B: lanes pop their queues and run the strictly rounded intersection + the
//           functor with its 4 specular shifts, so the divergent, transcendental-heavy shading runs with (nearly)
//           full lanes although only ~1 in 10 tests hits.
#include "launch_sizing.cuh"
#include "plane_device.cuh"
#include "warp_ops.cuh"

namespace gvpm {

// ---- build ---------------------------------------------------------------------------------------------------
// raw: caller-order AoS records (6 float4 per plane) -> Morton-sorted SoA planes + original index
__global__ void k_plane_pack_sorted(const float4 *__restrict__ raw, const uint32_t *__restrict__ sorted, uint32_t n,
                                    float4 *__restrict__ planes, uint32_t *__restrict__ orig) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = sorted[i];
  orig[i] = s;
#pragma unroll
  for (int k = 0; k < GVPM_PLANE_PLANES; ++k) planes[(size_t)k * n + i] = raw[(size_t)s * GVPM_PLANE_PLANES + k];
}

// one warp per leaf of 32 planes: AABB of the 4 corners of every parallelogram
__global__ void k_plane_leaf_boxes(const float4 *__restrict__ planes, uint32_t n, uint32_t nLeaves,
                                   float4 *__restrict__ lo, float4 *__restrict__ hi) {
  const uint32_t leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (leaf >= nLeaves) return;
  const uint32_t i = leaf * 32 + lane;
  float l[3] = {INFINITY, INFINITY, INFINITY}, h[3] = {-INFINITY, -INFINITY, -INFINITY};
  if (i < n) {
    const float4 q0 = planes[i], q1 = planes[(size_t)n + i], q2 = planes[2 * (size_t)n + i];
    const float o[3] = {q0.x, q0.y, q0.z}, a[3] = {q1.x, q1.y, q1.z}, b[3] = {q2.x, q2.y, q2.z};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float p0 = o[c], p1 = o[c] + a[c], p2 = o[c] + b[c], p3 = o[c] + a[c] + b[c];
      l[c] = fminf(fminf(p0, p1), fminf(p2, p3));
      h[c] = fmaxf(fmaxf(p0, p1), fmaxf(p2, p3));
    }
  }
  warp_box(l, h);
  if (lane == 0) {
    lo[leaf] = make_float4(l[0], l[1], l[2], 0.f);
    hi[leaf] = make_float4(h[0], h[1], h[2], 0.f);
  }
}

// ---- gather --------------------------------------------------------------------------------------------------
constexpr int kPlWarps = 4;               // 128 rays per CTA
constexpr int kPlChunk = 512;             // planes staged per chunk (16 leaves)
constexpr int kPlLeaves = kPlChunk / 32;
constexpr int kPlQCap = 96;               // candidate queue entries per lane (52 KB of shared memory per CTA: 4 CTAs per SM)
constexpr int kPlSub = 64;                // planes tested between queue-level checks
static_assert(kPlQCap > kPlSub, "queue must hold one sub-step");
static_assert(kPlWarps == 4 && (kPlChunk / kPlWarps) % 32 == 0, "the bundle test splits a chunk over four warps");

struct PlaneShared {
  float4 tst[kPlChunk][3];                       // Q0-Q2 of the staged chunk
  uint16_t queue[kPlWarps][kPlQCap][32];         // per-lane candidate queues (chunk-relative plane index)
  float red[kPlWarps][6];                        // ray-block bounds reduction
  float bounds[6];
  float tred[kPlWarps][8];                       // ray-bundle reduction: xmin, xmax, ymin, ymax, delta, mint min, maxt max, cos min
  float bundle[8];
  uint16_t live[kPlChunk];                       // planes of the chunk the bundle test keeps (chunk-relative, ascending)
  uint16_t liveW[kPlWarps][kPlChunk / kPlWarps]; // per-warp part of it
  uint32_t nLive;
  uint32_t amask[kPlWarps];
  uint32_t leafMask;
  uint32_t block;
};

// Bundle test: can ANY ray of the CTA's ray block meet the plane?  The rays of a block start (nearly) in one point c0
// (primary rays of a pinhole; delta = largest distance of an origin to c0) and their directions lie in the pyramid
// spanned by four corner directions dk.  For rays through c0 the plane coordinates t0 = (d.A)/(d.N), t1 = (d.B)/(d.N)
// (A = e1 x T, B = T x e0, N = e1 x e0, T = c0 - ori) are linear-fractional in d: where d.N keeps its sign over the
// pyramid their extremes are taken at the corners, so the plane is out of every ray's reach when all four corners
// put t0 (or t1) on the same side of [0, 1].  Conservative: slack for delta and rounding, planes whose d.N changes
// sign (or nearly vanishes) are kept.  Everything kept goes through plane_candidate and the strict test per ray.
__device__ __forceinline__ bool plane_bundle_reject(const float4 q0, const float4 q1, const float4 q2, const float *c0,
                                                    const float (*dk)[3], float delta) {
  const float tx = c0[0] - q0.x, ty = c0[1] - q0.y, tz = c0[2] - q0.z;
  const float nx = q2.y * q1.z - q2.z * q1.y, ny = q2.z * q1.x - q2.x * q1.z, nz = q2.x * q1.y - q2.y * q1.x;   // e1 x e0
  const float ax = q2.y * tz - q2.z * ty, ay = q2.z * tx - q2.x * tz, az = q2.x * ty - q2.y * tx;               // e1 x T
  const float bx = ty * q1.z - tz * q1.y, by = tz * q1.x - tx * q1.z, bz = tx * q1.y - ty * q1.x;               // T x e0
  const float tn = fabsf(tx) + fabsf(ty) + fabsf(tz);
  // |a| error: (delta + rounding of T) * |d| * |e1|; q0.w = |e0|, q1.w = |e1|, |dk| <= 2
  const float sa = 2.f * (delta + 4e-6f * tn) * q1.w, sb = 2.f * (delta + 4e-6f * tn) * q0.w;
  bool pos = true, neg = true, a_lo = true, a_hi = true, b_lo = true, b_hi = true;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float det = dk[k][0] * nx + dk[k][1] * ny + dk[k][2] * nz;
    const float a = dk[k][0] * ax + dk[k][1] * ay + dk[k][2] * az;
    const float b = dk[k][0] * bx + dk[k][1] * by + dk[k][2] * bz;
    const float ad = fabsf(det), tiny = 1e-4f * q0.w * q1.w;
    pos = pos && det > tiny;
    neg = neg && det < -tiny;
    const float s = det < 0.f ? -1.f : 1.f;
    const float e = 1e-3f * ad;
    a_lo = a_lo && a * s < -(e + sa);
    a_hi = a_hi && (a * s - ad) > (e + sa);
    b_lo = b_lo && b * s < -(e + sb);
    b_hi = b_hi && (b * s - ad) > (e + sb);
  }
  return (pos || neg) && (a_lo || a_hi || b_lo || b_hi);
}

// relaxed conservative form of intersectPlane0D: never rejects a pair the strictly rounded test accepts.
// Margins: the relaxed (FMA) and the strict evaluations of det, T.P, d.Q, e1.Q each differ from the exact value by
// at most ~12 ulp-of-magnitude; kEps covers twice that with slack.
__device__ __forceinline__ bool plane_candidate(const float4 q0, const float4 q1, const float4 q2, float ox, float oy,
                                                float oz, float dx, float dy, float dz, float mint, float maxt) {
  constexpr float kEps = 4e-6f;
  const float px = dy * q2.z - dz * q2.y, py = dz * q2.x - dx * q2.z, pz = dx * q2.y - dy * q2.x;
  const float det = q1.x * px + q1.y * py + q1.z * pz;
  const float ad = fabsf(det);
  const float l01 = q0.w * q1.w;
  const float dd = kEps * l01;
  if (ad + dd < 1e-5f) return false;
  if (ad <= dd) return true;  // sign of det uncertain: let the strict test decide
  const float tx = ox - q0.x, ty = oy - q0.y, tz = oz - q0.z;
  const float tn = kEps * (fabsf(tx) + fabsf(ty) + fabsf(tz));
  const float s = det < 0.f ? -1.f : 1.f;
  const float hiB = ad * (1.f + kEps) + dd;
  const float a0 = (tx * px + ty * py + tz * pz) * s;
  const float d0 = tn * q1.w;
  if (a0 < -d0 || a0 > hiB + d0) return false;
  const float qx = ty * q1.z - tz * q1.y, qy = tz * q1.x - tx * q1.z, qz = tx * q1.y - ty * q1.x;
  const float a1 = (dx * qx + dy * qy + dz * qz) * s;
  const float d1 = tn * q0.w;
  if (a1 < -d1 || a1 > hiB + d1) return false;
  const float ac = (q2.x * qx + q2.y * qy + q2.z * qz) * s;
  const float dc = tn * l01 + kEps * fabsf(ac);
  if (ac + dc <= mint * (ad - dd)) return false;
  if (ac - dc >= maxt * (ad + dd)) return false;
  return true;
}

template <bool kDump>
__global__ void __launch_bounds__(kPlWarps * 32, 4) k_plane_gather(const __grid_constant__ GatherParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PlaneShared &S = *reinterpret_cast<PlaneShared *>(smem_raw);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const uint32_t nPl = P.n_planes;
  const uint32_t nBlocks = (P.n_rays + kPlWarps * 32 - 1) / (kPlWarps * 32);
  const uint32_t nLeavesTotal = (nPl + 31) / 32;
  const float4 *Q = P.plane_rec;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) S.block = atomicAdd(P.work_counter, 1u);
    __syncthreads();
    const uint32_t blk = S.block;
    if (blk >= nBlocks) break;
    const uint32_t ray = blk * (kPlWarps * 32) + threadIdx.x;
    const bool haveRay = ray < P.n_rays;
    const float4 *rec = P.rays + (size_t)(haveRay ? ray : 0) * GVPM_RAY_FLOAT4;
    const float4 b0 = ldg4(rec), b1 = ldg4(rec + 1);
    const float ox = b0.x, oy = b0.y, oz = b0.z, mint = b0.w, dx = b1.x, dy = b1.y, dz = b1.z, maxt = b1.w;
    const bool active = haveRay && maxt > mint;
    // bounds of the CTA's ray segments (padded: the strictly rounded tCam of a grazing plane can be off by a few
    // per cent of the segment, DESIGN.md §4)
    {
      float l[3] = {INFINITY, INFINITY, INFINITY}, h[3] = {-INFINITY, -INFINITY, -INFINITY};
      if (active) {
        const float len = maxt - mint, t0 = mint - 0.05f * len, t1 = maxt + 0.05f * len;
        const float o[3] = {ox, oy, oz}, d[3] = {dx, dy, dz};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float pa = o[c] + d[c] * t0, pb = o[c] + d[c] * t1;
          l[c] = fminf(pa, pb);
          h[c] = fmaxf(pa, pb);
        }
      }
      warp_box(l, h);
      if (lane == 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) { S.red[w][c] = l[c]; S.red[w][3 + c] = h[c]; }
      }
      __syncthreads();
      if (threadIdx.x < 6) {
        float v = S.red[0][threadIdx.x];
        for (int i = 1; i < kPlWarps; ++i)
          v = threadIdx.x < 3 ? fminf(v, S.red[i][threadIdx.x]) : fmaxf(v, S.red[i][threadIdx.x]);
        S.bounds[threadIdx.x] = v;
      }
      __syncthreads();
    }
    // the ray bundle of the block: reference ray = the block's first active ray
    {
      const uint32_t am = __ballot_sync(0xffffffffu, active);
      if (lane == 0) S.amask[w] = am;
      __syncthreads();
      int fw = -1;
      for (int i = kPlWarps - 1; i >= 0; --i) if (S.amask[i] != 0u) fw = i;
      if (fw == w && lane == __ffs(am) - 1) {
        S.bundle[0] = ox; S.bundle[1] = oy; S.bundle[2] = oz;
        S.bundle[3] = dx; S.bundle[4] = dy; S.bundle[5] = dz;
      }
      if (fw < 0 && threadIdx.x == 0) {
        S.bundle[0] = S.bundle[1] = S.bundle[2] = 0.f;
        S.bundle[3] = S.bundle[4] = 0.f; S.bundle[5] = 1.f;
      }
      __syncthreads();
    }
    float c0[3] = {S.bundle[0], S.bundle[1], S.bundle[2]}, bm[3] = {S.bundle[3], S.bundle[4], S.bundle[5]};
    float bu[3], bv[3];
    {   // any orthonormal basis around bm
      float t[3] = {0.f, 0.f, 0.f};
      if (fabsf(bm[0]) <= fabsf(bm[1]) && fabsf(bm[0]) <= fabsf(bm[2])) t[0] = 1.f; else if (fabsf(bm[1]) <= fabsf(bm[2])) t[1] = 1.f; else t[2] = 1.f;
      bu[0] = t[1] * bm[2] - t[2] * bm[1]; bu[1] = t[2] * bm[0] - t[0] * bm[2]; bu[2] = t[0] * bm[1] - t[1] * bm[0];
      const float il = rsqrtf(bu[0] * bu[0] + bu[1] * bu[1] + bu[2] * bu[2]);
      bu[0] *= il; bu[1] *= il; bu[2] *= il;
      bv[0] = bm[1] * bu[2] - bm[2] * bu[1]; bv[1] = bm[2] * bu[0] - bm[0] * bu[2]; bv[2] = bm[0] * bu[1] - bm[1] * bu[0];
    }
    __syncthreads();
    {
      float r8[8] = {INFINITY, -INFINITY, INFINITY, -INFINITY, 0.f, INFINITY, -INFINITY, 1.f};
      if (active) {
        const float z = dx * bm[0] + dy * bm[1] + dz * bm[2];
        const float iz = 1.f / fmaxf(z, 1e-6f);
        const float x = (dx * bu[0] + dy * bu[1] + dz * bu[2]) * iz, y = (dx * bv[0] + dy * bv[1] + dz * bv[2]) * iz;
        const float ex = ox - c0[0], ey = oy - c0[1], ez = oz - c0[2];
        r8[0] = x; r8[1] = x; r8[2] = y; r8[3] = y;
        r8[4] = sqrtf(ex * ex + ey * ey + ez * ez);
        r8[5] = mint; r8[6] = maxt; r8[7] = z;
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) r8[k] = (k == 0 || k == 2 || k == 5 || k == 7) ? warp_min(r8[k]) : warp_max(r8[k]);
      if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) S.tred[w][k] = r8[k];
      }
      __syncthreads();
      if (threadIdx.x < 8) {
        const int k = threadIdx.x;
        float v = S.tred[0][k];
        for (int i = 1; i < kPlWarps; ++i)
          v = (k == 0 || k == 2 || k == 5 || k == 7) ? fminf(v, S.tred[i][k]) : fmaxf(v, S.tred[i][k]);
        S.bundle[k] = v;
      }
      __syncthreads();
    }
    // corner directions of the bundle's pyramid (rectangle in the plane at distance 1 along bm, slightly enlarged)
    float dk[4][3];
    float bdelta = S.bundle[4];
    const bool bundleOk = S.bundle[7] > 0.5f && S.bundle[0] <= S.bundle[1];
    {
      const float px = 1e-5f + 1e-3f * (S.bundle[1] - S.bundle[0]), py = 1e-5f + 1e-3f * (S.bundle[3] - S.bundle[2]);
      const float xs[2] = {S.bundle[0] - px, S.bundle[1] + px}, ys[2] = {S.bundle[2] - py, S.bundle[3] + py};
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int c = 0; c < 3; ++c) dk[k][c] = bm[c] + xs[k & 1] * bu[c] + ys[k >> 1] * bv[c];
      const float cm = fmaxf(fmaxf(fabsf(c0[0]), fabsf(c0[1])), fabsf(c0[2]));
      bdelta = bdelta * 1.001f + 4e-6f * cm;
    }
    float bl[3], bh[3];
    {
      const float ext = fmaxf(fmaxf(S.bounds[3] - S.bounds[0], S.bounds[4] - S.bounds[1]), S.bounds[5] - S.bounds[2]);
      const float mag = fmaxf(fmaxf(fabsf(S.bounds[0]), fabsf(S.bounds[3])),
                              fmaxf(fmaxf(fabsf(S.bounds[1]), fabsf(S.bounds[4])), fmaxf(fabsf(S.bounds[2]), fabsf(S.bounds[5]))));
      const float pad = 1e-4f * (ext + mag) + 1e-6f;
#pragma unroll
      for (int c = 0; c < 3; ++c) { bl[c] = S.bounds[c] - pad; bh[c] = S.bounds[3 + c] + pad; }
    }
    const bool blockActive = bl[0] <= bh[0];  // at least one active ray
    float a[GVPM_OUT_FLOATS];
#pragma unroll
    for (int j = 0; j < GVPM_OUT_FLOATS; ++j) a[j] = 0.f;
    uint32_t hits = 0, qn = 0;
    const uint64_t dumpBase = (kDump && haveRay) ? P.nbr_offsets[ray] : 0;

    auto drain = [&](uint32_t chunkBase) {
      // phase B: strictly rounded test + functor for the queued candidates of this chunk
      while (__any_sync(0xffffffffu, qn > 0)) {
        if (qn > 0) {
          const uint32_t p = S.queue[w][--qn][lane];
          const float4 q0 = S.tst[p][0], q1 = S.tst[p][1], q2 = S.tst[p][2];
          PlaneIts its;
          const v3 ro(ox, oy, oz), rd(dx, dy, dz);
          if (plane_intersect(v3(q0.x, q0.y, q0.z), v3(q1.x, q1.y, q1.z), v3(q2.x, q2.y, q2.z), sf(q0.w), sf(q1.w), ro, rd,
                              sf(mint), sf(maxt), its)) {
            const uint32_t gi = chunkBase + p;
            if (kDump) {
              P.nbr_idx[dumpBase + hits] = __ldg(P.plane_orig + gi) | 0x80000000u;
            } else {
              PlaneRec pl;
              pl.ori = v3(q0.x, q0.y, q0.z); pl.length0 = sf(q0.w);
              pl.e0 = v3(q1.x, q1.y, q1.z); pl.length1 = sf(q1.w);
              pl.e1 = v3(q2.x, q2.y, q2.z); pl.edgeID = (int)__float_as_uint(q2.w);
              const float4 q3 = ldg4(Q + 3 * (size_t)nPl + gi), q4 = ldg4(Q + 4 * (size_t)nPl + gi),
                           q5 = ldg4(Q + 5 * (size_t)nPl + gi);
              pl.flux = v3(q3.x, q3.y, q3.z);
              pl.w0 = v3(q4.x, q4.y, q4.z);
              pl.w1 = v3(q5.x, q5.y, q5.z);
              plane_functor(P, rec, rd, pl, its, a);
            }
            ++hits;
          }
        }
      }
    };

    if (blockActive) {
      for (uint32_t chunkBase = 0; chunkBase < nPl; chunkBase += kPlChunk) {
        const uint32_t leaf0 = chunkBase >> 5;
        // leaf boxes of the chunk against the ray-block bounds
        __syncthreads();  // previous chunk fully consumed (queues drained below)
        if (w == 0) {
          bool ov = false;
          const uint32_t lf = leaf0 + lane;
          if (lane < kPlLeaves && lf < nLeavesTotal) {
            const float4 lo = ldg4(P.tree.lo + lf), hi = ldg4(P.tree.hi + lf);
            ov = lo.x <= bh[0] && hi.x >= bl[0] && lo.y <= bh[1] && hi.y >= bl[1] && lo.z <= bh[2] && hi.z >= bl[2];
          }
          const uint32_t m = __ballot_sync(0xffffffffu, ov);
          if (lane == 0) S.leafMask = m;
        }
        __syncthreads();
        const uint32_t leafMask = S.leafMask;
        if (leafMask == 0) continue;
        // stage Q0-Q2 of the overlapping leaves
        for (int i = threadIdx.x; i < kPlChunk * 3; i += kPlWarps * 32) {
          const int k = i / kPlChunk, p = i - k * kPlChunk;
          const uint32_t gi = chunkBase + p;
          if ((leafMask >> (p >> 5) & 1u) && gi < nPl) S.tst[p][k] = ldg4(Q + (size_t)k * nPl + gi);
        }
        __syncthreads();
        // bundle test: planes no ray of the block can meet are dropped for the whole block (one thread per plane).
        // Warp w tests the w-th quarter of the chunk and lists its survivors in plane order; the four lists are then
        // concatenated, so the order of the live list (hence every ray's accumulation order) is the plane order.
        {
          const int nIn = (int)min((uint32_t)kPlChunk, nPl - chunkBase);
          constexpr int kPerWarp = kPlChunk / kPlWarps;
          uint32_t cntW = 0;
          for (int p0 = 0; p0 < kPerWarp; p0 += 32) {
            const int p = w * kPerWarp + p0 + lane;
            bool keep = p < nIn && (leafMask >> (p >> 5) & 1u);
            if (keep && bundleOk) keep = !plane_bundle_reject(S.tst[p][0], S.tst[p][1], S.tst[p][2], c0, dk, bdelta);
            const uint32_t m = __ballot_sync(0xffffffffu, keep);
            if (keep) S.liveW[w][cntW + __popc(m & ((1u << lane) - 1u))] = (uint16_t)p;
            cntW += __popc(m);
          }
          if (lane == 0) S.amask[w] = cntW;
          __syncthreads();
          uint32_t off = 0;
          for (int i = 0; i < w; ++i) off += S.amask[i];
          for (uint32_t j = lane; j < cntW; j += 32) S.live[off + j] = S.liveW[w][j];
          if (threadIdx.x == 0) S.nLive = S.amask[0] + S.amask[1] + S.amask[2] + S.amask[3];
        }
        __syncthreads();
        const int nLive = (int)S.nLive;
        // phase A in sub-steps, phase B whenever a queue could overflow in the next sub-step
        for (int sub = 0; sub < nLive; sub += kPlSub) {
          if (active) {
            const int pend = min(sub + kPlSub, nLive);
            for (int j = sub; j < pend; ++j) {
              const int p = S.live[j];
              if (plane_candidate(S.tst[p][0], S.tst[p][1], S.tst[p][2], ox, oy, oz, dx, dy, dz, mint, maxt))
                S.queue[w][qn++][lane] = (uint16_t)p;
            }
          }
          if (__any_sync(0xffffffffu, qn + kPlSub > kPlQCap)) drain(chunkBase);
        }
        drain(chunkBase);
      }
    }
    if (haveRay) {
      if (!kDump) {
        float *o = P.out + (size_t)ray * GVPM_OUT_FLOATS;
#pragma unroll
        for (int j = 0; j < GVPM_OUT_FLOATS; ++j) o[j] = a[j];
      }
      if (P.counts) { P.counts[2 * (size_t)ray] = hits; P.counts[2 * (size_t)ray + 1] = hits; }
    }
  }
}

// ---- host-side launchers -----------------------------------------------------------------------
void launch_plane_pack_sorted(const float4 *raw, const uint32_t *sorted, uint32_t n, float4 *planes, uint32_t *orig,
                              cudaStream_t st) {
  if (n) k_plane_pack_sorted<<<(n + 255) / 256, 256, 0, st>>>(raw, sorted, n, planes, orig);
}
void launch_plane_leaf_boxes(const float4 *planes, uint32_t n, uint32_t nLeaves, float4 *lo, float4 *hi, cudaStream_t st) {
  if (nLeaves) k_plane_leaf_boxes<<<(nLeaves + 7) / 8, 256, 0, st>>>(planes, n, nLeaves, lo, hi);
}

cudaError_t launch_plane_gather(const GatherParams &P, bool dump, int sm_count, cudaStream_t stream) {
  if (P.n_rays == 0) return cudaSuccess;
  const size_t smem = sizeof(PlaneShared);
  const unsigned need = (P.n_rays + kPlWarps * 32 - 1) / (kPlWarps * 32);   // persistent: CTAs pull ray blocks
  const unsigned grid = dump ? persistent_grid<k_plane_gather<true>>(sm_count, kPlWarps * 32, need, smem)
                             : persistent_grid<k_plane_gather<false>>(sm_count, kPlWarps * 32, need, smem);
  if (grid == 0) return cudaGetLastError();   // the shared-memory attribute was refused
  if (dump) k_plane_gather<true><<<grid, kPlWarps * 32, smem, stream>>>(P);
  else k_plane_gather<false><<<grid, kPlWarps * 32, smem, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace gvpm
