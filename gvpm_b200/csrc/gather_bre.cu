// gather_bre.cu — G-BRE gather in two kernels (DESIGN.md §4).
//
// k_bre_traverse: one warp per TILE of 32 consecutive camera rays, one ray per lane.  The warp walks the
//   implicit 32-ary AABB hierarchy over the Morton-sorted photons without a node stack (one ballot mask per
//   level is the whole traversal state): lane c tests child c of the current node against the tile's central
//   ray fattened by the tile's spread (two coalesced 128-bit loads per lane), so the cost of the walk is
//   shared by 32 rays.  At a leaf, lane c holds photon c (one 128-bit load) and tests it ONCE against the fat
//   ray; the few photons inside are then broadcast one by one and every lane tests its own ray with a relaxed
//   FMA predicate, pushing candidates into its own shared-memory queue.  When a queue fills (and at the end of
//   the tile) every lane runs the reference's predicate in strictly rounded arithmetic (gvpm_accel.h:293-301,
//   shift_volume_photon.cpp:707-724) and the depth/mode/pathSet filters on its queued candidates with all
//   lanes busy, and the survivors go to the global (ray, photon) pair list as one contiguous run per ray.
//   Tiles whose rays are not coherent fall back to quads of 4 lanes, then to single rays; results never
//   depend on the grouping.
// k_bre_shade: one THREAD per (ray, photon) pair, so the divergent shift code (null shift, diffuse
//   reconnection, MIS; bre_device.cuh) always runs with full warps whatever the number of
//   neighbours per ray.  27 accumulators per thread in registers, a segmented warp scan by ray id
//   (shuffles) folds the lanes of one ray, and the last lane of each run adds 27 floats to the ray's
//   output row.
#include "bre_device.cuh"
#include "launch_sizing.cuh"
#include "warp_ops.cuh"

namespace gvpm {

#ifndef GVPM_TRAV_WARPS
#define GVPM_TRAV_WARPS 4
#endif
#ifndef GVPM_TRAV_MIN_BLOCKS
#define GVPM_TRAV_MIN_BLOCKS 6
#endif
#ifndef GVPM_SHADE_THREADS
#define GVPM_SHADE_THREADS 128
#endif
#ifndef GVPM_SHADE_MIN_BLOCKS
// 96 registers, no spills.  Tuned on cfg5 (B200, 1000 W): 4: 2.90 ms, 5: 2.63, 6: 2.69, 8: 2.82.  A phase A/B hand-off
// that re-reads the photon record in phase B instead of carrying it through shared memory fits 80 / 72 registers at 6 / 7
// (with spills) but shades slower at every bound, 5 / 6 / 7: 2.75 / 2.75 / 2.78 ms against 2.44 (profiles/r3_shade_records.md)
#define GVPM_SHADE_MIN_BLOCKS 5
#endif
#ifndef GVPM_TILE_QUEUE
#define GVPM_TILE_QUEUE 32
#endif
constexpr int kTravWarps = GVPM_TRAV_WARPS;
constexpr int kTileQ = GVPM_TILE_QUEUE;  // candidate queue entries per lane
#ifndef GVPM_LEAF_BATCH
#define GVPM_LEAF_BATCH 4   // tuned on cfg5 (tools/build_variants.sh + tools/time_gather.py): 1: 3.22 ms, 2: 2.45, 4: 2.32
#endif
constexpr int kLeafBatch = GVPM_LEAF_BATCH;  // leaves whose photon loads are in flight together
#ifndef GVPM_TILE_BATCH
#define GVPM_TILE_BATCH 16
#endif
constexpr int kTileBatch = GVPM_TILE_BATCH;  // photons tested between queue-room checks
static_assert(kTileBatch <= kTileQ, "a batch must fit in an empty queue");

struct TileShared {
  float4 ph[2 * 32 * kLeafBatch];  // photons of the current leaf batch inside the fat ray: entry i of list b at [2i + b]
  uint32_t queue[kTileQ][32];  // [entry][lane]: sorted photon slots waiting for the strict test
  uint32_t mask[GVPM_MAX_LEVELS];
  uint32_t base[GVPM_MAX_LEVELS];
};

__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}

// per-lane view of the lane's own camera ray during the traversal
struct LaneRay {
  float ox, oy, oz, dx, dy, dz, mint, elen, xi;
  int px, py, eid;
};

// strict predicate + filters on the queued candidates of every lane (all lanes busy), survivors -> pair list / dump.
// Warp-collective: every lane of the warp must call it.
template <int MODE>
__device__ __forceinline__ void flush_candidates(const GatherParams &P, uint32_t (*queue)[32], int lane, const LaneRay &L,
                                                 bool have, uint32_t ray, uint32_t &qn, uint32_t &nGeom, uint32_t &nContrib) {
  constexpr bool DUMP = (MODE & 1) != 0, SPPM = (MODE & 2) != 0;
  const uint32_t maxq = __reduce_max_sync(0xffffffffu, qn);
  BaseRay R;
  R.o = v3(L.ox, L.oy, L.oz); R.d = v3(L.dx, L.dy, L.dz);
  R.mint = sf(L.mint); R.edgeLen = sf(L.elen); R.xi = sf(L.xi);
  R.px = L.px; R.py = L.py; R.edgeId = L.eid;
  R.maxt = sf(0.f);
  if (SPPM && have) R.maxt = sf(__ldg(&P.rays[(size_t)ray * GVPM_RAY_FLOAT4 + 1].w));
  uint32_t keep = 0;
  for (uint32_t k = 0; k < maxq; ++k) {
    if (k < qn) {
      const uint32_t slot = queue[k][lane];
      const float4 q0 = ldg4(P.planes + slot);
      sf tB, pc;
      const bool geom = base_distance<SPPM>(P, R, v3(q0.x, q0.y, q0.z), SPPM ? __ldg(P.orig + slot) : 0u, tB, pc);
      const bool contrib = geom && filters_pass<SPPM>(P, R, __float_as_uint(q0.w));
      if (DUMP && geom)
        P.nbr_idx[P.nbr_offsets[ray] + nGeom] = __ldg(P.orig + slot) | (contrib ? 0x80000000u : 0u);
      nGeom += geom ? 1u : 0u;
      nContrib += contrib ? 1u : 0u;
      if (!DUMP && contrib) queue[keep++][lane] = slot;
    }
  }
  qn = 0;
  if (!DUMP) {
    const uint32_t incl = warp_inclusive_scan(keep, lane);
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    if (total) {
      unsigned long long base = 0;
      if (lane == 0) base = atomicAdd(P.pair_counter, (unsigned long long)total);
      base = __shfl_sync(0xffffffffu, base, 0) + (incl - keep);
      for (uint32_t k = 0; k < keep; ++k)
        if (base + k < P.pair_cap) P.pairs[base + k] = make_uint2(ray, __ldg(P.orig + queue[k][lane]));
    }
  }
  __syncwarp();
}

// MODE bit 0: dump the neighbour sets instead of emitting pairs; bit 1: sppm's primal predicate (bre_device.cuh)
template <int MODE>
__global__ void __launch_bounds__(kTravWarps * 32, GVPM_TRAV_MIN_BLOCKS)
k_bre_traverse(const __grid_constant__ GatherParams P) {
  constexpr bool DUMP = (MODE & 1) != 0, SPPM = (MODE & 2) != 0;
  __shared__ TileShared sh[kTravWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  TileShared &S = sh[w];
  const Tree &T = P.tree;
  const int top = T.levels - 1;
  const uint32_t nTiles = (P.ray_end - P.ray_begin + 31) / 32;
  const float coordMag = T.n ? __ldg(P.bounds + 6) : 0.f;
  // groups whose rays drift apart by more than this are split (performance only)
  float spreadMax = 16.f * P.radius;
  if (T.n) {
    const float ex = __ldg(P.bounds + 3) - __ldg(P.bounds), ey = __ldg(P.bounds + 4) - __ldg(P.bounds + 1),
                ez = __ldg(P.bounds + 5) - __ldg(P.bounds + 2);
    spreadMax = fmaxf(spreadMax, 0.01f * sqrtf(ex * ex + ey * ey + ez * ez));
  }
  // the filters only drop photons: apply them before queueing unless the caller wants the geometric counts
  const bool prefilter = !DUMP && !SPPM && P.counts == nullptr;   // (sppm's own filter is applied at the flush only)
  const bool split = prefilter && P.cfg.path_set;                 // per-parity photon lists (see the leaf code)

  for (;;) {
    uint32_t tile = 0;
    if (lane == 0) tile = atomicAdd(P.work_counter, 1u);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    if (tile >= nTiles) break;
    const uint32_t ray = P.ray_begin + tile * 32 + lane;
    const bool have = ray < P.ray_end;
    LaneRay L;
    {
      const float4 *rec = P.rays + (size_t)(have ? ray : P.ray_begin) * GVPM_RAY_FLOAT4;
      const float4 b0 = ldg4(rec), b1 = ldg4(rec + 1), b2 = ldg4(rec + 2), b3 = ldg4(rec + 3);
      L.ox = b0.x; L.oy = b0.y; L.oz = b0.z; L.mint = b0.w;
      L.dx = b1.x; L.dy = b1.y; L.dz = b1.z; L.elen = b2.w;
      // sppm's primal query reads maxt, not edge_len (bre.cpp:206,240): a caller that leaves edge_len unset still gets
      // the whole segment walked
      if (SPPM) L.elen = fmaxf(L.elen, b1.w);
      L.xi = b3.x;
      L.px = (int)__float_as_uint(b3.y); L.py = (int)__float_as_uint(b3.z); L.eid = (int)__float_as_uint(b3.w);
    }
    const bool active = have && T.n > 0 && L.elen >= L.mint;
    const uint32_t actMask = __ballot_sync(0xffffffffu, active);
    const int parity = (L.px + L.py) % 2;
    uint32_t nGeom = 0, nContrib = 0, qn = 0;

    auto flush = [&]() { flush_candidates<MODE>(P, S.queue, lane, L, have, ray, qn, nGeom, nContrib); };

    // one stackless walk for the lanes of `gm`, sharing the fat ray (co, cd) of half-width `spread`
    auto traverse_group = [&](uint32_t gm, float cox, float coy, float coz, float cdx, float cdy, float cdz,
                              float sx, float sy, float sz, float tloG, float thiG, float omag) {
      // (sx, sy, sz): per-axis bound of |ray_j(t) - axis(t)| over the group and t in [0, tEnd]: the fat ray is the
      // axis swept by that box (much tighter than a sphere for the usual wide-and-flat pixel tile).
      // Conservative culling: relaxed arithmetic made safe by `fpad` (a few ulp of the coordinate magnitudes:
      // rounding of the slab test and of the strict predicate) plus the group spread.
      const float spread = sqrtf(sx * sx + sy * sy + sz * sz);
      const float fpad = (omag + coordMag + fabsf(thiG) + P.radius + spread) * 3.8147e-6f;  // 2^-18
      const float oxp = cox + (sx + fpad), oxm = cox - (sx + fpad), oyp = coy + (sy + fpad), oym = coy - (sy + fpad),
                  ozp = coz + (sz + fpad), ozm = coz - (sz + fpad);
      const float ix = 1.f / cdx, iy = 1.f / cdy, iz = 1.f / cdz;
      const float tloBox = tloG - 4.f * fpad - spread;                 // axial range of the fat ray
      const float thiBox = thiG + P.radius + 4.f * fpad + spread;
      const float tloRay = tloG - 4.f * fpad;                          // per-ray disk distance bound
      const float rpad2 = (P.radius + fpad) * (P.radius + fpad);
      // a photon within r of ray j at parameter t_j: q = p - axis(dd) (dd = its own axial coordinate) differs from
      // p - axis(t_j) by (dd - t_j) * cd with |dd - t_j| <= spread + r, so per axis
      //   |q_a| <= s_a + r + (spread + r) * |cd_a|
      const float slop = spread + P.radius + 2.f * fpad;
      const float fx = sx + P.radius + 2.f * fpad + slop * fabsf(cdx), fy = sy + P.radius + 2.f * fpad + slop * fabsf(cdy),
                  fz = sz + P.radius + 2.f * fpad + slop * fabsf(cdz);
      const float tloFat = tloBox - P.radius, thiFat = thiBox;
      const bool mine = gm >> lane & 1u;

      uint32_t cur, base = 0;
      int l = top;
      cur = __ballot_sync(0xffffffffu, (uint32_t)lane < T.cnt[top] &&
                                           box_hit(T, T.off[top] + lane, oxp, oxm, oyp, oym, ozp, ozm, ix, iy,
                                                   iz, tloBox, thiBox));
      for (;;) {
        if (cur == 0) {
          if (l == top) break;
          ++l;
          cur = S.mask[l];
          base = S.base[l];
          continue;
        }
        if (l > 0) {
          const int c = __ffs(cur) - 1;
          cur &= cur - 1;
          const uint32_t node = base + c;
          S.mask[l] = cur;
          S.base[l] = base;
          --l;
          base = node << 5;
          const uint32_t idx = base + lane;
          cur = __ballot_sync(0xffffffffu, idx < T.cnt[l] && box_hit(T, T.off[l] + idx, oxp, oxm, oyp, oym, ozp,
                                                                       ozm, ix, iy, iz, tloBox, thiBox));
          continue;
        }
        // ---- leaves: `cur` lists the hit leaves of one parent.  Their photon loads are independent, so they are
        // issued kLeafBatch at a time (the walk is otherwise one long chain of dependent L2-latency loads).
        // Lane holds photon (leaf*32 + lane), tested once against the fat ray.
        int leafC[kLeafBatch];
        float4 leafQ[kLeafBatch];
#pragma unroll
        for (int b = 0; b < kLeafBatch; ++b) {
          leafC[b] = -1;
          leafQ[b] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (cur) {
            const int c = __ffs(cur) - 1;
            cur &= cur - 1;
            const uint32_t pi = ((base + (uint32_t)c) << 5) + lane;
            if (pi < T.n) {
              leafC[b] = c;
              leafQ[b] = ldg4(P.planes + pi);
            }
          }
        }
        // the photons inside the fat ray are compacted into shared memory (all leaves of the batch together) and
        // broadcast from there; w = lane | leaf-in-parent << 5 | meta << 10
        __syncwarp();
        // With the pathSet checkerboard a photon only ever matches rays of its own pixel parity: the in-fat photons go
        // to two lists (interleaved, so that lanes of either parity read different banks) and every lane walks only
        // the list of its parity - half the per-ray tests.  Without the prefilter everything goes to list 0.
        uint32_t total0 = 0, total1 = 0;
#pragma unroll
        for (int b = 0; b < kLeafBatch; ++b) {
          const float4 q0 = leafQ[b];
          const float cx = q0.x - cox, cy = q0.y - coy, cz = q0.z - coz;
          const float dd = cx * cdx + cy * cdy + cz * cdz;
          const float qx = cx - dd * cdx, qy = cy - dd * cdy, qz = cz - dd * cdz;
          const bool inFat = leafC[b] >= 0 && fabsf(qx) < fx && fabsf(qy) < fy && fabsf(qz) < fz && dd > tloFat &&
                             dd < thiFat;
          const uint32_t pb = split ? ((__float_as_uint(q0.w) >> 10) & 1u) : 0u;   // meta bit 10 = pathID parity
          const uint32_t pm0 = __ballot_sync(0xffffffffu, inFat && pb == 0u);
          const uint32_t pm1 = __ballot_sync(0xffffffffu, inFat && pb != 0u);
          if (inFat) {
            const uint32_t lt = (1u << lane) - 1u;
            const uint32_t pos = pb ? total1 + __popc(pm1 & lt) : total0 + __popc(pm0 & lt);
            S.ph[2u * pos + pb] = make_float4(
                q0.x, q0.y, q0.z,
                __uint_as_float((uint32_t)lane | ((uint32_t)leafC[b] << 5) | (__float_as_uint(q0.w) << 10)));
          }
          total0 += __popc(pm0);
          total1 += __popc(pm1);
        }
        __syncwarp();
        const uint32_t slot0 = base << 5;
        const uint32_t total = max(total0, total1);
        const uint32_t myList = split ? (uint32_t)parity : 0u;
        const uint32_t myTotal = myList ? total1 : total0;
        for (uint32_t i0 = 0; i0 < total; i0 += kTileBatch) {
          const uint32_t i1 = min(total, i0 + (uint32_t)kTileBatch);
          // a lane pushes at most one entry per photon: make room for the whole batch up front
          if (__any_sync(0xffffffffu, qn + (i1 - i0) > (uint32_t)kTileQ)) flush();
          if (mine) {
            const uint32_t e1 = min(i1, myTotal);
#pragma unroll 2
            for (uint32_t i = i0; i < e1; ++i) {
              const float4 ph = S.ph[2u * i + myList];
              // relaxed (FMA) pre-test of the lane's own ray, conservative by fpad
              const float cx = ph.x - L.ox, cy = ph.y - L.oy, cz = ph.z - L.oz;
              const float dd = cx * L.dx + cy * L.dy + cz * L.dz;
              const float qx = cx - dd * L.dx, qy = cy - dd * L.dy, qz = cz - dd * L.dz;
              bool cand = (qx * qx + qy * qy + qz * qz) < rpad2 && dd > tloRay;
              const uint32_t w = __float_as_uint(ph.w);
              if (prefilter) {
                // meta << 10: bit 20 = pathID parity (already matched through the list when split), bits 12-19 = depth
                if (!split && P.cfg.path_set && (int)((w >> 20) & 1u) != parity) cand = false;
                if (P.cfg.max_depth > 0 && (int)((w >> 12) & 255u) + L.eid > P.cfg.max_depth) cand = false;
              }
              if (cand) S.queue[qn++][lane] = slot0 + (w & 1023u);
            }
          }
        }
      }
    };

    if (actMask) {
      // tile centre: mean origin / mean direction of the active rays
      const float cnt = (float)__popc(actMask), inv = 1.f / cnt;
      const float mox = warp_sum(active ? L.ox : 0.f) * inv, moy = warp_sum(active ? L.oy : 0.f) * inv,
                  moz = warp_sum(active ? L.oz : 0.f) * inv;
      float mdx = warp_sum(active ? L.dx : 0.f), mdy = warp_sum(active ? L.dy : 0.f), mdz = warp_sum(active ? L.dz : 0.f);
      const float mlen = sqrtf(mdx * mdx + mdy * mdy + mdz * mdz);
      const float tEnd = warp_max(active ? L.elen : 0.f) + P.radius;
      float dvx = 0.f, dvy = 0.f, dvz = 0.f;
      bool okDir = mlen > 0.5f * cnt;  // nearly parallel rays only
      if (okDir) {
        const float il = 1.f / mlen;
        mdx *= il; mdy *= il; mdz *= il;
        if (active) {
          // per-axis distance between corresponding points of the lane's ray and the central ray over [0, tEnd]
          // (linear in t, so attained at an end)
          const float ax = L.ox - mox, ay = L.oy - moy, az = L.oz - moz;
          const float bx = ax + tEnd * (L.dx - mdx), by = ay + tEnd * (L.dy - mdy), bz = az + tEnd * (L.dz - mdz);
          dvx = fmaxf(fabsf(ax), fabsf(bx)); dvy = fmaxf(fabsf(ay), fabsf(by)); dvz = fmaxf(fabsf(az), fabsf(bz));
        }
      }
      const float s32x = warp_max(dvx) * 1.0001f, s32y = warp_max(dvy) * 1.0001f, s32z = warp_max(dvz) * 1.0001f;
      const float spread32 = sqrtf(s32x * s32x + s32y * s32y + s32z * s32z);
      const float amag = active ? fmaxf(fmaxf(fabsf(L.ox), fabsf(L.oy)), fabsf(L.oz)) : 0.f;
      if (okDir && spread32 <= spreadMax) {
        const float tloG = warp_min(active ? L.mint : 3.4e38f), thiG = warp_max(active ? L.elen : -3.4e38f);
        traverse_group(actMask, mox, moy, moz, mdx, mdy, mdz, s32x, s32y, s32z, tloG, thiG, warp_max(amag));
      } else {
        // quads of 4 consecutive lanes, then single rays
        const float qc = quad_sum(active ? 1.f : 0.f), qi = qc > 0.f ? 1.f / qc : 0.f;
        const float qox = quad_sum(active ? L.ox : 0.f) * qi, qoy = quad_sum(active ? L.oy : 0.f) * qi,
                    qoz = quad_sum(active ? L.oz : 0.f) * qi;
        float qdx = quad_sum(active ? L.dx : 0.f), qdy = quad_sum(active ? L.dy : 0.f), qdz = quad_sum(active ? L.dz : 0.f);
        const float qlen = sqrtf(qdx * qdx + qdy * qdy + qdz * qdz);
        const bool qok = qlen > 0.5f * qc && qc > 0.f;
        float qvx = 0.f, qvy = 0.f, qvz = 0.f;
        if (qok) {
          const float il = 1.f / qlen;
          qdx *= il; qdy *= il; qdz *= il;
          if (active) {
            const float ax = L.ox - qox, ay = L.oy - qoy, az = L.oz - qoz;
            const float bx = ax + tEnd * (L.dx - qdx), by = ay + tEnd * (L.dy - qdy), bz = az + tEnd * (L.dz - qdz);
            qvx = fmaxf(fabsf(ax), fabsf(bx)); qvy = fmaxf(fabsf(ay), fabsf(by)); qvz = fmaxf(fabsf(az), fabsf(bz));
          }
        }
        const float qsx = quad_max(qvx) * 1.0001f, qsy = quad_max(qvy) * 1.0001f, qsz = quad_max(qvz) * 1.0001f;
        const float qspread = sqrtf(qsx * qsx + qsy * qsy + qsz * qsz);
        const float qtlo = -quad_max(active ? -L.mint : -3.4e38f), qthi = quad_max(active ? L.elen : -3.4e38f);
        const float qmag = quad_max(amag);
        for (int q = 0; q < 8; ++q) {
          const uint32_t gm = actMask & (0xFu << (4 * q));
          if (!gm) continue;
          const int ld = __ffs(gm) - 1;
          const bool useQuad = __shfl_sync(0xffffffffu, qok && qspread <= spreadMax, ld);
          if (useQuad) {
            traverse_group(gm, __shfl_sync(0xffffffffu, qox, ld), __shfl_sync(0xffffffffu, qoy, ld),
                           __shfl_sync(0xffffffffu, qoz, ld), __shfl_sync(0xffffffffu, qdx, ld),
                           __shfl_sync(0xffffffffu, qdy, ld), __shfl_sync(0xffffffffu, qdz, ld),
                           __shfl_sync(0xffffffffu, qsx, ld), __shfl_sync(0xffffffffu, qsy, ld),
                           __shfl_sync(0xffffffffu, qsz, ld), __shfl_sync(0xffffffffu, qtlo, ld),
                           __shfl_sync(0xffffffffu, qthi, ld), __shfl_sync(0xffffffffu, qmag, ld));
          } else {
            for (uint32_t m = gm; m; m &= m - 1) {
              const int j = __ffs(m) - 1;
              traverse_group(1u << j, __shfl_sync(0xffffffffu, L.ox, j), __shfl_sync(0xffffffffu, L.oy, j),
                             __shfl_sync(0xffffffffu, L.oz, j), __shfl_sync(0xffffffffu, L.dx, j),
                             __shfl_sync(0xffffffffu, L.dy, j), __shfl_sync(0xffffffffu, L.dz, j), 0.f, 0.f, 0.f,
                             __shfl_sync(0xffffffffu, L.mint, j), __shfl_sync(0xffffffffu, L.elen, j),
                             __shfl_sync(0xffffffffu, amag, j));
            }
          }
        }
      }
      if (__any_sync(0xffffffffu, qn > 0)) flush();
    }
    if (P.counts && have) {
      P.counts[2 * (size_t)ray] = nGeom;
      P.counts[2 * (size_t)ray + 1] = nContrib;
    }
  }
}


// ---- frustum-grid traversal (gvpm_device.cuh FrustumGrid; built by gvpm_build_points_for_rays when every uploaded ray's
// line passes through one point) ---------------------------------------------------------------------------------------
// One ray per lane, one tile of 32 consecutive rays per warp.  No hierarchy walk: the ray's projected direction gives its
// cell in every footprint class, the 3x3 cells around it hold every photon that can be a neighbour (three contiguous
// slot ranges per class, one per cell row), and each candidate costs one 128-bit load (neighbouring pixels read the
// same cells: L1) plus the relaxed pre-test.  Candidate queues, the strict predicate and the pair emission are the ones
// of k_bre_traverse (flush_candidates), so the neighbour sets are bit-identical.
#ifndef GVPM_GRID_MIN_BLOCKS
#define GVPM_GRID_MIN_BLOCKS 6
#endif
struct GridShared {
  uint32_t queue[kTileQ][32];
};
template <int MODE>
__global__ void __launch_bounds__(kTravWarps * 32, GVPM_GRID_MIN_BLOCKS)
k_bre_grid_traverse(const __grid_constant__ GatherParams P) {
  constexpr bool DUMP = (MODE & 1) != 0, SPPM = (MODE & 2) != 0;
  __shared__ GridShared sh[kTravWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  GridShared &S = sh[w];
  const FrustumGrid &G = P.grid;
  const uint32_t nTiles = (P.ray_end - P.ray_begin + 31) / 32;
  const float coordMag = __ldg(P.bounds + 6);
  const bool prefilter = !DUMP && !SPPM && P.counts == nullptr;
  const uint32_t nGridsBuilt = G.parity_split ? 2u : 1u;
  const uint32_t nearBeg = __ldg(P.cell_start + nGridsBuilt * G.n_cells), nearEnd = __ldg(P.cell_start + nGridsBuilt * G.n_cells + 1);
  // with the pathSet prefilter a ray only ever pairs with photons of its pixel's parity: it scans that grid alone
  const bool onlyMine = G.parity_split && prefilter && P.cfg.path_set;
  const uint32_t nPass = onlyMine ? 1u : nGridsBuilt;
  if (P.build_ovf && __ldg(P.build_ovf)) {   // incomplete grid (capi_points.cu build_frustum): report it instead of gathering
    if (blockIdx.x == 0 && threadIdx.x == 0) *P.pair_counter = 1ull << 62;
    return;
  }

  for (;;) {
    uint32_t tile = 0;
    if (lane == 0) tile = atomicAdd(P.work_counter, 1u);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    if (tile >= nTiles) break;
    const uint32_t ray = P.ray_begin + tile * 32 + lane;
    const bool have = ray < P.ray_end;
    LaneRay L;
    {
      const float4 *rec = P.rays + (size_t)(have ? ray : P.ray_begin) * GVPM_RAY_FLOAT4;
      const float4 b0 = ldg4(rec), b1 = ldg4(rec + 1), b2 = ldg4(rec + 2), b3 = ldg4(rec + 3);
      L.ox = b0.x; L.oy = b0.y; L.oz = b0.z; L.mint = b0.w;
      L.dx = b1.x; L.dy = b1.y; L.dz = b1.z; L.elen = b2.w;
      if (SPPM) L.elen = fmaxf(L.elen, b1.w);
      L.xi = b3.x;
      L.px = (int)__float_as_uint(b3.y); L.py = (int)__float_as_uint(b3.z); L.eid = (int)__float_as_uint(b3.w);
    }
    const bool active = have && P.tree.n > 0 && L.elen >= L.mint;
    const int parity = (L.px + L.py) % 2;
    uint32_t nGeom = 0, nContrib = 0, qn = 0;
    auto flush = [&]() { flush_candidates<MODE>(P, S.queue, lane, L, have, ray, qn, nGeom, nContrib); };
    if (__any_sync(0xffffffffu, active)) {
      // relaxed pre-test constants of the lane's own ray (conservative by fpad, as in k_bre_traverse)
      const float omag = fmaxf(fmaxf(fabsf(L.ox), fabsf(L.oy)), fabsf(L.oz));
      const float fpad = (omag + coordMag + fabsf(L.elen) + P.radius) * 3.8147e-6f;  // 2^-18
      const float rpad2 = (P.radius + fpad) * (P.radius + fpad);
      const float tloRay = L.mint - 4.f * fpad;
      auto test = [&](const float4 ph, uint32_t slot) {
        const float cx = ph.x - L.ox, cy = ph.y - L.oy, cz = ph.z - L.oz;
        const float dd = cx * L.dx + cy * L.dy + cz * L.dz;
        const float qx = cx - dd * L.dx, qy = cy - dd * L.dy, qz = cz - dd * L.dz;
        bool cand = (qx * qx + qy * qy + qz * qz) < rpad2 && dd > tloRay;
        if (prefilter) {
          const uint32_t meta = __float_as_uint(ph.w);
          if (P.cfg.path_set && (int)((meta >> 10) & 1u) != parity) cand = false;
          if (P.cfg.max_depth > 0 && (int)((meta >> 2) & 255u) + L.eid > P.cfg.max_depth) cand = false;
        }
        if (cand) S.queue[qn++][lane] = slot;
      };
      float x = 0.f, y = 0.f, z = 1.f;
      if (active) {
        z = L.dx * G.m[0] + L.dy * G.m[1] + L.dz * G.m[2];
        const float iz = 1.f / z;
        x = (L.dx * G.u[0] + L.dy * G.u[1] + L.dz * G.u[2]) * iz;
        y = (L.dx * G.v[0] + L.dy * G.v[1] + L.dz * G.v[2]) * iz;
      }
      // One loop over the footprint classes, then the NEAR bucket (photons too close to C for any class: every ray
      // tests them), then one empty round that flushes what is left: a single copy of the candidate loop and of
      // flush_candidates (this kernel's instruction-fetch stalls grow with its code size).
      for (int c = 0; c <= G.classes + 1; ++c) {
        const bool isNear = c == G.classes, isLast = c == G.classes + 1;
        const int cc = min(c, G.classes - 1);
        const uint32_t nx = G.nx[cc], ny = G.ny[cc], base = G.base[cc];
        if (!isNear && !isLast) {
          // empty class (in every grid): nothing to do (warp-uniform)
          bool empty = true;
          for (uint32_t g = 0; g < nGridsBuilt; ++g)
            empty = empty && __ldg(P.cell_start + g * G.n_cells + base) == __ldg(P.cell_start + g * G.n_cells + base + nx * ny);
          if (empty) continue;
        }
        int x0 = 0, x1 = 0, y0 = 0, y1 = -1;
        if (active && !isNear && !isLast) {
          const float ic = 1.f / G.csize[cc];
          int cx = (int)floorf((x - G.gx0) * ic), cy = (int)floorf((y - G.gy0) * ic);
          cx = min(max(cx, 0), (int)nx - 1);
          cy = min(max(cy, 0), (int)ny - 1);
          x0 = max(cx - 1, 0); x1 = min(cx + 1, (int)nx - 1);
          y0 = max(cy - 1, 0); y1 = min(cy + 1, (int)ny - 1);
        }
        const uint32_t nPassC = (isNear || isLast) ? 1u : nPass;
        for (uint32_t pass = 0; pass < nPassC; ++pass) {
          const uint32_t gbase = (onlyMine ? (uint32_t)parity : pass) * G.n_cells + base;
          uint32_t s0 = 0u, s1 = 0u, s2 = 0u, n0 = 0u, n1 = 0u, n2 = 0u;
          auto row = [&](int yy, uint32_t &sr, uint32_t &nr) {
            const uint32_t rowBase = gbase + (uint32_t)yy * nx;
            sr = __ldg(P.cell_start + rowBase + x0);
            nr = __ldg(P.cell_start + rowBase + x1 + 1) - sr;
          };
          if (y0 <= y1) row(y0, s0, n0);
          if (y0 + 1 <= y1) row(y0 + 1, s1, n1);
          if (y0 + 2 <= y1) row(y0 + 2, s2, n2);
          if (isNear && active) { s0 = nearBeg; n0 = nearEnd - nearBeg; }
          const uint32_t n01 = n0 + n1, tot = n01 + n2;
          const uint32_t wmax = isLast ? 1u : __reduce_max_sync(0xffffffffu, tot);
          // four candidates per step: their loads are issued together (each lane reads its own cells; neighbouring
          // pixels share them, so most of these hit L1)
          for (uint32_t j0 = 0; j0 < wmax; j0 += kTileBatch) {
            if (__any_sync(0xffffffffu, qn + (uint32_t)kTileBatch > (uint32_t)kTileQ || (isLast && qn > 0u))) flush();
#pragma unroll
            for (uint32_t u0 = 0; u0 < (uint32_t)kTileBatch; u0 += 4) {
              float4 ph[4];
              uint32_t sl[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const uint32_t j = j0 + u0 + u;
                sl[u] = j < n0 ? s0 + j : (j < n01 ? s1 + (j - n0) : s2 + (j - n01));
                if (j < tot) ph[u] = ldg4(P.planes + sl[u]);
              }
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if (j0 + u0 + u < tot) test(ph[u], sl[u]);
            }
          }
        }
      }
    }
    if (P.counts && have) {
      P.counts[2 * (size_t)ray] = nGeom;
      P.counts[2 * (size_t)ray + 1] = nContrib;
    }
  }
}

template <bool SPPM>
__global__ void __launch_bounds__(GVPM_SHADE_THREADS, GVPM_SHADE_MIN_BLOCKS)
k_bre_shade(const __grid_constant__ GatherParams P) {
  __shared__ ShadeShared shade_sh[SPPM ? 1 : GVPM_SHADE_THREADS / 32];
  const int lane = threadIdx.x & 31;
  unsigned long long total = *P.pair_counter;
  if (total >= (1ull << 62)) return;   // incomplete perspective grid: nothing to shade (the host reports it)
  if (total > P.pair_cap) total = P.pair_cap;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  // software pipeline over the grid-stride loop: the pair of the NEXT iteration is already in registers, so its
  // 128-byte photon record (a random HBM line) is prefetched while the current pair is shaded, and the pair of the
  // iteration after that is requested
  const unsigned long long first = (unsigned long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31);
  const uint2 none = make_uint2(0xffffffffu, 0u);
  uint2 cur = none, nxt = none;
  if (first + lane < total) cur = P.pairs[first + lane];
  if (first + stride + lane < total) nxt = P.pairs[first + stride + lane];
  for (unsigned long long i0 = first; i0 < total; i0 += stride) {
    const unsigned long long i = i0 + lane;
    const bool valid = i < total;
    const uint2 pr = cur;
    if (nxt.x != 0xffffffffu) {
      asm volatile("prefetch.global.L1 [%0];" ::"l"(P.aos + (size_t)nxt.y * 8));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(P.rays + (size_t)nxt.x * GVPM_RAY_FLOAT4));
    }
    cur = nxt;
    nxt = (i + 2 * stride < total) ? P.pairs[i + 2 * stride] : none;
    float a[GVPM_OUT_FLOATS];
#pragma unroll
    for (int j = 0; j < GVPM_OUT_FLOATS; ++j) a[j] = 0.f;
    if (SPPM) {
      if (valid) bre_photon<SPPM>(P, P.rays + (size_t)pr.x * GVPM_RAY_FLOAT4, pr.y, a);
    } else {
      bre_pairs_warp(P, pr, valid, a, shade_sh[threadIdx.x >> 5], lane);
    }
    // per-ray sums over RUNS of equal ray id (a ray's pairs arrive in contiguous runs, one per flush; the same ray
    // may own several runs, each adds its own partial sum)
    warp_run_sum(pr.x, a, valid, P.out, lane);
  }
}

// ---- host-side launchers (called from the capi_*.cu units) -------------------------------------------
// persistent grids: warps pull tiles of 32 rays from a counter
template <int MODE> static void launch_traverse_mode(const GatherParams &P, int sm_count, cudaStream_t stream) {
  const unsigned tiles = (P.ray_end - P.ray_begin + 31) / 32;
  const unsigned need = (tiles + kTravWarps - 1) / kTravWarps;
  if (P.cell_start != nullptr) {   // frustum grid built for this ray set
    const unsigned grid = persistent_grid<k_bre_grid_traverse<MODE>>(sm_count, kTravWarps * 32, need);
    k_bre_grid_traverse<MODE><<<grid, kTravWarps * 32, 0, stream>>>(P);
  } else {
    const unsigned grid = persistent_grid<k_bre_traverse<MODE>>(sm_count, kTravWarps * 32, need);
    k_bre_traverse<MODE><<<grid, kTravWarps * 32, 0, stream>>>(P);
  }
}
template <bool SPPM> static void launch_shade_mode(const GatherParams &P, unsigned long long total, int sm_count,
                                                   cudaStream_t stream) {
  // total == ~0: the count is only known on the device (the kernel reads it): size the grid for a full pair list
  if (total == ~0ull || total > P.pair_cap) total = P.pair_cap;
  const unsigned grid = stride_grid<k_bre_shade<SPPM>>(sm_count, GVPM_SHADE_THREADS, total);
  k_bre_shade<SPPM><<<grid, GVPM_SHADE_THREADS, 0, stream>>>(P);
}

cudaError_t launch_bre_traverse(const GatherParams &P, bool dump, int sm_count, cudaStream_t stream) {
  if (P.ray_end <= P.ray_begin) return cudaSuccess;
  static void (*const kByMode[4])(const GatherParams &, int, cudaStream_t) = {
      launch_traverse_mode<0>, launch_traverse_mode<1>, launch_traverse_mode<2>, launch_traverse_mode<3>};
  kByMode[(dump ? 1 : 0) | (P.cfg.sppm_primal ? 2 : 0)](P, sm_count, stream);
  return cudaGetLastError();
}

cudaError_t launch_bre_shade(const GatherParams &P, unsigned long long total, int sm_count, cudaStream_t stream) {
  if (total == 0) return cudaSuccess;
  if (P.cfg.sppm_primal) launch_shade_mode<true>(P, total, sm_count, stream);
  else launch_shade_mode<false>(P, total, sm_count, stream);
  return cudaGetLastError();
}

}  // namespace gvpm
