// occluder_device.cuh — reconnection shadow rays: any-hit against the occluder triangles (gvpm_set_occluders), over
// the flat list (small sets, the synthetic walls) or down the occluder BVH (occluder_bvh.cu builds it).  Included by
// bre_device.cuh, so by every shade kernel that casts shadow rays.
//   Triangle::rayIntersect                      include/mitsuba/core/triangle.h:109-145
#pragma once
#include "gvpm_device.cuh"

namespace gvpm {

__device__ __forceinline__ float4 ldg4(const float4 *p) { return __ldg(p); }

// any-hit over the occluder list.  Two conservative culls precede the strictly rounded Moller-Trumbore test
// (|d| = 1): (1) the origin is farther from the triangle's plane than maxt; (2) the ray meets the plane at a
// parameter that is outside [mint, maxt] by more than the rounding of the strict test (the parent vertex of a
// reconnection usually lies ON a wall, whose plane it then meets at t ~ 0 < mint).  Single exit, so the lanes of a
// warp reconverge right after the loop.
__device__ __forceinline__ bool occluder_hit(const GatherParams &P, uint32_t t, v3 o, v3 d, sf mint, sf maxt,
                                             float omag) {
  const float4 pl = ldg4(P.tri_plane + t);
  const float sdist = pl.x * o.x.v + pl.y * o.y.v + pl.z * o.z.v + pl.w;
  if (fabsf(sdist) > maxt.v * 1.001f + 1e-5f) return false;
  const float nd = pl.x * d.x.v + pl.y * d.y.v + pl.z * d.z.v;
  const float and_ = fabsf(nd);
  if (and_ > 1e-3f) {
    // plane parameter tp = -sdist/nd; the strict tt differs from it by < aux.x * |o - p0| / |nd| (+ relative).
    // Compared after multiplying through by |nd| (no division).
    const float2 aux = __ldg(P.tri_aux + t);
    const float num = nd < 0.f ? sdist : -sdist;  // tp * |nd|
    const float slack = aux.x * (omag + aux.y + 1e-3f) * 1.7321f + 2e-6f * fabsf(num);
    if (num + slack < mint.v * and_ || num - slack > maxt.v * and_) return false;
  }
  const float *tv = P.tri + 9 * t;
  v3 p0(__ldg(tv), __ldg(tv + 1), __ldg(tv + 2)), p1(__ldg(tv + 3), __ldg(tv + 4), __ldg(tv + 5)),
      p2(__ldg(tv + 6), __ldg(tv + 7), __ldg(tv + 8));
  v3 edge1 = p1 - p0, edge2 = p2 - p0;
  v3 pvec = cross(d, edge2);
  sf det = dot(edge1, pvec);
  if (det.v == 0.f) return false;
  sf inv_det = sf(1.f) / det;
  v3 tvec = o - p0;
  sf u = dot(tvec, pvec) * inv_det;
  if (u.v < 0.f || u.v > 1.f) return false;
  v3 qvec = cross(tvec, edge1);
  sf v = dot(d, qvec) * inv_det;
  if (v.v >= 0.f && (u + v).v <= 1.f) {
    sf tt = dot(edge2, qvec) * inv_det;
    if (tt >= mint && tt <= maxt) return true;
  }
  return false;
}

// ---- occluder BVH (occluder_bvh.cu) ------------------------------------------------------------------------------------
// A binary radix tree over the Hilbert keys of the triangle centroids, GVPM_OCC_LEAF triangles per leaf, nodes in
// depth-first order (the left child of node i is i + 1) with 3 float4 each:
//   [0] lo.xyz, word: an inner node's escape index (first node after its subtree), or GVPM_OCC_LEAF_BIT | first
//       triangle of a leaf (it holds triangles [first, min(first + GVPM_OCC_LEAF, n_tri)); its escape is i + 1)
//   [1] hi.xyz, kappa: the largest rounding-slack coefficient tri_aux.x below the node
//   [2] axis.xyz, phi: every plane normal below the node lies within phi of +-axis (phi >= pi/2: no bound, e.g. a
//       zero-area triangle below)
// The triangle arrays (tri, tri_plane, tri_aux) are in leaf order, so a leaf reads contiguous triangles.
#define GVPM_OCC_LEAF 4
#define GVPM_OCC_LEAF_BIT 0x80000000u
#define GVPM_OCC_NODE_FLOAT4 3

// Stackless any-hit walk.  Contract: true exactly when the list loop over the same triangles is, because a leaf runs
// occluder_hit itself and a node is skipped only when no triangle below it can pass occluder_hit.
//
// Why the skip is safe.  A node is skipped only when its normal cone guarantees |n.d| > 1.001e-3 for every triangle
// below (cmin below; 1e-5 covers the rounding of the cone test, of |d| = 1 and of the float plane normals), so every
// triangle below runs occluder_hit's parameter cull and, to pass, has its exact plane parameter tp = -sdist/(n.d) in
// [mint - St, maxt + St] with
//   St = slack / |n.d| <= (kappa * 1.7321 * (omag + V + 1e-3) / cmin + 2e-6 * T) / (1 - 2e-6)
// (slack of occluder_hit with aux.x <= kappa, aux.y <= V = largest |coordinate| of the node box, |tp| <= T + St,
// T = max(|mint|, |maxt|)).  The plane point o + tp d is then within E of the triangle's closed area: the accepted
// barycentrics (u, v) differ from the exact ones by the relative rounding of det, < 6 eps l1 l2 / (|e1 x e2| |n.d|)
// = 0.36 aux.x / |n.d|, plus the rounding of the numerators, < 3 eps |o - p0| l1 l2 / (|e1 x e2| |n.d|); times the edge
// lengths (<= 2 * 1.7321 * V) that is E < 2 * aux.x * 1.7321 * (omag + V) / |n.d| <= 2 St.  The walk pads the box by
// pad = 4 St (twice what the argument needs) plus 2^-20 * (V + omag + T) for the rounding of the slab test itself, and
// tests the interval [mint - pad, maxt + pad]: a triangle that passes occluder_hit never sits in a skipped node.
// Grazing rays (|n.d| <= 1e-3) and zero-area or degenerate triangles (no plane: an unbounded cone, or a kappa so large
// that the pad covers everything) make the strict test decide with a tt of arbitrary error, so their nodes are never
// skipped on geometry: the cone test keeps them.
__device__ __forceinline__ bool occluded_bvh(const GatherParams &P, v3 o, v3 d, sf mint, sf maxt) {
  if (maxt < mint) return false;
  const float omag = fmaxf(fmaxf(fabsf(o.x.v), fabsf(o.y.v)), fabsf(o.z.v));
  const float T = fmaxf(fabsf(mint.v), fabsf(maxt.v));
  // a zero direction component is replaced by +-1e-20 (the segment moves by < T * 1e-20, inside the pad): the slab
  // products stay free of 0 * inf
  const float dx = fabsf(d.x.v) < 1e-20f ? copysignf(1e-20f, d.x.v) : d.x.v;
  const float dy = fabsf(d.y.v) < 1e-20f ? copysignf(1e-20f, d.y.v) : d.y.v;
  const float dz = fabsf(d.z.v) < 1e-20f ? copysignf(1e-20f, d.z.v) : d.z.v;
  const float ix = 1.f / dx, iy = 1.f / dy, iz = 1.f / dz;
  bool hit = false;
  uint32_t i = 0;
  while (i < P.n_occ_nodes && !hit) {
    const float4 *nd = P.occ_nodes + (size_t)GVPM_OCC_NODE_FLOAT4 * i;
    const float4 a = ldg4(nd), b = ldg4(nd + 1), c = ldg4(nd + 2);
    const uint32_t w = __float_as_uint(a.w);
    const bool leaf = (w & GVPM_OCC_LEAF_BIT) != 0u;
    bool enter = true;
    float sphi, cphi;
    __sincosf(c.w, &sphi, &cphi);
    const float ad = fabsf(c.x * d.x.v + c.y * d.y.v + c.z * d.z.v);
    const float cmin = ad * cphi - sqrtf(fmaxf(0.f, 1.f - ad * ad)) * sphi - 1e-5f;
    if (cmin > 1.001e-3f) {
      const float V = fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(b.x)), fmaxf(fabsf(a.y), fabsf(b.y))),
                            fmaxf(fabsf(a.z), fabsf(b.z)));
      const float St = (b.w * 1.7321f * (omag + V + 1e-3f) / cmin + 2e-6f * T) * 1.00001f;
      const float pad = 4.f * St + 9.5367431640625e-7f * (V + omag + T) + 1e-30f;
      float t1 = ((a.x - pad) - o.x.v) * ix, t2 = ((b.x + pad) - o.x.v) * ix;
      float tn = fminf(t1, t2), tf = fmaxf(t1, t2);
      t1 = ((a.y - pad) - o.y.v) * iy; t2 = ((b.y + pad) - o.y.v) * iy;
      tn = fmaxf(tn, fminf(t1, t2)); tf = fminf(tf, fmaxf(t1, t2));
      t1 = ((a.z - pad) - o.z.v) * iz; t2 = ((b.z + pad) - o.z.v) * iz;
      tn = fmaxf(tn, fminf(t1, t2)); tf = fminf(tf, fmaxf(t1, t2));
      enter = tn <= tf && tf >= mint.v - pad && tn <= maxt.v + pad;
    }
    if (enter && leaf) {
      const uint32_t first = w & ~GVPM_OCC_LEAF_BIT;
      const uint32_t last = min(first + GVPM_OCC_LEAF, P.n_tri);
      for (uint32_t t = first; t < last && !hit; ++t) hit = occluder_hit(P, t, o, d, mint, maxt, omag);
    }
    i = (enter || leaf) ? i + 1 : w;
  }
  return hit;
}

// ---- closest hit on the mesh scene (MeshScene, gvpm_set_trace_mesh) ------------------------------------------------------
// occluder_hit's culls and strict test on triangle s of the mesh, returning the strict parameter tt when the test
// accepts it in [mint, maxt], else +inf.  The culls are occluder_hit's, so they never reject a triangle whose strict tt
// lies in [mint, maxt].
__device__ __forceinline__ float mesh_tri_t(const MeshScene &M, uint32_t s, v3 o, v3 d, sf mint, sf maxt, float omag) {
  const float4 pl = ldg4(M.plane + s);
  const float sdist = pl.x * o.x.v + pl.y * o.y.v + pl.z * o.z.v + pl.w;
  if (fabsf(sdist) > maxt.v * 1.001f + 1e-5f) return INFINITY;
  const float nd = pl.x * d.x.v + pl.y * d.y.v + pl.z * d.z.v;
  const float and_ = fabsf(nd);
  if (and_ > 1e-3f) {
    const float2 aux = __ldg(M.aux + s);
    const float num = nd < 0.f ? sdist : -sdist;
    const float slack = aux.x * (omag + aux.y + 1e-3f) * 1.7321f + 2e-6f * fabsf(num);
    if (num + slack < mint.v * and_ || num - slack > maxt.v * and_) return INFINITY;
  }
  const float *tv = M.tri + 9 * (size_t)s;
  v3 p0(__ldg(tv), __ldg(tv + 1), __ldg(tv + 2)), p1(__ldg(tv + 3), __ldg(tv + 4), __ldg(tv + 5)),
      p2(__ldg(tv + 6), __ldg(tv + 7), __ldg(tv + 8));
  v3 edge1 = p1 - p0, edge2 = p2 - p0;
  v3 pvec = cross(d, edge2);
  sf det = dot(edge1, pvec);
  if (det.v == 0.f) return INFINITY;
  sf inv_det = sf(1.f) / det;
  v3 tvec = o - p0;
  sf u = dot(tvec, pvec) * inv_det;
  if (u.v < 0.f || u.v > 1.f) return INFINITY;
  v3 qvec = cross(tvec, edge1);
  sf v = dot(d, qvec) * inv_det;
  if (v.v >= 0.f && (u + v).v <= 1.f) {
    sf tt = dot(edge2, qvec) * inv_det;
    if (tt >= mint && tt <= maxt) return tt.v;
  }
  return INFINITY;
}

// Closest hit: the triangle with the smallest strict tt in (1e-6, bound], ties to the smaller caller index, never the
// triangle `skip` (the one the ray starts on); slot = kMeshNone when there is none.  The brute-force loop over all
// triangles with the same rule gives the same answer.
constexpr uint32_t kMeshNone = 0xffffffffu;
struct MeshHit { float t; uint32_t slot, idx; };
// The stackless walk of occluded_bvh with a shrinking upper bound: maxt = the best tt found so far (the box exit at
// first).  occluded_bvh's argument holds for any interval [mint, maxt]: a node is skipped only when no triangle below
// it can pass the culls and strict test of occluder_hit (here mesh_tri_t) with a tt in [mint, maxt].  Here the interval
// at the time of the skip is [1e-6, B], B the best tt so far, and B only decreases: a skipped triangle has no tt in
// [1e-6, B], so it cannot beat B, nor the final answer <= B, nor tie with it (a tie needs tt = final <= B).  The pad uses
// T from the first bound, which is >= every later one, so it is never smaller than the argument needs.  Skipping
// `skip` and keeping the smaller index on equal tt are decisions on triangles that the walk did reach, in any order.
__device__ __forceinline__ MeshHit closest_hit_bvh(const MeshScene &M, v3 o, v3 d, sf bound, uint32_t skip) {
  MeshHit best{bound.v, kMeshNone, kMeshNone};
  const sf mint(1e-6f);
  if (bound < mint) return best;
  const float omag = fmaxf(fmaxf(fabsf(o.x.v), fabsf(o.y.v)), fabsf(o.z.v));
  const float T = fmaxf(fabsf(mint.v), fabsf(bound.v));
  const float dx = fabsf(d.x.v) < 1e-20f ? copysignf(1e-20f, d.x.v) : d.x.v;
  const float dy = fabsf(d.y.v) < 1e-20f ? copysignf(1e-20f, d.y.v) : d.y.v;
  const float dz = fabsf(d.z.v) < 1e-20f ? copysignf(1e-20f, d.z.v) : d.z.v;
  const float ix = 1.f / dx, iy = 1.f / dy, iz = 1.f / dz;
  uint32_t i = 0;
  while (i < M.n_nodes) {
    const float4 *nd = M.nodes + (size_t)GVPM_OCC_NODE_FLOAT4 * i;
    const float4 a = ldg4(nd), b = ldg4(nd + 1), c = ldg4(nd + 2);
    const uint32_t w = __float_as_uint(a.w);
    const bool leaf = (w & GVPM_OCC_LEAF_BIT) != 0u;
    bool enter = true;
    float sphi, cphi;
    __sincosf(c.w, &sphi, &cphi);
    const float ad = fabsf(c.x * d.x.v + c.y * d.y.v + c.z * d.z.v);
    const float cmin = ad * cphi - sqrtf(fmaxf(0.f, 1.f - ad * ad)) * sphi - 1e-5f;
    if (cmin > 1.001e-3f) {
      const float V = fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(b.x)), fmaxf(fabsf(a.y), fabsf(b.y))),
                            fmaxf(fabsf(a.z), fabsf(b.z)));
      const float St = (b.w * 1.7321f * (omag + V + 1e-3f) / cmin + 2e-6f * T) * 1.00001f;
      const float pad = 4.f * St + 9.5367431640625e-7f * (V + omag + T) + 1e-30f;
      float t1 = ((a.x - pad) - o.x.v) * ix, t2 = ((b.x + pad) - o.x.v) * ix;
      float tn = fminf(t1, t2), tf = fmaxf(t1, t2);
      t1 = ((a.y - pad) - o.y.v) * iy; t2 = ((b.y + pad) - o.y.v) * iy;
      tn = fmaxf(tn, fminf(t1, t2)); tf = fminf(tf, fmaxf(t1, t2));
      t1 = ((a.z - pad) - o.z.v) * iz; t2 = ((b.z + pad) - o.z.v) * iz;
      tn = fmaxf(tn, fminf(t1, t2)); tf = fminf(tf, fmaxf(t1, t2));
      enter = tn <= tf && tf >= mint.v - pad && tn <= best.t + pad;
    }
    if (enter && leaf) {
      const uint32_t first = w & ~GVPM_OCC_LEAF_BIT;
      const uint32_t last = min(first + GVPM_OCC_LEAF, M.n_tri);
      for (uint32_t s = first; s < last; ++s) {
        const uint32_t idx = __ldg(M.perm + s);
        if (idx == skip) continue;
        const float tt = mesh_tri_t(M, s, o, d, mint, sf(best.t), omag);
        if (tt > 1e-6f && (tt < best.t || (tt == best.t && idx < best.idx))) best = MeshHit{tt, s, idx};
      }
    }
    i = (enter || leaf) ? i + 1 : w;
  }
  return best;
}

// BVH: compile-time variant of the shade kernels (the list instantiations carry none of the walk)
template <bool BVH>
__device__ __forceinline__ bool occluded(const GatherParams &P, v3 o, v3 d, sf mint, sf maxt) {
  if (BVH) return occluded_bvh(P, o, d, mint, maxt);
  bool hit = false;
  if (maxt < mint) return false;
  const float omag = fmaxf(fmaxf(fabsf(o.x.v), fabsf(o.y.v)), fabsf(o.z.v));
  for (uint32_t t = 0; t < P.n_tri && !hit; ++t) hit = occluder_hit(P, t, o, d, mint, maxt, omag);
  return hit;
}
// Shadow rays of one (ray, photon) pair share their origin (the parent vertex): the triangles whose plane lies
// within `bound` of it are found once per pair (bit t of the mask, n_tri <= 32); a shadow ray whose plane-distance
// cull radius fits inside `bound` then visits only those.
struct OccluderNear { uint32_t mask; float bound; };
__device__ __forceinline__ OccluderNear occluders_near(const GatherParams &P, v3 o, float bound) {
  OccluderNear n;
  n.mask = 0u;
  n.bound = P.n_tri <= 32u ? bound : -1.f;
  // unrolled 4-fold, so 4 plane loads are in flight: nvcc's own choice (16-fold, all 16 loads in flight) made this loop
  // the register peak of the shade kernels
  if (P.n_tri <= 32u)
#pragma unroll 4
    for (uint32_t t = 0; t < P.n_tri; ++t) {
      const float4 pl = ldg4(P.tri_plane + t);
      if (fabsf(pl.x * o.x.v + pl.y * o.y.v + pl.z * o.z.v + pl.w) <= bound) n.mask |= 1u << t;
    }
  return n;
}
template <bool BVH>
__device__ __forceinline__ bool occluded_near(const GatherParams &P, const OccluderNear &n, v3 o, v3 d, sf mint, sf maxt) {
  if (!(maxt.v * 1.001f + 1e-5f <= n.bound)) return occluded<BVH>(P, o, d, mint, maxt);
  bool hit = false;
  if (maxt < mint) return false;
  const float omag = fmaxf(fmaxf(fabsf(o.x.v), fabsf(o.y.v)), fabsf(o.z.v));
  for (uint32_t m = n.mask; m != 0u && !hit; m &= m - 1u) hit = occluder_hit(P, __ffs(m) - 1, o, d, mint, maxt, omag);
  return hit;
}

}  // namespace gvpm
