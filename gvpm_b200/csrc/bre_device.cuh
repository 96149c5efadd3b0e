// bre_device.cuh — device functions of the G-BRE gather shared by the traversal and shading kernels.
// Reference lines restated here:
//   neighbour predicate                         gvpm/gvpm_accel.h:293-301
//   VolumeGradientBREQuery::operator()          gvpm/shift/shift_volume_photon.cpp:658-856
//   shiftNull / shiftPhotonDiffuse / getShiftPos    shift_volume_photon.cpp:119-158,382-486,858-896
//   diffuseReconnection                         gvpm/shift/operation/shift_diffuse.cpp:11-134
//   HomogeneousMedium::eval, phase eval         src/medium/homogeneous.cpp:432-513, src/phase/hg.cpp:107-110
//   Triangle::rayIntersect                      include/mitsuba/core/triangle.h:109-145
#pragma once
#include "gvpm_device.cuh"

namespace gvpm {

__device__ __forceinline__ float4 ldg4(const float4 *p) { return __ldg(p); }

// conservative slab test of a box (inflated by the radius at build time) against the ray interval
// [tlo, thi]; the rounding/packet pad is folded into the origin: (lo - pad) - o == lo - (o + pad)
__device__ __forceinline__ bool box_hit(const Tree &t, uint32_t i, float oxp, float oxm, float oyp, float oym,
                                        float ozp, float ozm, float ix, float iy, float iz, float tlo,
                                        float thi) {
  const float4 lo = ldg4(t.lo + i), hi = ldg4(t.hi + i);
  float t1 = (lo.x - oxp) * ix, t2 = (hi.x - oxm) * ix;
  float tn = fminf(t1, t2), tf = fmaxf(t1, t2);
  t1 = (lo.y - oyp) * iy; t2 = (hi.y - oym) * iy;
  tn = fmaxf(tn, fminf(t1, t2)); tf = fminf(tf, fmaxf(t1, t2));
  t1 = (lo.z - ozp) * iz; t2 = (hi.z - ozm) * iz;
  tn = fmaxf(tn, fminf(t1, t2)); tf = fminf(tf, fmaxf(t1, t2));
  return tn <= tf && tf >= tlo && tn <= thi;
}

// 1/max(2*deltaT, 0.0001) as the reference evaluates it in double then rounds to Float
// (shift_volume_photon.cpp:723): identical to this fp32 form (checked exhaustively-ish in tests/).
__device__ __forceinline__ sf chord_pdf(sf deltaT) {
  sf x2 = deltaT * sf(2.f);
  return (x2.v <= 0.0001f) ? sf(10000.f) : frcp(x2);   // a pdf: radiometric only (2 ulp)
}

struct MediumRec { sf T, pdfSuccess, pdfFailure; };

// HomogeneousMedium::eval with equal sigma_t over channels (enforced at gvpm_set_medium as the
// reference does, homogeneous.cpp:188-201): transmittance is one scalar.
__device__ __forceinline__ MediumRec medium_eval(const GatherParams &P, sf mint, sf maxt) {
  MediumRec r;
  sf distance = maxt - mint;
  sf st(P.sigma_t[0]);
  sf tmp(expf(((-st) * distance).v));
  sf ps = st * tmp;
  ps = ((ps + ps) + ps) / sf(3.f);
  r.pdfSuccess = ps * sf(P.sampling_weight);
  const sf pf = ((tmp + tmp) + tmp) / sf(3.f);
  r.pdfFailure = pf * sf(P.sampling_weight) + (sf(1.f) - sf(P.sampling_weight));
  r.T = tmp;
  if (r.T.v < 1e-20f) r.T = sf(0.f);
  return r;
}

__device__ __forceinline__ sf phase_eval(const GatherParams &P, v3 wi, v3 wo) {
  if (P.phase_type == GVPM_PHASE_ISOTROPIC) return sf(GVPM_INV_FOURPI);
  sf g(P.hg_g);
  sf temp = sf(1.f) + g * g + sf(2.f) * g * dot(wi, wo);
  return sf(GVPM_INV_FOURPI) * (sf(1.f) - g * g) / (temp * ssqrt(temp));
}

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
__device__ __forceinline__ bool occluded(const GatherParams &P, v3 o, v3 d, sf mint, sf maxt) {
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
  if (P.n_tri <= 32u)
    for (uint32_t t = 0; t < P.n_tri; ++t) {
      const float4 pl = ldg4(P.tri_plane + t);
      if (fabsf(pl.x * o.x.v + pl.y * o.y.v + pl.z * o.z.v + pl.w) <= bound) n.mask |= 1u << t;
    }
  return n;
}
__device__ __forceinline__ bool occluded_near(const GatherParams &P, const OccluderNear &n, v3 o, v3 d, sf mint, sf maxt) {
  if (!(maxt.v * 1.001f + 1e-5f <= n.bound)) return occluded(P, o, d, mint, maxt);
  bool hit = false;
  if (maxt < mint) return false;
  const float omag = fmaxf(fmaxf(fabsf(o.x.v), fabsf(o.y.v)), fabsf(o.z.v));
  for (uint32_t m = n.mask; m != 0u && !hit; m &= m - 1u) hit = occluder_hit(P, __ffs(m) - 1, o, d, mint, maxt, omag);
  return hit;
}

// coordinateSystemCoherent, src/libcore/util.cpp:592-599
__device__ __forceinline__ void coherent_frame(v3 n, v3 &b1, v3 &b2) {
  const sf sign(copysignf(1.0f, n.z.v));
  const sf a = sf(-1.0f) / (sign + n.z);
  const sf b = n.x * n.y * a;
  b1 = v3(sf(1.0f) + sign * n.x * n.x * a, sign * b, -sign * n.x);
  b2 = v3(b, sign + n.y * n.y * a, -n.y);
}

struct BaseRay {
  v3 o, d, eye;
  sf mint, maxt, edgeLen, xi;
  int px, py, edgeId;
};

// works on shared or global (read-only) record pointers
__device__ __forceinline__ BaseRay load_base_ray(const float4 *rec) {
  BaseRay R;
  const float4 b0 = rec[0], b1 = rec[1], b2 = rec[2], b3 = rec[3];
  R.o = v3(b0.x, b0.y, b0.z); R.mint = sf(b0.w);
  R.d = v3(b1.x, b1.y, b1.z); R.maxt = sf(b1.w);
  R.eye = v3(b2.x, b2.y, b2.z); R.edgeLen = sf(b2.w);
  R.xi = sf(b3.x);
  R.px = (int)__float_as_uint(b3.y); R.py = (int)__float_as_uint(b3.z);
  R.edgeId = (int)__float_as_uint(b3.w);
  return R;
}

__device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}

// sppm's primal BeamRadianceEstimator::query (photonmapper/bre.cpp:167-259): the ray is re-based at ray(mint)
// (:169), the predicate is diskDistance > 0 && distSqr < r^2 (:204), the 3-D kernel stops early when
// diskDistance - 2r > maxt (:206), draws its uniform PER PHOTON (:217; here a counter-based hash of the ray and
// the caller's photon index) and keeps t' in [0, maxt]; the 2-D kernel keeps diskDistance <= maxt (:240).
// tBase is the distance from the re-based origin, pdfCam returns 1 / invPdfSampling.
__device__ __forceinline__ float sppm_uniform(const GatherParams &P, const BaseRay &R, uint32_t photonIndex) {
  uint32_t h = hash32(P.cfg.rng_seed ^ 0x9E3779B9u);
  h = hash32(h ^ (uint32_t)R.px);
  h = hash32(h ^ ((uint32_t)R.py * 0x85EBCA6Bu));
  h = hash32(h ^ ((uint32_t)R.edgeId * 0xC2B2AE35u));
  h = hash32(h ^ photonIndex);
  return (float)(h >> 8) * (1.0f / 16777216.0f);
}
__device__ __forceinline__ bool sppm_distance(const GatherParams &P, const BaseRay &R, v3 p, uint32_t photonIndex,
                                              sf &tBase, sf &invPdf) {
  const v3 ro = R.o + R.mint * R.d;
  const sf rmaxt = R.maxt - R.mint;
  const v3 oc = p - ro;
  const sf dd = dot(oc, R.d);
  const sf r(P.radius), radSqr = r * r;
  const sf distSqr = length_sq((ro + dd * R.d) - p);
  if (!(dd.v > 0.f && distSqr < radSqr)) return false;
  if (P.cfg.kernel_3d) {
    if (dd - (r * sf(2.f)) > rmaxt) return false;
    const sf deltaT = ssqrt(radSqr - distSqr);
    const sf tminKernel = dd - deltaT;
    const sf tRand = tminKernel + (sf(2.f) * deltaT) * sf(sppm_uniform(P, R, photonIndex));
    if (tRand.v < 0.f || tRand > rmaxt) return false;
    tBase = tRand;
    invPdf = smax(sf(2.0f) * deltaT, sf(0.0001f));
  } else {
    if (dd > rmaxt) return false;
    tBase = dd;
    invPdf = sf(1.f);
  }
  return true;
}

// Neighbour predicate + kernel-chord sampling of the 3-D kernel (gvpm_accel.h:297-301,
// shift_volume_photon.cpp:707-724).  False when the photon is outside the geometric neighbour set.
// SPPM (compile-time, so the gvpm kernels carry none of it): sppm's primal query instead, see sppm_distance.
template <bool SPPM>
__device__ __forceinline__ bool base_distance(const GatherParams &P, const BaseRay &R, v3 p, uint32_t photonIndex,
                                              sf &tBase, sf &pdfCam) {
  if (SPPM) return sppm_distance(P, R, p, photonIndex, tBase, pdfCam);  // photonIndex: the caller's (original) index
  v3 oc = p - R.o;
  sf dd = dot(oc, R.d);
  sf distSqr = length_sq((R.o + dd * R.d) - p);
  if (!(dd > R.mint && distSqr < sf(P.radius_sq))) return false;
  if (P.cfg.kernel_3d) {
    sf r(P.radius);
    sf deltaT = safe_sqrt(r * r - distSqr);
    sf tminKernel = dd - deltaT;
    sf tRand = tminKernel + (deltaT * sf(2.f)) * R.xi;
    if (tRand < R.mint || tRand > R.edgeLen) return false;
    tBase = tRand;
    pdfCam = chord_pdf(deltaT);
  } else {
    if (dd > R.edgeLen) return false;  // explicit bound, DESIGN.md §6 (bre.cpp:240-242)
    tBase = dd;
    pdfCam = sf(1.f);
  }
  return true;
}

// depth / interaction-mode / pathSet filters, shift_volume_photon.cpp:670-697
template <bool SPPM>
__device__ __forceinline__ bool filters_pass(const GatherParams &P, const BaseRay &R, uint32_t meta) {
  int type = meta & 3, depth = (meta >> 2) & 255, parity = (meta >> 10) & 1;
  int pathLen = depth + R.edgeId;
  if (SPPM)  // bre.cpp:195-198 with maxDepth = m_maxDepth - beam.depth (sppm.cpp:978); nothing else
    return !(P.cfg.max_depth != -1 && depth > P.cfg.max_depth - R.edgeId);
  if (P.cfg.max_depth > 0 && pathLen > P.cfg.max_depth) return false;
  if (P.cfg.min_depth != 0 && pathLen < P.cfg.min_depth) return false;
  int m = P.cfg.lighting_mode;
  if (!((m & GVPM_SURF2MEDIA) && (m & GVPM_MEDIA2MEDIA))) {
    if (type == GVPM_PARENT_MEDIUM && !(m & GVPM_MEDIA2MEDIA)) return false;
    if (type != GVPM_PARENT_MEDIUM && !(m & GVPM_SURF2MEDIA)) return false;
  }
  if (P.cfg.path_set && parity != ((R.px + R.py) % 2)) return false;
  return true;
}

__device__ __forceinline__ void acc_add(float *a, int j, v3 c) {
  a[3 * j] += c.x.v; a[3 * j + 1] += c.y.v; a[3 * j + 2] += c.z.v;
}

// A photon record as the shift code reads it (8 x 128-bit loads, DESIGN.md §3; unused fields cost no load)
struct PhotonRec {
  v3 p, flux, parent, wiW, pn, prefix, albedo, wi;
  sf parentPdf, edgePdf, rrW, cosI, nEdge, lBase;
  int ptype;
};
__device__ __forceinline__ PhotonRec load_photon_orig(const GatherParams &P, uint32_t origIndex);
__device__ __forceinline__ PhotonRec load_photon(const GatherParams &P, uint32_t pi) {
  return load_photon_orig(P, __ldg(P.orig + pi));
}
// same, by the caller's photon index (the BRE pair list carries it, so the shading kernel can prefetch the record)
__device__ __forceinline__ PhotonRec load_photon_orig(const GatherParams &P, uint32_t origIndex) {
  // one aligned 128-byte record in the caller's order (gvpm_device.cuh photon_record), reached through the sorted
  // slot's original index: 4 sectors per photon instead of 7 half-used ones from per-field planes
  const float4 *r = P.aos + (size_t)origIndex * 8;
  const float4 q0 = ldg4(r), q1 = ldg4(r + 1), q2 = ldg4(r + 2), q3 = ldg4(r + 3), q4 = ldg4(r + 4), q5 = ldg4(r + 5),
               q6 = ldg4(r + 6), q7 = ldg4(r + 7);
  PhotonRec ph;
  ph.p = v3(q0.x, q0.y, q0.z); ph.flux = v3(q1.x, q1.y, q1.z); ph.parent = v3(q2.x, q2.y, q2.z);
  ph.wiW = v3(q3.x, q3.y, q3.z); ph.pn = v3(q4.x, q4.y, q4.z); ph.prefix = v3(q5.x, q5.y, q5.z);
  ph.albedo = v3(q6.x, q6.y, q6.z); ph.wi = v3(q7.y, q7.z, q7.w);
  ph.parentPdf = sf(q1.w); ph.edgePdf = sf(q2.w); ph.rrW = sf(q3.w);
  ph.cosI = sf(q4.w); ph.nEdge = sf(q5.w); ph.lBase = sf(q6.w);
  ph.ptype = __float_as_uint(q0.w) & 3;
  return ph;
}

// AbstractVolumeGradientRecord::shiftNull, shift_volume_photon.cpp:119-158 (jacobian = 1); flux, wi: the photon's
__device__ __forceinline__ void shift_null(const GatherParams &P, v3 flux, v3 wi, v3 dk, v3 eyeK, sf sensor, sf Tshift,
                                           sf pdfBase, sf pdfShift, v3 &S, sf &weight) {
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);
  v3 c = (sigS * flux) * phase_eval(P, wi, -dk);
  S = (c * Tshift) * eyeK;
  weight = sf(0.5f);
  if (P.cfg.use_mis) {
    if (pdfShift.v == 0.f || pdfBase.v == 0.f) weight = sf(1.f);
    else weight = frcp(sf(1.f) + sensor * fdiv(pdfShift, pdfBase));
  }
}

// AbstractVolumeGradientRecord::getShiftPos, shift_volume_photon.cpp:858-896
__device__ __forceinline__ v3 get_shift_pos(const GatherParams &P, sf rr2, v3 p, v3 zBase, v3 zShift, v3 dBase,
                                            v3 dk, bool coherent) {
  v3 offsetPos = zShift + (p - zBase);
  if (coherent) {  // coherent frames for the 2-D kernel, :866-873
    v3 bs, bt, ns, nt;
    coherent_frame(dBase, bs, bt);
    coherent_frame(dk, ns, nt);
    const v3 v = p - zBase;
    const v3 local(dot(v, bs), dot(v, bt), dot(v, dBase));
    offsetPos = zShift + ((ns * local.x + nt * local.y) + dk * local.z);
  }
  if (P.cfg.use_shift_null) {
    sf offDistSqr = length_sq(zBase - offsetPos);
    if (offDistSqr < rr2) {
      v3 dShift = zShift - zBase;
      dShift = dShift / length(dShift);
      sf cosD = dot(dShift, -(offsetPos - zShift));
      offsetPos = offsetPos + (dShift * cosD) * sf(2.f);
    }
  }
  return offsetPos;
}

// shiftPhoton -> shiftPhotonDiffuse (shift_volume_photon.cpp:49-117,382-486) with diffuseReconnection
// (shift_diffuse.cpp:11-134) inlined for {area emitter, diffuse surface, medium} parents.
// S, weight keep their defaults (0, 1) when the shift fails.  Written without early returns so that the lanes of a
// warp reconverge after every decision (the reference's `return false` paths are the untaken branches).
// The terms that depend on the photon alone (wiW, cosI, nEdge) come from its record; `near` is the pair's
// occluders_near of the parent (pair_occluders).
// Shadow rays run from the parent towards the offset photon over maxt = lProj * shadow_maxt_scale; twice the base edge
// length bounds lProj for every coherent offset (longer ones fall back to the full occluder loop).  Built per pair, not
// per photon: the occluders and shadow_maxt_scale may change between the build and the gather.
__device__ __forceinline__ OccluderNear pair_occluders(const GatherParams &P, v3 parent, sf lBase) {
  return occluders_near(P, parent, 2.f * (lBase.v * P.cfg.shadow_maxt_scale * 1.001f + 1e-5f));
}
__device__ __forceinline__ void shift_photon_diffuse(const GatherParams &P, const PhotonRec &ph, const OccluderNear &near,
                                                     v3 offsetPos, v3 dk, v3 eyeK, sf sensor, sf Tshift, sf pdfBase,
                                                     sf pdfShift, v3 &S, sf &weight) {
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);
  v3 dProj = offsetPos - ph.parent;
  const sf lProj = length(dProj);
  dProj = dProj / lProj;
  // manifold shift (glossy parent): out of scope, fails like useManifold=false
  bool ok = ph.ptype != GVPM_PARENT_OTHER;
  if (ok) ok = !occluded_near(P, near, ph.parent, dProj, sf(P.cfg.epsilon), lProj * sf(P.cfg.shadow_maxt_scale));
  // type-specific terms of diffuseReconnection
  const v3 wiW = ph.wiW;
  const sf cosO = dot(ph.pn, dProj);
  v3 thr(1.f, 1.f, 1.f);
  sf pdfValue(0.f);
  bool early = false;
  if (ph.ptype == GVPM_PARENT_MEDIUM) {
    const sf phv = phase_eval(P, wiW, dProj);
    thr = sigS * phv;
    pdfValue = phv;
  } else {
    // side test on surface / emitter parents, :404-412 (the sign of a quotient is the sign test the reference does)
    const sf signDot = cosO / ph.nEdge;
    if (signDot.v < 0.f) ok = false;
    if (ph.ptype == GVPM_PARENT_SURFACE) {  // bsdfs/diffuse.cpp:110-127
      const sf cosI = ph.cosI;
      if (cosI.v <= 0.f || cosO.v <= 0.f) {
        thr = v3(0.f, 0.f, 0.f);
      } else {
        thr = ph.albedo * (sf(GVPM_INV_PI) * cosO);
        pdfValue = sf(GVPM_INV_PI) * cosO;
      }
      if ((cosI * cosI).v <= 0.f || (cosO * cosO).v <= 0.f) early = true;
    } else {  // emitter sample, emitters/area.cpp:132-150
      sf dp = cosO;
      if (dp.v < 0.f) dp = sf(0.f);
      const sf e = sf(GVPM_INV_PI) * dp;
      thr = v3(e, e, e);
      pdfValue = e;
    }
  }
  sf sPdf(0.f);
  if (!early) {
    const sf GOp = sf(1.f) / (lProj * lProj);
    sPdf = pdfValue * GOp;
    thr = thr * GOp;
    if (ph.parentPdf.v == 0.f) {
      sPdf = sf(0.f);
    } else {
      const MediumRec mr = medium_eval(P, sf(0.f), lProj);
      sPdf = sPdf * mr.pdfSuccess;
      // thr / parentPdf * rrW * (T / edgePdf): radiometric only
      thr = thr * (fdiv(ph.rrW, ph.parentPdf) * fdiv(mr.T, ph.edgePdf));
    }
  }
  if (ok) {
    if (sPdf.v == 0.f) {
      weight = sf(1.f);
    } else {
      const v3 photonWeight = ph.prefix * thr;
      const v3 c = (sigS * photonWeight) * phase_eval(P, -dProj, -dk);
      S = (c * Tshift) * eyeK;
      weight = sf(0.5f);
      if (P.cfg.use_mis) {
        const sf basePdf = (pdfBase * ph.parentPdf) * ph.edgePdf;
        const sf offsetPdf = sPdf * pdfShift;
        if (offsetPdf.v == 0.f || basePdf.v == 0.f) {
          weight = sf(1.f);
        } else {
          const sf q = sensor * fdiv(offsetPdf, basePdf);
          weight = P.cfg.power_heuristic ? frcp(sf(1.f) + q * q) : frcp(sf(1.f) + q);
        }
      }
    }
  }
}

// One contributing (ray, photon) pair: VolumeGradientBREQuery::operator() after the filters.
// rec: the ray's 20 float4 (base + 4 offsets); pi: the photon's ORIGINAL index; a: 27 accumulators (registers of the
// caller).
template <bool SPPM>
__device__ __forceinline__ void bre_photon(const GatherParams &P, const float4 *__restrict__ rec, uint32_t pi,
                                           float *a) {
  const BaseRay R = load_base_ray(rec);
  const PhotonRec ph = load_photon_orig(P, pi);
  const sf r(P.radius), rr2 = r * r;
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);

  sf tBase, pdfCam;
  if (!base_distance<SPPM>(P, R, ph.p, pi, tBase, pdfCam)) return;  // cannot happen for an emitted pair
  if (SPPM) {
    // result += T(0..t') * power * phase(wi, -d) * weight * invPdfSampling (bre.cpp:224-233,244-252), * beam.weight
    const v3 wi = ph.wi;
    const MediumRec mB = medium_eval(P, sf(0.f), tBase);
    const sf weight = sf(1.f) / sf(P.kernel_vol);
    const v3 c = ((ph.flux * mB.T) * phase_eval(P, wi, -R.d)) * (weight * pdfCam);
    acc_add(a, 0, c * R.eye);
    return;
  }
  const sf rrG = P.cfg.path_set ? sf(2.f) : sf(1.f);
  const v3 wi = ph.wi;
  const MediumRec mBase = medium_eval(P, R.mint, tBase);
  const v3 contrib = (sigS * ph.flux) * phase_eval(P, wi, -R.d);
  const v3 baseContrib = (contrib * mBase.T) * R.eye;
  const sf norm = sf(P.kernel_vol) * pdfCam;
  const sf recip = frcp(norm);
  acc_add(a, 0, (baseContrib * recip) * rrG);

  const MediumRec mShift = medium_eval(P, sf(P.cfg.epsilon), tBase);
  const v3 zBase = R.o + tBase * R.d;
  const OccluderNear near = pair_occluders(P, ph.parent, ph.lBase);

  // The offset loop is kept rolled (one copy of the shift code); k is warp-uniform, so the accumulation goes
  // through a switch with static register indices instead of a local-memory staging array.
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    const float4 s0 = ldg4(rec + 4 * (k + 1)), s1 = ldg4(rec + 4 * (k + 1) + 1), s2 = ldg4(rec + 4 * (k + 1) + 2);
    sf weight(1.f);
    v3 S(0.f, 0.f, 0.f);
    if (__float_as_uint(s2.w) != 0u) {  // validVolumeEdge, shift_cameraPath.h:135-140
      const v3 ok(s0.x, s0.y, s0.z), dk(s1.x, s1.y, s1.z), eyeK(s2.x, s2.y, s2.z);
      const sf lenK(s0.w), sensor(s1.w);
      const v3 zShift = ok + tBase * dk;
      bool done = false;
      if (P.cfg.use_shift_null && P.cfg.kernel_3d) {  // :776-802
        sf ZPtoY = length_sq(zShift - ph.p);
        if (ZPtoY < rr2 && tBase < lenK) {
          sf dd = dot(ph.p - ok, dk);
          sf ds = length_sq((ok + dd * dk) - ph.p);
          sf pdfShift = chord_pdf(safe_sqrt(rr2 - ds));
          shift_null(P, ph.flux, wi, dk, eyeK, sensor, mShift.T, pdfCam, pdfShift, S, weight);
          done = true;
        }
      }
      if (!done && lenK >= tBase) {  // :809-838
        const v3 offsetPos = get_shift_pos(P, rr2, ph.p, zBase, zShift, R.d, dk, !P.cfg.kernel_3d);
        sf pdfShift(1.f);
        if (P.cfg.kernel_3d) {
          sf dd = dot(offsetPos - ok, dk);
          sf ds = length_sq((ok + dd * dk) - offsetPos);
          pdfShift = chord_pdf(safe_sqrt(rr2 - ds));
        }
        shift_photon_diffuse(P, ph, near, offsetPos, dk, eyeK, sensor, mShift.T, pdfCam, pdfShift, S, weight);
      }
    }
    if ((k == 1 && R.px == P.cfg.film_w - 1) || (k == 2 && R.py == P.cfg.film_h - 1)) weight = sf(1.f);
    const sf rw = rrG * weight;
    const v3 wB = (baseContrib * rw) * recip, wS = (S * rw) * recip;
    switch (k) {
      case 0: acc_add(a, 5, wB); acc_add(a, 1, wS); break;
      case 1: acc_add(a, 6, wB); acc_add(a, 2, wS); break;
      case 2: acc_add(a, 7, wB); acc_add(a, 3, wS); break;
      default: acc_add(a, 8, wB); acc_add(a, 4, wS); break;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Warp-cooperative form of bre_photon<false> (same arithmetic, same accumulation order, bit-identical results).
// In a warp of 32 pairs roughly half of the (pair, offset) combinations take the cheap null shift and half the
// expensive diffuse reconnection, so the per-lane offset loop ran the reconnection four times with ~18 of 32 lanes
// busy.  Here phase A (lane = pair) does the base term, classifies the four offsets, finishes null shifts and
// invalid offsets on the spot and queues the reconnections as (pair, k) tasks; phase B hands the tasks out 32 at a
// time, so the reconnection code always runs with full lanes (the pair's context travels through shared memory);
// phase C (lane = pair) folds the four results in k order.
#define GVPM_CTX_STRIDE 33
struct ShadeShared {               // per warp
  float ctx[32][GVPM_CTX_STRIDE];  // odd stride: lanes reading one field of 32 different pairs hit 32 banks
  float4 res[32][5];               // (S.xyz, weight) per (pair, k); row stride 5 float4: conflict-free 128-bit access
  uint8_t tasks[128];              // (pair << 2) | k
};
enum {  // float slots of ctx[pair]
  CX_P = 0, CX_PARENT = 3, CX_PN = 6, CX_PREFIX = 9, CX_ALBEDO = 12, CX_PARENTPDF = 15, CX_EDGEPDF = 16, CX_RRW = 17,
  CX_PTYPE = 18, CX_WIW = 19, CX_COSI = 22, CX_NEDGE = 23, CX_NEARMASK = 24, CX_NEARBOUND = 25, CX_ZBASE = 26,
  CX_TBASE = 29, CX_PDFCAM = 30, CX_TSHIFT = 31, CX_RAY = 32
};

__device__ __forceinline__ void bre_pairs_warp(const GatherParams &P, uint2 pr, bool valid, float *a, ShadeShared &W,
                                               int lane) {
  const sf r(P.radius), rr2 = r * r;
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);
  const sf rrG = P.cfg.path_set ? sf(2.f) : sf(1.f);
  const float4 *rec = P.rays + (size_t)(valid ? pr.x : 0u) * GVPM_RAY_FLOAT4;
  BaseRay R;
  v3 baseContrib(0.f, 0.f, 0.f);
  sf recip(0.f), tBase(0.f), pdfCam(1.f);
  bool live = valid;
  uint32_t nTasks = 0;
  // ---- phase A ------------------------------------------------------------------------------------------------
  PhotonRec ph;
  v3 wi(0.f, 0.f, 0.f);
  sf Tshift(0.f);
  v3 zBase(0.f, 0.f, 0.f);
  if (live) {
    R = load_base_ray(rec);
    ph = load_photon_orig(P, pr.y);
    live = base_distance<false>(P, R, ph.p, pr.y, tBase, pdfCam);  // always true for an emitted pair
  }
  if (live) {
    wi = ph.wi;
    const MediumRec mBase = medium_eval(P, R.mint, tBase);
    const v3 contrib = (sigS * ph.flux) * phase_eval(P, wi, -R.d);
    baseContrib = (contrib * mBase.T) * R.eye;
    const sf norm = sf(P.kernel_vol) * pdfCam;
    recip = frcp(norm);
    acc_add(a, 0, (baseContrib * recip) * rrG);
    Tshift = medium_eval(P, sf(P.cfg.epsilon), tBase).T;
    zBase = R.o + tBase * R.d;
    const OccluderNear near = pair_occluders(P, ph.parent, ph.lBase);
    float *c = W.ctx[lane];
    c[CX_P] = ph.p.x.v; c[CX_P + 1] = ph.p.y.v; c[CX_P + 2] = ph.p.z.v;
    c[CX_PARENT] = ph.parent.x.v; c[CX_PARENT + 1] = ph.parent.y.v; c[CX_PARENT + 2] = ph.parent.z.v;
    c[CX_PN] = ph.pn.x.v; c[CX_PN + 1] = ph.pn.y.v; c[CX_PN + 2] = ph.pn.z.v;
    c[CX_PREFIX] = ph.prefix.x.v; c[CX_PREFIX + 1] = ph.prefix.y.v; c[CX_PREFIX + 2] = ph.prefix.z.v;
    c[CX_ALBEDO] = ph.albedo.x.v; c[CX_ALBEDO + 1] = ph.albedo.y.v; c[CX_ALBEDO + 2] = ph.albedo.z.v;
    c[CX_PARENTPDF] = ph.parentPdf.v; c[CX_EDGEPDF] = ph.edgePdf.v; c[CX_RRW] = ph.rrW.v;
    c[CX_PTYPE] = __int_as_float(ph.ptype);
    c[CX_WIW] = ph.wiW.x.v; c[CX_WIW + 1] = ph.wiW.y.v; c[CX_WIW + 2] = ph.wiW.z.v;
    c[CX_COSI] = ph.cosI.v; c[CX_NEDGE] = ph.nEdge.v;
    c[CX_NEARMASK] = __uint_as_float(near.mask); c[CX_NEARBOUND] = near.bound;
    c[CX_ZBASE] = zBase.x.v; c[CX_ZBASE + 1] = zBase.y.v; c[CX_ZBASE + 2] = zBase.z.v;
    c[CX_TBASE] = tBase.v; c[CX_PDFCAM] = pdfCam.v; c[CX_TSHIFT] = Tshift.v;
    c[CX_RAY] = __uint_as_float(pr.x);
  }
  // the offset records are requested one iteration ahead (the loop is rolled: their L1/L2 latency was exposed at
  // the top of every iteration)
  float4 n0 = ldg4(rec + 4), n1 = ldg4(rec + 5), n2 = ldg4(rec + 6);
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    bool reconnect = false;
    const float4 s0 = n0, s1 = n1, s2 = n2;
    if (k < 3) {
      n0 = ldg4(rec + 4 * (k + 2));
      n1 = ldg4(rec + 4 * (k + 2) + 1);
      n2 = ldg4(rec + 4 * (k + 2) + 2);
    }
    if (live) {
      sf weight(1.f);
      v3 S(0.f, 0.f, 0.f);
      if (__float_as_uint(s2.w) != 0u) {  // validVolumeEdge, shift_cameraPath.h:135-140
        const v3 ok(s0.x, s0.y, s0.z), dk(s1.x, s1.y, s1.z), eyeK(s2.x, s2.y, s2.z);
        const sf lenK(s0.w), sensor(s1.w);
        const v3 zShift = ok + tBase * dk;
        bool done = false;
        if (P.cfg.use_shift_null && P.cfg.kernel_3d) {  // :776-802
          sf ZPtoY = length_sq(zShift - ph.p);
          if (ZPtoY < rr2 && tBase < lenK) {
            sf dd = dot(ph.p - ok, dk);
            sf ds = length_sq((ok + dd * dk) - ph.p);
            sf pdfShift = chord_pdf(safe_sqrt(rr2 - ds));
            shift_null(P, ph.flux, wi, dk, eyeK, sensor, Tshift, pdfCam, pdfShift, S, weight);
            done = true;
          }
        }
        reconnect = !done && lenK >= tBase;  // :809-838
      }
      if (!reconnect) W.res[lane][k] = make_float4(S.x.v, S.y.v, S.z.v, weight.v);
    }
    const uint32_t m = __ballot_sync(0xffffffffu, reconnect);
    if (reconnect) W.tasks[nTasks + __popc(m & ((1u << lane) - 1u))] = (uint8_t)((lane << 2) | k);
    nTasks += __popc(m);
  }
  __syncwarp();
  // ---- phase B: one reconnection per lane, 32 at a time -------------------------------------------------------------
  for (uint32_t t0 = 0; t0 < nTasks; t0 += 32) {
    if (t0 + lane < nTasks) {
      const uint32_t task = W.tasks[t0 + lane];
      const int owner = task >> 2, k = task & 3;
      const float *c = W.ctx[owner];
      PhotonRec q;
      q.p = v3(c[CX_P], c[CX_P + 1], c[CX_P + 2]);
      q.parent = v3(c[CX_PARENT], c[CX_PARENT + 1], c[CX_PARENT + 2]);
      q.pn = v3(c[CX_PN], c[CX_PN + 1], c[CX_PN + 2]);
      q.prefix = v3(c[CX_PREFIX], c[CX_PREFIX + 1], c[CX_PREFIX + 2]);
      q.albedo = v3(c[CX_ALBEDO], c[CX_ALBEDO + 1], c[CX_ALBEDO + 2]);
      q.parentPdf = sf(c[CX_PARENTPDF]); q.edgePdf = sf(c[CX_EDGEPDF]); q.rrW = sf(c[CX_RRW]);
      q.ptype = __float_as_int(c[CX_PTYPE]);
      q.wiW = v3(c[CX_WIW], c[CX_WIW + 1], c[CX_WIW + 2]);
      q.cosI = sf(c[CX_COSI]); q.nEdge = sf(c[CX_NEDGE]);
      OccluderNear near;
      near.mask = __float_as_uint(c[CX_NEARMASK]); near.bound = c[CX_NEARBOUND];
      const v3 zB(c[CX_ZBASE], c[CX_ZBASE + 1], c[CX_ZBASE + 2]);
      const sf tB(c[CX_TBASE]), pC(c[CX_PDFCAM]), Ts(c[CX_TSHIFT]);
      const float4 *orec = P.rays + (size_t)__float_as_uint(c[CX_RAY]) * GVPM_RAY_FLOAT4;
      const float4 s0 = ldg4(orec + 4 * (k + 1)), s1 = ldg4(orec + 4 * (k + 1) + 1), s2 = ldg4(orec + 4 * (k + 1) + 2);
      const v3 ok(s0.x, s0.y, s0.z), dk(s1.x, s1.y, s1.z), eyeK(s2.x, s2.y, s2.z);
      const sf sensor(s1.w);
      const v3 zShift = ok + tB * dk;
      v3 dBase(0.f, 0.f, 0.f);
      if (!P.cfg.kernel_3d) {  // the 2-D kernel's coherent frames need the base direction
        const float4 b1 = ldg4(orec + 1);
        dBase = v3(b1.x, b1.y, b1.z);
      }
      const v3 offsetPos = get_shift_pos(P, rr2, q.p, zB, zShift, dBase, dk, !P.cfg.kernel_3d);
      sf pdfShift(1.f);
      if (P.cfg.kernel_3d) {
        sf dd = dot(offsetPos - ok, dk);
        sf ds = length_sq((ok + dd * dk) - offsetPos);
        pdfShift = chord_pdf(safe_sqrt(rr2 - ds));
      }
      sf weight(1.f);
      v3 S(0.f, 0.f, 0.f);
      shift_photon_diffuse(P, q, near, offsetPos, dk, eyeK, sensor, Ts, pC, pdfShift, S, weight);
      W.res[owner][k] = make_float4(S.x.v, S.y.v, S.z.v, weight.v);
    }
  }
  __syncwarp();
  // ---- phase C: fold the four offsets in k order ------------------------------------------------------------------------
  if (live) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float4 rs = W.res[lane][k];
      sf weight(rs.w);
      const v3 S(rs.x, rs.y, rs.z);
      if ((k == 1 && R.px == P.cfg.film_w - 1) || (k == 2 && R.py == P.cfg.film_h - 1)) weight = sf(1.f);
      const sf rw = rrG * weight;
      const v3 wB = (baseContrib * rw) * recip, wS = (S * rw) * recip;
      acc_add(a, 5 + k, wB);
      acc_add(a, 1 + k, wS);
    }
  }
  __syncwarp();
}

}  // namespace gvpm
