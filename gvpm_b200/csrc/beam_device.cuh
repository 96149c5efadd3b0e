// beam_device.cuh — device functions of the G-Beams gather: "beam3d" (EBeamBeam3D_Optimized) and "beam1d"
// (EBeamBeam1D with newShiftBeam, gvpm.cpp:96-98).
// Reference lines restated here:
//   PhotonBeam::rayIntersectInternal1D, getContrib          photonmapper/beams_struct.h:136-185,250-311
//   shift(), localMatrix(), getShiftPos1D                   gvpm/shift/shift_volume_beams.cpp:36-96
//   BeamKernelRecord::eval / null-shift ctor / kernelPDF   gvpm/shift/shift_volume_beams.h:39-143,195-283,298-336
//   cylinderIntersection                                    photonmapper/beams_3d_intersections.h:77-140
//   solveQuadraticDouble, coordinateSystem                  src/libcore/util.cpp:487-525,600-609
//   BeamGradRadianceQuery::operator(), getShiftPos          gvpm/shift/shift_volume_beams.cpp:98-353
//   shiftBeamDiffuse, shiftNull3D                           shift_volume_beams.cpp:410-539,748-786
//   diffuseReconnectionPhotonBeam                           gvpm/shift/operation/shift_diffuse.cpp:136-268
#pragma once
#include "bre_device.cuh"

namespace gvpm {

// Beam record: 8 float4 (128 B, SURVEY.md §8d)
//   B0 origin.xyz, length | B1 dir.xyz, meta | B2 flux.xyz, parent_pdf | B3 prefix.xyz, rr_weight
//   B4 parent_n.xyz, end.x | B5 albedo.xyz, end.y | B6 pred.xyz, end.z | B7 end_n.xyz, -
// meta: bits 0-1 parent type, 2-9 depth, 10 pathID parity, 11 end vertex on a surface
#define GVPM_BEAM_FLOAT4 8
struct BeamRec {
  v3 o, dir, end, flux, prefix, pn, albedo, pred, endN;
  sf length, parentPdf, rrW;
  int ptype;
  bool endOnSurface;
};
__device__ __forceinline__ BeamRec load_beam(const GatherParams &P, uint32_t bi) {
  const float4 *b = P.beams + (size_t)bi * GVPM_BEAM_FLOAT4;
  const float4 b0 = ldg4(b), b1 = ldg4(b + 1), b2 = ldg4(b + 2), b3 = ldg4(b + 3), b4 = ldg4(b + 4), b5 = ldg4(b + 5),
               b6 = ldg4(b + 6), b7 = ldg4(b + 7);
  BeamRec r;
  r.o = v3(b0.x, b0.y, b0.z); r.length = sf(b0.w);
  r.dir = v3(b1.x, b1.y, b1.z);
  const uint32_t meta = __float_as_uint(b1.w);
  r.ptype = meta & 3;
  r.endOnSurface = (meta >> 11) & 1;
  r.flux = v3(b2.x, b2.y, b2.z); r.parentPdf = sf(b2.w);
  r.prefix = v3(b3.x, b3.y, b3.z); r.rrW = sf(b3.w);
  r.pn = v3(b4.x, b4.y, b4.z);
  r.albedo = v3(b5.x, b5.y, b5.z);
  r.pred = v3(b6.x, b6.y, b6.z);
  r.end = v3(b4.w, b5.w, b6.w);
  r.endN = v3(b7.x, b7.y, b7.z);
  return r;
}

// coordinateSystem(a, b, c): Frame(n) constructor
__device__ __forceinline__ void coordinate_system(v3 a, v3 &b, v3 &c) {
  if (fabsf(a.x.v) > fabsf(a.y.v)) {
    const sf invLen = sf(1.f) / ssqrt(a.x * a.x + a.z * a.z);
    c = v3(a.z * invLen, sf(0.f), -a.x * invLen);
  } else {
    const sf invLen = sf(1.f) / ssqrt(a.y * a.y + a.z * a.z);
    c = v3(sf(0.f), a.z * invLen, -a.y * invLen);
  }
  b = cross(c, a);
}

__device__ __forceinline__ bool solve_quadratic_double(sd a, sd b, sd c, sd &x0, sd &x1) {
  if (a.v == 0.0) {
    if (b.v != 0.0) { x0 = x1 = sd(-c.v) / b; return true; }
    return false;
  }
  const sd discrim = b * b - sd(4.0) * a * c;
  if (discrim.v < 0.0) return false;
  const sd sqrtDiscrim = dsqrt(discrim);
  sd temp;
  if (b.v < 0.0) temp = sd(-0.5) * (b - sqrtDiscrim); else temp = sd(-0.5) * (b + sqrtDiscrim);
  x0 = temp / a;
  x1 = c / temp;
  if (x0.v > x1.v) { const sd t = x0; x0 = x1; x1 = t; }
  return true;
}

// cylinder = segment (co, cd, [0, cMaxt]) of radius `radius`; view ray = (vo, vd, maxt = vMaxt)
__device__ __noinline__ bool cylinder_intersection(v3 co, v3 cd, sf cMaxt, v3 vo, v3 vd, float vMaxt, sf radius,
                                                      double &tNearOut, double &tFarOut) {
  const v3 d1d2c = cross(vd, cd);
  const sf sinThetaSqr = dot(d1d2c, d1d2c);
  const sf ad = dot(co - vo, d1d2c);
  if ((ad * ad).v >= ((radius * radius) * sinThetaSqr).v) return false;
  v3 s, t;
  coordinate_system(cd, s, t);
  // worldToObject = (translate(co) * fromFrame(Frame(cd))).inverse() applied to the view ray: the 4x4 product
  // leaves the rotation rows untouched and puts -dot(axis, co) in the last column (matrix.h:744-756,
  // transform.cpp:28-45,216-227), so a point maps to dot(axis, p) + (-dot(axis, co)) (transform.h:108-125)
  const v3 lo(dot(vo, s) - dot(co, s), dot(vo, t) - dot(co, t), dot(vo, cd) - dot(co, cd)),
      ld(dot(vd, s), dot(vd, t), dot(vd, cd));
  const sd ox((double)lo.x.v), oy((double)lo.y.v), dx((double)ld.x.v), dy((double)ld.y.v);
  const sd A = dx * dx + dy * dy;
  const sd B = sd(2.0) * (dx * ox + dy * oy);
  const sd C = ox * ox + oy * oy - sd((double)(radius * radius).v);
  sd tNear, tFar;
  if (!solve_quadratic_double(A, B, C, tNear, tFar)) return false;
  if (tNear.v > (double)vMaxt || tFar.v < 0.0) return false;
  const sd loz((double)lo.z.v), ldz((double)ld.z.v);
  const sd zPosNear = loz + ldz * tNear;
  const sd zPosFar = loz + ldz * tFar;
  const double lMax = (double)cMaxt.v;
  tFarOut = tFar.v;
  if (zPosNear.v < 0.0) {
    if (zPosFar.v < 0.0) return false;
    const float th = (float)(tNear + (tFar - tNear) * zPosNear / (zPosNear - zPosFar)).v;
    tNearOut = (double)th;
    return true;
  } else if (zPosNear.v >= 0.0 && zPosNear.v < lMax) {
    tNearOut = tNear.v;
    return true;
  } else if (zPosNear.v > lMax) {
    if (zPosFar.v > lMax) return false;
    const float th = (float)(tNear + (tFar - tNear) * (zPosNear - sd(lMax)) / (zPosNear - zPosFar)).v;
    tNearOut = (double)th;
    return true;
  }
  return false;
}

// 1.0 / std::max(x, 0.0001) in double
__device__ __forceinline__ sd inv_max_double(sd x) { return sd(1.0) / sd(fmax(x.v, 0.0001)); }

// the two uniforms per (camera ray, beam) that replace sampler->next1D() (DESIGN.md §6)
__device__ __forceinline__ float beam_uniform(const GatherParams &P, const BaseRay &R, uint32_t beamIndex,
                                              uint32_t dim) {
  uint32_t h = hash32(P.cfg.rng_seed ^ 0x9E3779B9u);
  h = hash32(h ^ (uint32_t)R.px);
  h = hash32(h ^ ((uint32_t)R.py * 0x85EBCA6Bu));
  h = hash32(h ^ ((uint32_t)R.edgeId * 0xC2B2AE35u));
  h = hash32(h ^ beamIndex);
  h = hash32(h ^ (dim * 0x27D4EB2Fu));
  return (float)(h >> 8) * (1.0f / 16777216.0f);
}

struct BeamKernelRec {
  sf v, w, pdfKernel, pdfEdgeFailure, weightKernel, u;
  v3 contrib;
  bool valid;
  __device__ sf pdf() const { return pdfEdgeFailure * pdfKernel; }
};

__device__ __forceinline__ bool is_zero(v3 c) { return c.x.v == 0.f && c.y.v == 0.f && c.z.v == 0.f; }

// second half of BeamKernelRecord::eval / the null ctor: sample (or reuse) the camera distance inside
// the kernel sphere around beam(v); returns false when the record is invalid
__device__ __forceinline__ bool beam_kernel_camera(const GatherParams &P, const BeamRec &beam, v3 camO, v3 camD,
                                                   sf camMint, sf camMaxt, sf v, bool sampleW, sf xi2, sf wIn,
                                                   sf &w, sf &pdfKernel) {
  const sf r(P.radius);
  if (v.v < 0.f || v > beam.length) return false;
  const v3 kernelCentroid = beam.o + beam.dir * v;
  const sf distToProj = dot(kernelCentroid - camO, camD);
  const sf distSqr = length_sq((camO + distToProj * camD) - kernelCentroid);
  const sf radSqr = r * r;
  if (distSqr >= radSqr) return false;
  const sf deltaT = safe_sqrt(radSqr - distSqr);
  w = sampleW ? distToProj - deltaT + sf(2.f) * deltaT * xi2 : wIn;
  pdfKernel = sf((float)(sd((double)pdfKernel.v) * inv_max_double(sd(2.0) * sd((double)deltaT.v))).v);
  if (w < camMint || w > camMaxt) return false;
  return true;
}

// BeamKernelRecord::eval for the whole beam; tNear is returned for the sub-beam ownership rule
__device__ __forceinline__ BeamKernelRec beam_kernel_eval(const GatherParams &P, const BeamRec &beam,
                                                          const BaseRay &R, uint32_t beamIndex, double &tNearBeam) {
  BeamKernelRec k;
  k.valid = false;
  k.contrib = v3(0.f, 0.f, 0.f);
  k.v = k.w = k.pdfKernel = k.pdfEdgeFailure = k.weightKernel = k.u = sf(0.f);
  const sf r(P.radius);
  const v3 camStart = R.o + R.mint * R.d;
  double tFarBeam;
  if (!cylinder_intersection(camStart, R.d, R.maxt - R.mint, beam.o, beam.dir, beam.length.v, r, tNearBeam, tFarBeam))
    return k;
  if (tNearBeam < 0.0) {
  } else if (tNearBeam > 0.0 && tNearBeam < (double)beam.length.v) {
  } else {
    return k;
  }
  const sf xi1(beam_uniform(P, R, beamIndex, 0)), xi2(beam_uniform(P, R, beamIndex, 1));
  const sd span = sd(tFarBeam) - sd(tNearBeam);
  k.v = sf((float)(sd(tNearBeam) + span * sd((double)xi1.v)).v);
  k.pdfKernel = sf((float)inv_max_double(span).v);
  if (!beam_kernel_camera(P, beam, R.o, R.d, R.mint, R.maxt, k.v, true, xi2, sf(0.f), k.w, k.pdfKernel)) return k;
  const MediumRec mRecBeam = medium_eval(P, sf(0.f), k.v), mRecCamera = medium_eval(P, sf(0.f), k.w);
  const sf phaseTerm = phase_eval(P, -beam.dir, -R.d);
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);
  k.contrib = ((((beam.flux * mRecBeam.T) * sigS) * mRecCamera.T) * phaseTerm) / k.pdfKernel;
  k.weightKernel = sf(P.weight_kernel);
  if (!P.cfg.long_beams) {
    k.contrib = k.contrib / mRecBeam.pdfFailure;
    k.pdfEdgeFailure = mRecBeam.pdfFailure;
  } else {
    k.pdfEdgeFailure = sf(1.f);
  }
  k.valid = !is_zero(k.contrib);
  return k;
}

// PhotonBeam::rayIntersectInternal1D: closest approach of the camera line and the beam line, strictly rounded fp32
// in the reference's operation order (this decides the (ray, beam) index set of the 1-D kernel)
__device__ __forceinline__ bool beam_intersect_1d(v3 p1, v3 bdir, sf blen, sf radius, v3 ro, v3 rd, sf rmint, sf rmaxt,
                                                  sf tminBeam, sf tmaxBeam, sf &u, sf &v, sf &w, sf &sinTheta) {
  const v3 d1d2c = cross(rd, bdir);
  const sf sinThetaSqr = dot(d1d2c, d1d2c);
  const sf ad = dot(p1 - ro, d1d2c);
  if ((ad * ad).v >= ((radius * radius) * sinThetaSqr).v) return false;
  const sf d1d2 = dot(rd, bdir);
  const sf d1d2Sqr = d1d2 * d1d2;
  const sf d1d2SqrMinus1 = d1d2Sqr - sf(1.0f);
  if (d1d2SqrMinus1.v < 1e-5f && d1d2SqrMinus1.v > -1e-5f) return false;
  const sf d1O1 = dot(rd, ro);
  const sf d1O2 = dot(rd, p1);
  w = (d1O1 - d1O2 - d1d2 * (dot(bdir, ro) - dot(bdir, p1))) / d1d2SqrMinus1;
  if (w.v <= rmint.v || w.v >= rmaxt.v) return false;
  v = (w + d1O1 - d1O2) / d1d2;
  if (v.v <= 0.f || v.v >= blen.v || isnan(v.v)) return false;
  if (tminBeam.v >= v.v || tmaxBeam.v < v.v) return false;
  const sf sinThetaConst = ssqrt(sinThetaSqr);
  u = sf(fabsf(ad.v)) / sinThetaConst;
  sinTheta = sinThetaConst;
  return true;
}

// BeamKernelRecord::eval, EBeamBeam1D branch + PhotonBeam::getContrib, for the whole beam (tmin = 0, tmax = length)
__device__ __forceinline__ BeamKernelRec beam_kernel_eval_1d(const GatherParams &P, const BeamRec &beam,
                                                             const BaseRay &R) {
  BeamKernelRec k;
  k.valid = false;
  k.contrib = v3(0.f, 0.f, 0.f);
  k.v = k.w = k.pdfKernel = k.pdfEdgeFailure = k.weightKernel = k.u = sf(0.f);
  if (!beam_intersect_1d(beam.o, beam.dir, beam.length, sf(P.radius), R.o, R.d, R.mint, R.maxt, sf(0.f), beam.length,
                         k.u, k.v, k.w, k.pdfKernel))
    return k;
  const MediumRec mRecCamera = medium_eval(P, sf(0.f), k.w), mRec = medium_eval(P, sf(0.f), k.v);
  k.weightKernel = sf(P.weight_kernel);
  const sf phaseTerm = phase_eval(P, -beam.dir, -R.d);
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);
  v3 beamContrib = (((mRec.T * mRecCamera.T) * sigS) * beam.flux) * phaseTerm;
  if (!P.cfg.long_beams) {
    k.pdfEdgeFailure = mRec.pdfFailure;
    if (mRec.pdfFailure.v == 0.f && mRec.T.v != 0.f) return k;
    beamContrib = beamContrib / mRec.pdfFailure;
  } else {
    k.pdfEdgeFailure = sf(1.f);
  }
  k.contrib = beamContrib;
  if (!is_zero(k.contrib)) k.contrib = k.contrib / k.pdfKernel;
  k.valid = !is_zero(k.contrib);
  return k;
}

// shift() + localMatrix(): the point at distance u from the camera ray (at camera distance w) in the plane through
// the beam origin a.  Radiance-only arithmetic (asinf / cosf / sinf within a few ulp of libm).
__device__ __forceinline__ v3 beam_shift_1d(v3 ro, v3 rd, v3 a, sf u, sf w, bool flip) {
  const sf d = dot(a - ro, rd);
  const v3 tD = ro + d * rd;
  const v3 s = normalize(a - tD);
  const v3 t = cross(rd, s);
  const sf localAy = dot(a - tD, s);
  const float q = fminf(1.f, fmaxf(-1.f, (u / sf(fabsf(localAy.v))).v));
  float phi = (float)(1.57079632679489661923 - (double)asinf(q));
  if (flip) phi = -phi;
  const sf ly = u * sf(cosf(phi)), lz = u * sf(sinf(phi));
  const v3 worldU = (rd * sf(0.f) + s * ly) + t * lz;
  return (ro + w * rd) + worldU;
}
// BeamGradRadianceQuery::getShiftPos1D
__device__ __forceinline__ v3 beam_shift_pos_1d(const BaseRay &R, v3 ok, v3 dk, v3 a, v3 bBeamDir, sf w, sf u) {
  const v3 back = normalize(beam_shift_1d(R.o, R.d, a, u, w, false) - a);
  const bool flipAngle = length_sq(back - bBeamDir).v > 0.001f;
  return beam_shift_1d(ok, dk, a, u, w, flipAngle);
}

// BeamKernelRecord(ori, medium, beam, cameraRay): the null-shift re-evaluation on the offset ray
__device__ __forceinline__ BeamKernelRec beam_kernel_null(const GatherParams &P, const BeamKernelRec &ori,
                                                          const BeamRec &beam, v3 camO, v3 camD, sf camMint,
                                                          sf camMaxt) {
  BeamKernelRec k;
  k.valid = false;
  k.contrib = v3(0.f, 0.f, 0.f);
  k.v = k.w = k.pdfKernel = k.pdfEdgeFailure = k.weightKernel = k.u = sf(0.f);
  const sf r(P.radius);
  const v3 camStart = camO + camMint * camD;
  double tNearBeam, tFarBeam;
  if (!cylinder_intersection(camStart, camD, camMaxt - camMint, beam.o, beam.dir, beam.length.v, r, tNearBeam, tFarBeam))
    return k;
  k.v = ori.v;
  k.pdfKernel = sf((float)inv_max_double(sd(tFarBeam) - sd(tNearBeam)).v);
  if (!beam_kernel_camera(P, beam, camO, camD, camMint, camMaxt, k.v, false, sf(0.f), ori.w, k.w, k.pdfKernel)) return k;
  k.contrib = ori.contrib * (ori.pdfKernel / k.pdfKernel);
  k.weightKernel = ori.weightKernel;
  k.pdfEdgeFailure = P.cfg.long_beams ? sf(1.f) : ori.pdfEdgeFailure;
  k.valid = !is_zero(k.contrib);
  return k;
}

// BeamKernelRecord::kernelPDF (3-D optimized): infinite beam from orgBeam along dBeam
template <bool K1D>
__device__ __forceinline__ sf beam_kernel_pdf(const GatherParams &P, v3 camO, v3 camD, sf camMaxt, v3 orgBeam,
                                              v3 dBeam, sf newDLength) {
  if (K1D) return ssqrt(length_sq(cross(camD, dBeam)));
  const sf r(P.radius);
  double tNearBeam, tFarBeam;
  if (!cylinder_intersection(camO, camD, camMaxt, orgBeam, dBeam, INFINITY, r, tNearBeam, tFarBeam)) return sf(0.f);
  sf pdfK((float)inv_max_double(sd(tFarBeam) - sd(tNearBeam)).v);
  const v3 kernelCentroid = orgBeam + dBeam * newDLength;
  const sf distToProj = dot(kernelCentroid - camO, camD);
  const sf distSqr = length_sq((camO + distToProj * camD) - kernelCentroid);
  const sf radSqr = r * r;
  if (!(distSqr < radSqr)) return sf(0.f);
  const sf deltaT = safe_sqrt(radSqr - distSqr);
  return sf((float)(sd((double)pdfK.v) * inv_max_double(sd(2.0) * sd((double)deltaT.v))).v);
}

// BeamGradRadianceQuery::getShiftPos (coherent = true)
__device__ __forceinline__ v3 beam_shift_pos(const GatherParams &P, const BaseRay &R, v3 ok, v3 dk, sf w, v3 u,
                                             sf newW) {
  const sf r(P.radius);
  const v3 sAt = ok + newW * dk;
  v3 bs, bt, ns, nt;
  coherent_frame(R.d, bs, bt);
  coherent_frame(dk, ns, nt);
  const v3 local(dot(u, bs), dot(u, bt), dot(u, R.d));
  v3 newPos = sAt + ((ns * local.x + nt * local.y) + dk * local.z);
  if (P.cfg.use_shift_null) {
    const v3 bCamW = R.o + w * R.d;
    const sf offDistSqr = length_sq(bCamW - newPos);
    if (offDistSqr < r * r) {
      v3 dShift = sAt - bCamW;
      dShift = dShift / length(dShift);
      const sf cosD = dot(dShift, -(newPos - sAt));
      newPos = newPos + (dShift * cosD) * sf(2.f);
    }
  }
  return newPos;
}

// shiftBeam -> shiftBeamDiffuse + diffuseReconnectionPhotonBeam; S / weight keep (0, 1) on failure
template <bool K1D, bool BVH>
__device__ __forceinline__ void shift_beam_diffuse(const GatherParams &P, const BeamRec &beam, v3 ok, v3 dk, sf lenK,
                                                   v3 eyeK, sf sensor, sf shiftW, const BeamKernelRec &kRec,
                                                   v3 newPos, v3 &S, sf &weight) {
  if (shiftW > lenK) { weight = sf(1.f); return; }
  if (beam.ptype == GVPM_PARENT_OTHER) return;
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);
  v3 newPBDir = newPos - beam.o;
  const sf newPBDist = length(newPBDir);
  newPBDir = newPBDir / newPBDist;
  if (occluded<BVH>(P, beam.o, newPBDir, sf(P.cfg.epsilon), newPBDist)) { weight = sf(1.f); return; }
  const v3 basePos = beam.o + beam.dir * kRec.v;
  const sf pdfKernelAndDist = kRec.pdf();
  v3 thr(1.f, 1.f, 1.f);
  sf pdfValueSA(0.f), sPdf(0.f);
  bool failed = false;
  if (beam.ptype == GVPM_PARENT_SURFACE) {
    const v3 wiW = normalize(beam.pred - beam.o);
    const sf cosI = dot(beam.pn, wiW), cosO = dot(beam.pn, newPBDir);
    if (cosI.v <= 0.f || cosO.v <= 0.f) {
      thr = v3(0.f, 0.f, 0.f);
    } else {
      thr = thr * (beam.albedo * (sf(GVPM_INV_PI) * cosO));
      pdfValueSA = sf(GVPM_INV_PI) * cosO;
    }
    if ((cosI * cosI).v <= 0.f || (cosO * cosO).v <= 0.f) failed = true;
  } else if (beam.ptype == GVPM_PARENT_MEDIUM) {
    const v3 pWi = normalize(beam.pred - beam.o);
    const sf phv = phase_eval(P, pWi, newPBDir);
    thr = thr * (sigS * phv);
    pdfValueSA = phv;
  } else {
    sf dp = dot(newPBDir, beam.pn);
    if (dp.v < 0.f) dp = sf(0.f);
    const sf e = sf(GVPM_INV_PI) * dp;
    thr = thr * v3(e, e, e);
    pdfValueSA = e;
  }
  const sf lenSqBase = length_sq(beam.o - beam.end), lenSqKernel = length_sq(beam.o - basePos);
  const sf absCosEnd(fabsf(dot(beam.endN, beam.dir).v));
  if (!failed) {
    const sf GOpNew = frcp(newPBDist * newPBDist);   // radiometric from here on: fast reciprocals (2 ulp), as in the BRE shading
    sPdf = pdfValueSA * GOpNew;
    thr = thr * GOpNew;
    sf pdfBasePos = beam.parentPdf * lenSqBase;
    if (beam.endOnSurface) pdfBasePos = fdiv(pdfBasePos, absCosEnd);
    const sf GOpBase = frcp(lenSqKernel);
    pdfBasePos = pdfBasePos * GOpBase;
    if (pdfBasePos.v == 0.f) {
      sPdf = sf(0.f);
    } else {
      thr = thr * frcp(pdfBasePos);
      thr = thr * beam.rrW;
      const MediumRec m = medium_eval(P, sf(0.f), newPBDist);
      if (!P.cfg.long_beams) sPdf = sPdf * m.pdfFailure;
      thr = thr * (m.T * frcp(pdfKernelAndDist));
    }
  }
  if (sPdf.v == 0.f) { weight = sf(1.f); return; }
  const sf shiftKernelPDF = beam_kernel_pdf<K1D>(P, ok, dk, lenK, beam.o, newPBDir, newPBDist);
  if (shiftKernelPDF.v == 0.f) { weight = sf(1.f); return; }
  v3 shiftPhotonWeight = beam.prefix * thr;
  const MediumRec mRecShift = medium_eval(P, sf(0.f), shiftW);
  const sf phaseTerm = phase_eval(P, -newPBDir, -dk);
  shiftPhotonWeight = shiftPhotonWeight * ((sigS * mRecShift.T) * phaseTerm);
  S = shiftPhotonWeight * eyeK;
  weight = sf(0.5f);
  if (P.cfg.use_mis) {
    sf basePdf = beam.parentPdf;
    basePdf = basePdf * lenSqBase;
    if (beam.endOnSurface) basePdf = fdiv(basePdf, absCosEnd);
    basePdf = fdiv(basePdf, lenSqKernel);
    basePdf = basePdf * pdfKernelAndDist;
    sf offsetPdf = shiftKernelPDF;
    offsetPdf = offsetPdf * sPdf;
    if (offsetPdf.v == 0.f || basePdf.v == 0.f) { weight = sf(1.f); return; }
    const sf q = fdiv(sensor * offsetPdf, basePdf);
    weight = P.cfg.power_heuristic ? frcp(sf(1.f) + q * q) : frcp(sf(1.f) + q);
  }
}

// BeamGradRadianceQuery::operator() for one (ray, beam) pair whose kernel record is valid and which
// passed the filters
template <bool K1D, bool BVH>
__device__ __forceinline__ void beam_functor(const GatherParams &P, const float4 *__restrict__ rec, const BaseRay &R,
                                             const BeamRec &beam, const BeamKernelRec &kRec, float *a) {
  const sf r(P.radius);
  const sf rrG = P.cfg.path_set ? sf(2.f) : sf(1.f);
  const v3 baseContrib = (R.eye * kRec.contrib) * kRec.weightKernel;
  acc_add(a, 0, baseContrib * rrG);
  float Sx[4], Sy[4], Sz[4], Wk[4];
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    const float4 s0 = ldg4(rec + 4 * (k + 1)), s1 = ldg4(rec + 4 * (k + 1) + 1), s2 = ldg4(rec + 4 * (k + 1) + 2);
    sf weight(1.f);
    v3 S(0.f, 0.f, 0.f);
    if (__float_as_uint(s2.w) != 0u) {
      const v3 ok(s0.x, s0.y, s0.z), dk(s1.x, s1.y, s1.z), eyeK(s2.x, s2.y, s2.z);
      const sf lenK(s0.w), sensor(s1.w), shiftW = kRec.w;
      bool alreadyShift = false;
      if (P.cfg.use_shift_null && !K1D) {   // "Ignored in case of Beam 1D kernel", :264-265
        const v3 kernelPos = beam.o + beam.dir * kRec.v;
        const sf ZPtoY = length_sq((ok + shiftW * dk) - kernelPos);
        if (ZPtoY < r * r && kRec.w <= lenK) {
          BeamKernelRec kS = beam_kernel_null(P, kRec, beam, ok, dk, sf(P.cfg.epsilon), lenK);
          if (kS.valid) {
            // shiftNull3D
            kS.contrib = kS.contrib * fdiv(kS.pdf(), kRec.pdf());
            S = kS.contrib * eyeK;
            weight = sf(0.5f);
            if (P.cfg.use_mis) {
              const sf basePdf = kRec.pdf(), offsetPdf = kS.pdf();
              if (offsetPdf.v == 0.f || basePdf.v == 0.f) {
                weight = sf(1.f);
              } else {
                const sf q = sensor * fdiv(offsetPdf, basePdf);
                weight = P.cfg.power_heuristic ? frcp(sf(1.f) + q * q) : frcp(sf(1.f) + q);
              }
            }
            alreadyShift = true;
          }
        }
      }
      if (K1D && !alreadyShift && kRec.w <= lenK) {   // newShiftBeam, :311-317
        const v3 offsetPos = beam_shift_pos_1d(R, ok, dk, beam.o, beam.dir, kRec.w, kRec.u);
        shift_beam_diffuse<K1D, BVH>(P, beam, ok, dk, lenK, eyeK, sensor, shiftW, kRec, offsetPos, S, weight);
      } else if (!alreadyShift && kRec.w <= lenK) {
        const sf dd = dot(beam.o - ok, dk);
        const sf minDistSqr = length_sq(beam.o - (ok + dd * dk));
        if (minDistSqr.v > 0.f) {
          const v3 u = (beam.o + beam.dir * kRec.v) - (R.o + kRec.w * R.d);
          const v3 offsetPos = beam_shift_pos(P, R, ok, dk, kRec.w, u, shiftW);
          shift_beam_diffuse<K1D, BVH>(P, beam, ok, dk, lenK, eyeK, sensor, shiftW, kRec, offsetPos, S, weight);
        } else {
          weight = sf(1.f);
        }
      }
    }
    S = S * kRec.weightKernel;
    if ((k == 1 && R.px == P.cfg.film_w - 1) || (k == 2 && R.py == P.cfg.film_h - 1)) weight = sf(1.f);
    Sx[k] = S.x.v; Sy[k] = S.y.v; Sz[k] = S.z.v; Wk[k] = weight.v;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const sf wk(Wk[k]);
    acc_add(a, 1 + k, (v3(Sx[k], Sy[k], Sz[k]) * wk) * rrG);
    acc_add(a, 5 + k, (baseContrib * wk) * rrG);
  }
}

// ---- sppm primal photon beams: BeamRadianceQuery::operator(), photonmapper/beams.h:29-223 ---------------------------
// One (camera beam, sub-beam) visit for technique P.sppm_beam_technique (gvpm_beam_technique).  sb = sub-beam record
// (t1, t2, beam index, flags: bit 0 first, bit 1 last, bits 2.. ordinal).  Every value that decides acceptance is
// strictly rounded in the reference's operation order.  Returns 0 = rejected, 1 = accepted; Li is the
// contribution (without beam.weight) when accepted.
__device__ __forceinline__ int sppm_beam_functor(const GatherParams &P, const BaseRay &R, const BeamRec &beam,
                                                 uint32_t beamIndex, float4 sb, v3 &Li) {
  const uint32_t flags = __float_as_uint(sb.w);
  const bool first = flags & 1u, last = flags & 2u;
  const sf tmin(sb.x);
  sf tmax(sb.y);
  if (tmax > beam.length) tmax = beam.length;                                            // :30-32
  const sf r(P.radius), eps(P.cfg.epsilon);
  const v3 sigS(P.sigma_s[0], P.sigma_s[1], P.sigma_s[2]);
  const int technique = P.sppm_beam_technique;
  Li = v3(0.f, 0.f, 0.f);
  if (technique == GVPM_BEAM_1D) {                                                       // :41-68
    sf u, v, w, sinTheta;
    if (!beam_intersect_1d(beam.o, beam.dir, beam.length, r, R.o, R.d, R.mint, R.maxt, first ? sf(0.f) : tmin,
                           last ? beam.length : tmax, u, v, w, sinTheta))
      return 0;
    if (r <= u) return 0;
    const MediumRec mRecCamera = medium_eval(P, eps, w), mRec = medium_eval(P, sf(0.f), v);
    const sf weightKernel = sf(0.5f) / r;
    v3 beamContrib = (((mRec.T * mRecCamera.T) * sigS) * beam.flux) * phase_eval(P, -beam.dir, -R.d);
    if (!P.cfg.long_beams) {                                                            // getContrib, beams_struct.h:157-172
      if (mRec.pdfFailure.v == 0.f && mRec.T.v != 0.f) return 1;
      beamContrib = beamContrib / mRec.pdfFailure;
    }
    Li = (beamContrib * weightKernel) / sinTheta;
    return 1;
  }
  sf beamSegmentRand, cameraSegmentRand, invPDF;
  const sf radSqr = r * r;
  if (technique == GVPM_BEAM_3D_NAIVE) {                                                 // :77-102
    const uint32_t k = flags >> 2;
    const sf xi1(beam_uniform(P, R, beamIndex, 2u + 2u * k)), xi2(beam_uniform(P, R, beamIndex, 3u + 2u * k));
    beamSegmentRand = tmin + (tmax - tmin) * xi1;
    invPDF = tmax - tmin;
    const v3 kernelCentroid = beam.o + beam.dir * beamSegmentRand;
    const sf distToProj = dot(kernelCentroid - R.o, R.d);
    const sf distSqr = length_sq((R.o + distToProj * R.d) - kernelCentroid);
    if (distSqr >= radSqr) return 0;
    const sf deltaT = safe_sqrt(radSqr - distSqr);
    cameraSegmentRand = (distToProj - deltaT) + sf(2.f) * deltaT * xi2;
    invPDF = sf((float)(sd((double)invPDF.v) * sd(fmax((sd(2.0) * sd((double)deltaT.v)).v, 0.0001))).v);
    if (cameraSegmentRand < R.mint || cameraSegmentRand > R.maxt) return 0;              // DESIGN.md §6
  } else {
    const sf xi1(beam_uniform(P, R, beamIndex, 0)), xi2(beam_uniform(P, R, beamIndex, 1));
    const v3 camStart = R.o + R.mint * R.d;                                              // _cam, :106-107
    const sf camLen = R.maxt - R.mint;
    double tNearBeam, tFarBeam;
    if (!cylinder_intersection(camStart, R.d, camLen, beam.o, beam.dir, beam.length.v, r, tNearBeam, tFarBeam)) return 0;
    if (!((first || tNearBeam >= (double)tmin.v) && (last || tNearBeam < (double)tmax.v))) return 0;   // :122-128
    if (!(tNearBeam < 0.0 || (tNearBeam > 0.0 && tNearBeam < (double)beam.length.v))) return 0;
    const sd span = sd(tFarBeam) - sd(tNearBeam);
    beamSegmentRand = sf((float)(sd(tNearBeam) + span * sd((double)xi1.v)).v);
    invPDF = sf((float)fmax(span.v, 0.0001));
    if (beamSegmentRand.v < 0.f || beamSegmentRand > beam.length) return 0;
    if (technique == GVPM_BEAM_3D_EGSR) {                                                // :138-150
      double tNearCam, tFarCam;
      if (!cylinder_intersection(beam.o, beam.dir, beam.length, camStart, R.d, camLen.v, r, tNearCam, tFarCam)) return 0;
      const sd spanCam = sd(tFarCam) - sd(tNearCam);
      cameraSegmentRand = sf((float)(sd(tNearCam) + spanCam * sd((double)xi2.v)).v);
      invPDF = sf((float)(sd((double)invPDF.v) * sd(fmax(spanCam.v, 0.0001))).v);
    } else {                                                                             // :151-170
      const v3 kernelCentroid = beam.o + beam.dir * beamSegmentRand;
      const sf distToProj = dot(kernelCentroid - R.o, R.d);
      const sf distSqr = length_sq((R.o + distToProj * R.d) - kernelCentroid);
      if (distSqr >= radSqr) return 0;
      const sf deltaT = safe_sqrt(radSqr - distSqr);
      cameraSegmentRand = distToProj - deltaT + sf(2.f) * deltaT * xi2;
      invPDF = sf((float)(sd((double)invPDF.v) * sd(fmax((sd(2.0) * sd((double)deltaT.v)).v, 0.0001))).v);
    }
    if (cameraSegmentRand < R.mint || cameraSegmentRand > R.maxt) return 0;              // :173-175
    if (technique == GVPM_BEAM_3D_EGSR) {                                                // :178-187
      const v3 kernelCentroid = beam.o + beam.dir * beamSegmentRand;
      const sf distSqr = length_sq((R.o + cameraSegmentRand * R.d) - kernelCentroid);
      if (distSqr >= radSqr) return 0;
    }
  }
  const MediumRec mRecBeam = medium_eval(P, sf(0.f), beamSegmentRand), mRecCamera = medium_eval(P, eps, cameraSegmentRand);
  const sf phaseTerm = phase_eval(P, -beam.dir, -R.d);
  v3 beamContrib = ((((beam.flux * mRecBeam.T) * sigS) * mRecCamera.T) * phaseTerm) * (invPDF / sf(P.kernel_vol));
  if (!P.cfg.long_beams) beamContrib = beamContrib / mRecBeam.pdfFailure;                // :213-217
  Li = beamContrib;
  return 1;
}

}  // namespace gvpm
