// prims_ref.cpp — TEST INFRASTRUCTURE.  CPU restatement of gvpm_trace_beams and gvpm_planes_from_beams
// (include/gvpm_b200.h), the checker the device beams and planes are compared with BIT FOR BIT
// (tests/test_gpu_trace_prims.py).  It reuses, unchanged, the scene, frame, sampling and polynomial log / exp / sin / cos
// routines of the photon tracer's restatement (oracle/gvpm_oracle_trace.cpp, included below), and restates its walk with
// the beam rule of LTBeamMap::tryAppendLT (gvpm/gvpm_beams.h:54-84) as the one difference.  tests/test_oracle_trace_prims.py
// pins the beams to that oracle's photons.  Compiled with -ffp-contract=off: every operation is rounded on its own.
#include "../oracle/gvpm_oracle_trace.cpp"

namespace {

struct BeamSink {
  gvpm_beam_soa *out;
  size_t cap, filled;
  uint32_t pathId;
  bool storedAny;
};

// one light path (the walk of gvpm_oracle_trace.cpp); beams beyond the capacity are counted but not stored
uint32_t walkBeams(const gvpm_box_scene &S, const gvpm_medium &med, uint64_t seed, uint64_t pathIdx, int maxDepth,
                   int rrDepth, int minDepth, BeamSink &sink) {
  Rng rng(seed, pathIdx);
  const float sigS = med.sigma_s[0], sigT = med.sigma_s[0] + med.sigma_a[0];
  float u1 = rng.uniform(), u2 = rng.uniform();
  V curPos{S.light_x0 + (S.light_x1 - S.light_x0) * u1, S.light_y, S.light_z0 + (S.light_z1 - S.light_z0) * u2};
  V curN{0, -1, 0}, curAlbedo{0, 0, 0}, curWeight{1, 1, 1}, prevPos{1, 1, 1};
  int curType = GVPM_PARENT_EMITTER, ci = 1;
  float curRr = 1.f;
  u1 = rng.uniform();
  u2 = rng.uniform();
  V dir = toWorld(curN, cosineHemisphere(u1, u2));
  float pdfOmega = std::max(0.f, dot(dir, curN)) * INV_PI;
  V thr{S.light_power, S.light_power, S.light_power};
  const int firstBeam = std::max(1, minDepth);
  uint32_t appended = 0;
  for (;;) {
    const Hit h = intersect(S, curPos, dir);
    const float t = -pmLog(1.0f - rng.uniform()) / sigT;
    const bool inMedium = t < h.t;
    const float L = inMedium ? t : h.t;
    if (!inMedium && h.escaped) break;
    const float T = pmExp(-sigT * L);
    const float edgePdf = inMedium ? sigT * T : T, ew = T / edgePdf;
    const V nvPos = curPos + dir * L;
    float pdfArea;
    int nvType;
    V nvN{0, 0, 0}, nvAlbedo{0, 0, 0}, nvWeight;
    if (inMedium) {
      nvType = GVPM_PARENT_MEDIUM;
      nvWeight = {sigS, sigS, sigS};
      pdfArea = pdfOmega / (L * L);
    } else {
      nvType = GVPM_PARENT_SURFACE;
      nvN = h.n;
      nvAlbedo = h.albedo;
      nvWeight = h.albedo;
      pdfArea = (pdfOmega * std::fabs(dot(h.n, dir))) / (L * L);
    }
    const V prefix = thr;
    const V step{(curWeight.x * curRr) * ew, (curWeight.y * curRr) * ew, (curWeight.z * curRr) * ew};
    const V flux = mul(thr, step);
    const int ni = ci + 1;
    if (ci >= firstBeam) {   // edge ci -> ci + 1; flux without the edge's transmittance (gvpm_beams.h:29-35)
      if (sink.filled < sink.cap) {
        const size_t i = sink.filled++;
        const gvpm_beam_soa &o = *sink.out;
        put(o.origin, i, curPos); put(o.end, i, nvPos);
        put(o.flux, i, V{(thr.x * curWeight.x) * curRr, (thr.y * curWeight.y) * curRr, (thr.z * curWeight.z) * curRr});
        put(o.prefix_flux, i, prefix); put(o.parent_n, i, curN); put(o.parent_albedo, i, curAlbedo);
        put(o.pred_pos, i, ci >= 2 ? prevPos : V{1, 1, 1}); put(o.end_n, i, nvN);
        const_cast<float *>(o.parent_pdf)[i] = pdfArea;
        const_cast<float *>(o.rr_weight)[i] = curRr;
        const_cast<uint8_t *>(o.parent_type)[i] = (uint8_t)curType;
        const_cast<uint8_t *>(o.end_on_surface)[i] = inMedium ? 0 : 1;
        const_cast<uint8_t *>(o.depth)[i] = (uint8_t)ci;
        const_cast<uint32_t *>(o.path_id)[i] = sink.pathId;
        sink.storedAny = true;
      }
      ++appended;
    }
    thr = flux;
    prevPos = curPos;
    curPos = nvPos; curN = nvN; curAlbedo = nvAlbedo; curWeight = nvWeight; curType = nvType; curRr = 1.f;
    ci = ni;
    if (ci >= maxDepth) break;
    if (ci - 1 >= rrDepth) {
      const float m = std::max(thr.x * curWeight.x, std::max(thr.y * curWeight.y, thr.z * curWeight.z));
      const float q = std::min(m, 0.95f);
      if (!(rng.uniform() < q)) break;
      curRr = 1.0f / q;
    }
    const V inDir = dir;
    if (curType == GVPM_PARENT_MEDIUM) {
      if (med.phase_type == GVPM_PHASE_HG && std::fabs(med.hg_g) > 1e-4f) {
        const float g = med.hg_g, u = rng.uniform();
        const float sq = (1.f - g * g) / ((1.f - g) + (2.f * g) * u);
        const float ct = ((1.f + g * g) - sq * sq) / (2.f * g);
        const float st = std::sqrt(std::max(0.f, 1.f - ct * ct));
        float sn, cs;
        pmSinCos2Pi(rng.uniform(), sn, cs);
        dir = toWorld(inDir, {st * cs, st * sn, ct});
        pdfOmega = hgEval(g, -dot(inDir, dir));
      } else {
        u1 = rng.uniform();
        u2 = rng.uniform();
        dir = uniformSphere(u1, u2);
        pdfOmega = INV_FOURPI;
      }
    } else {
      u1 = rng.uniform();
      u2 = rng.uniform();
      dir = toWorld(curN, cosineHemisphere(u1, u2));
      pdfOmega = std::max(0.f, dot(dir, curN)) * INV_PI;
      if (pdfOmega <= 0.f) break;
    }
    dir = unit(dir);
  }
  return appended;
}

}  // namespace

extern "C" {

// fills `out` (caller-allocated arrays of n entries) with exactly n beams; returns the number of light paths traced
long long prims_ref_trace_beams(const gvpm_box_scene *scene, const gvpm_medium *med, size_t n, uint64_t seed,
                                int max_depth, int rr_depth, int min_depth, gvpm_beam_soa *out) {
  if (!scene || !med || !out) return -1;
  BeamSink sink{out, n, 0, 0, false};
  const int md = max_depth > 0 ? max_depth : 64;
  uint64_t path = 0;
  while (sink.filled < n) {
    sink.storedAny = false;
    walkBeams(*scene, *med, seed, path, md, rr_depth, min_depth, sink);
    if (sink.storedAny) ++sink.pathId;
    ++path;
    if (path > (1ull << 40)) return -1;
  }
  return (long long)path;
}

// one photon plane per beam: setEndPoint + LTPhotonPlane::transformBeam (gvpm_host::transformBeam) with beam i drawing
// from PCG32(seed ^ 0xA0761D6478BD642F, i) and the polynomial log / sin / cos; returns n, or -1 (sampling_weight != 1)
long long prims_ref_planes_from_beams(const gvpm_beam_soa *beams, size_t n, const gvpm_medium *med, uint64_t seed,
                                      gvpm_plane_soa *out) {
  if (!beams || !med || !out || med->sampling_weight != 1.0f) return -1;
  const float Epsilon = 1e-4f, density = med->sigma_s[1] + med->sigma_a[1];
  for (size_t i = 0; i < n; ++i) {
    const float *o = beams->origin + 3 * i, *e = beams->end + 3 * i;
    V d{e[0] - o[0], e[1] - o[1], e[2] - o[2]};
    const float len = std::sqrt((d.x * d.x + d.y * d.y) + d.z * d.z), rcp = 1.0f / len;
    d = d * rcp;
    Rng rng(seed ^ 0xA0761D6478BD642FULL, i);
    const float rand = rng.uniform();
    const float length1 = -pmLog(1.f - rand) / density + Epsilon;
    V w1;
    for (;;) {
      const float sx = rng.uniform(), sy = rng.uniform();
      if (med->phase_type == GVPM_PHASE_ISOTROPIC) {
        const float z = 1.f - 2.f * sy, r = std::sqrt(std::max(0.f, 1.f - z * z));
        float sn, cs;
        pmSinCos2Pi(sx, sn, cs);
        w1 = {r * cs, r * sn, z};
      } else {
        const float g = med->hg_g;
        float cosTheta;
        if (std::fabs(g) < Epsilon) {
          cosTheta = 1.f - 2.f * sx;
        } else {
          const float sq = (1.f - g * g) / ((1.f - g) + (2.f * g) * sx);
          cosTheta = ((1.f + g * g) - sq * sq) / (2.f * g);
        }
        const float sinTheta = std::sqrt(std::max(0.f, 1.f - cosTheta * cosTheta));
        float sn, cs;
        pmSinCos2Pi(sy, sn, cs);
        const float lx = sinTheta * cs, ly = sinTheta * sn, lz = cosTheta;
        const float sign = std::copysign(1.0f, d.z), a = -1.0f / (sign + d.z), b = (d.x * d.y) * a;
        const V s{1.f + ((sign * d.x) * d.x) * a, sign * b, (-sign) * d.x}, t{b, sign + (d.y * d.y) * a, -d.y};
        w1 = (s * lx + t * ly) + d * lz;
      }
      if (std::fabs(dot(d, w1)) != 1.0f) break;
    }
    put(out->origin, i, V{o[0], o[1], o[2]});
    put(out->w0, i, d);
    const_cast<float *>(out->length0)[i] = len;
    put(out->w1, i, w1);
    const_cast<float *>(out->length1)[i] = length1;
    put(out->flux, i, V{beams->flux[3 * i], beams->flux[3 * i + 1], beams->flux[3 * i + 2]});
    const_cast<int32_t *>(out->edge_id)[i] = (int32_t)beams->depth[i];
  }
  return (long long)n;
}

}  // extern "C"
