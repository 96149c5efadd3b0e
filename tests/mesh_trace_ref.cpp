// mesh_trace_ref.cpp — TEST INFRASTRUCTURE.  CPU restatement of the mesh-scene generators (include/gvpm_b200.h:
// gvpm_set_trace_mesh, gvpm_trace_photons_mesh, gvpm_trace_beams_mesh, gvpm_generate_rays_mesh), the checker the device
// records are compared with BIT FOR BIT (tests/test_gpu_trace_mesh.py).  It reuses, unchanged, the RNG, frame, sampling
// and polynomial log / exp / sin / cos routines of the box tracer's restatement (oracle/gvpm_oracle_trace.cpp, included
// below) and restates the walk of that file and of tests/prims_ref.cpp with the mesh scene as the one difference: the
// emitter pick and the closest hit, here a brute-force loop over every triangle (no BVH).  Compiled with
// -ffp-contract=off: every operation is rounded on its own.
#include "../oracle/gvpm_oracle_trace.cpp"

#include <vector>

namespace {

constexpr uint32_t kNone = 0xffffffffu;

struct Mesh {
  float lo[3], hi[3], glo[3], ghi[3];   // the box and the box grown by 2e-6 of its extent
  size_t n;
  const float *tri, *albedo;
  float power;
  std::vector<uint32_t> emit;   // emissive triangles in index order
  std::vector<float> cdf;       // running fp32 sum of their areas
  uint32_t last = 0;            // the last one of non-zero area
  bool ok = false;
};

float area(const float *p) {
  const float e1x = p[3] - p[0], e1y = p[4] - p[1], e1z = p[5] - p[2];
  const float e2x = p[6] - p[0], e2y = p[7] - p[1], e2z = p[8] - p[2];
  const float cx = e1y * e2z - e1z * e2y, cy = e1z * e2x - e1x * e2z, cz = e1x * e2y - e1y * e2x;
  return 0.5f * std::sqrt((cx * cx + cy * cy) + cz * cz);
}

Mesh makeMesh(const gvpm_mesh_scene &s) {
  Mesh M;
  for (int a = 0; a < 3; ++a) {
    M.lo[a] = s.lo[a]; M.hi[a] = s.hi[a];
    const float m = 2e-6f * (M.hi[a] - M.lo[a]);
    M.glo[a] = M.lo[a] - m; M.ghi[a] = M.hi[a] + m;
  }
  M.n = s.n_tri; M.tri = s.tri; M.albedo = s.albedo; M.power = s.light_power;
  float total = 0.f;
  for (size_t t = 0; t < s.n_tri; ++t) {
    if (!s.emissive[t]) continue;
    const float a = area(s.tri + 9 * t);
    total = total + a;
    if (a > 0.f) { M.last = (uint32_t)M.emit.size(); M.ok = true; }
    M.emit.push_back((uint32_t)t);
    M.cdf.push_back(total);
  }
  return M;
}

V vert(const float *p, int k) { return {p[3 * k], p[3 * k + 1], p[3 * k + 2]}; }
V sub(V a, V b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }

// Triangle::rayIntersect, strictly rounded: the parameter, or +inf when the test rejects the ray
float triT(const float *p, V o, V d) {
  const V p0 = vert(p, 0), e1 = sub(vert(p, 1), p0), e2 = sub(vert(p, 2), p0);
  const V pvec = cross(d, e2);
  const float det = dot(e1, pvec);
  if (det == 0.f) return INFINITY;
  const float inv = 1.f / det;
  const V tvec = sub(o, p0);
  const float u = dot(tvec, pvec) * inv;
  if (u < 0.f || u > 1.f) return INFINITY;
  const V qvec = cross(tvec, e1);
  const float v = dot(d, qvec) * inv;
  if (v >= 0.f && u + v <= 1.f) return dot(e2, qvec) * inv;
  return INFINITY;
}

// the nearest triangle with 1e-6 < t <= bound, ties to the smaller index, never `skip`: its index, or kNone
uint32_t closest(const Mesh &M, V o, V d, float &bound, uint32_t skip) {
  uint32_t best = kNone;
  for (size_t t = 0; t < M.n; ++t) {
    if ((uint32_t)t == skip) continue;
    const float tt = triT(M.tri + 9 * t, o, d);
    if (tt > 1e-6f && tt <= bound && (tt < bound || (uint32_t)t < best)) { bound = tt; best = (uint32_t)t; }
  }
  return best;
}

float boxExit(const float *lo, const float *hi, V o, V d) {
  float t = INFINITY;
  for (int a = 0; a < 3; ++a) {
    const float dc = axisOf(d, a);
    if (dc == 0.f) continue;
    const float ta = ((dc > 0.f ? hi[a] : lo[a]) - axisOf(o, a)) / dc;
    if (ta < t) t = ta;
  }
  return t;
}

V triNormal(const float *p) {
  const V p0 = vert(p, 0);
  return unit(cross(sub(vert(p, 1), p0), sub(vert(p, 2), p0)));
}

struct MHit { float t; V n, albedo; bool escaped; uint32_t tri; };
MHit intersectMesh(const Mesh &M, V o, V d, uint32_t skip) {
  // triangles up to the exit of the grown box (every triangle lies in it), else the exit of the box itself
  float t = boxExit(M.glo, M.ghi, o, d);
  const uint32_t k = closest(M, o, d, t, skip);
  if (k == kNone) return {boxExit(M.lo, M.hi, o, d), {0, 0, 0}, {0, 0, 0}, true, kNone};
  const V n = triNormal(M.tri + 9 * (size_t)k);
  const float *a = M.albedo + 3 * (size_t)k;
  return {t, dot(n, d) > 0.f ? -n : n, {a[0], a[1], a[2]}, false, k};
}

uint32_t sampleEmitter(const Mesh &M, Rng &rng, V &pos, V &n) {
  const float target = rng.uniform() * M.cdf.back();
  const uint32_t k = std::min((uint32_t)(std::upper_bound(M.cdf.begin(), M.cdf.end(), target) - M.cdf.begin()), M.last);
  const float u1 = rng.uniform(), u2 = rng.uniform();
  const float *p = M.tri + 9 * (size_t)M.emit[k];
  const V p0 = vert(p, 0), e1 = sub(vert(p, 1), p0), e2 = sub(vert(p, 2), p0);
  const float su = std::sqrt(u1);
  pos = p0 + (e1 * (1.f - su) + e2 * (u2 * su));
  n = unit(cross(e1, e2));
  return M.emit[k];
}

struct Out {   // photons (ph) or beams (bm); records beyond cap are counted but not stored
  gvpm_photon_soa *ph;
  gvpm_beam_soa *bm;
  size_t cap, filled;
  uint32_t pathId;
  bool storedAny;
};

// one light path: the walk of gvpm_oracle_trace.cpp (photons) / prims_ref.cpp (beams) on the mesh
uint32_t walk(const Mesh &M, const gvpm_medium &med, uint64_t seed, uint64_t pathIdx, int maxDepth, int rrDepth,
              int minDepth, Out &out) {
  Rng rng(seed, pathIdx);
  const float sigS = med.sigma_s[0], sigT = med.sigma_s[0] + med.sigma_a[0];
  V curPos, curN, curAlbedo{0, 0, 0}, curWeight{1, 1, 1}, prevPos{1, 1, 1};
  uint32_t curTri = sampleEmitter(M, rng, curPos, curN);
  int curType = GVPM_PARENT_EMITTER, ci = 1;
  float curRr = 1.f;
  float u1 = rng.uniform(), u2 = rng.uniform();
  V dir = toWorld(curN, cosineHemisphere(u1, u2));
  float pdfOmega = std::max(0.f, dot(dir, curN)) * INV_PI;
  V thr{M.power, M.power, M.power};
  const int firstStored = std::max(2, minDepth + 1), firstBeam = std::max(1, minDepth);
  uint32_t appended = 0;
  for (;;) {
    const MHit h = intersectMesh(M, curPos, dir, curTri);
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
    if (out.bm && ci >= firstBeam) {
      if (out.filled < out.cap) {
        const size_t i = out.filled++;
        const gvpm_beam_soa &o = *out.bm;
        put(o.origin, i, curPos); put(o.end, i, nvPos);
        put(o.flux, i, V{(thr.x * curWeight.x) * curRr, (thr.y * curWeight.y) * curRr, (thr.z * curWeight.z) * curRr});
        put(o.prefix_flux, i, prefix); put(o.parent_n, i, curN); put(o.parent_albedo, i, curAlbedo);
        put(o.pred_pos, i, ci >= 2 ? prevPos : V{1, 1, 1}); put(o.end_n, i, nvN);
        const_cast<float *>(o.parent_pdf)[i] = pdfArea;
        const_cast<float *>(o.rr_weight)[i] = curRr;
        const_cast<uint8_t *>(o.parent_type)[i] = (uint8_t)curType;
        const_cast<uint8_t *>(o.end_on_surface)[i] = inMedium ? 0 : 1;
        const_cast<uint8_t *>(o.depth)[i] = (uint8_t)ci;
        const_cast<uint32_t *>(o.path_id)[i] = out.pathId;
        out.storedAny = true;
      }
      ++appended;
    }
    if (out.ph && inMedium && ni >= firstStored) {
      if (out.filled < out.cap) {
        const size_t i = out.filled++;
        const gvpm_photon_soa &o = *out.ph;
        put(o.pos, i, nvPos); put(o.flux, i, flux); put(o.parent_pos, i, curPos);
        put(o.pred_pos, i, ni >= 3 ? prevPos : V{1, 1, 1});
        put(o.parent_n, i, curN); put(o.prefix_flux, i, prefix); put(o.parent_albedo, i, curAlbedo);
        const_cast<float *>(o.parent_pdf)[i] = pdfArea;
        const_cast<float *>(o.edge_pdf)[i] = edgePdf;
        const_cast<float *>(o.rr_weight)[i] = curRr;
        const_cast<uint8_t *>(o.parent_type)[i] = (uint8_t)curType;
        const_cast<uint8_t *>(o.depth)[i] = (uint8_t)(ni - 1);
        const_cast<uint32_t *>(o.path_id)[i] = out.pathId;
        out.storedAny = true;
      }
      ++appended;
    }
    thr = flux;
    prevPos = curPos;
    curPos = nvPos; curN = nvN; curAlbedo = nvAlbedo; curWeight = nvWeight; curType = nvType; curRr = 1.f;
    curTri = inMedium ? kNone : h.tri;
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

long long trace(const gvpm_mesh_scene *scene, const gvpm_medium *med, size_t n, uint64_t seed, int max_depth,
                int rr_depth, int min_depth, Out out) {
  if (!scene || !med) return -1;
  const Mesh M = makeMesh(*scene);
  if (!M.ok) return -1;
  const int md = max_depth > 0 ? max_depth : 64;
  uint64_t path = 0;
  while (out.filled < n) {
    out.storedAny = false;
    walk(M, *med, seed, path, md, rr_depth, min_depth, out);
    if (out.storedAny) ++out.pathId;
    ++path;
    if (path > (1ull << 40)) return -1;
  }
  return (long long)path;
}

struct Cam { V pos, r, u, f; float tx; int w, h; bool inside; };

bool makeCam(const gvpm_lookat_camera &c, const Mesh &M, Cam &C) {
  auto unitOk = [](V a, V &out) {
    const float l = std::sqrt(dot(a, a));
    if (!(l > 0.f) || !std::isfinite(l)) return false;
    out = a * (1.0f / l);
    return true;
  };
  if (!unitOk({c.forward[0], c.forward[1], c.forward[2]}, C.f)) return false;
  if (!unitOk(cross({c.up[0], c.up[1], c.up[2]}, C.f), C.r)) return false;
  C.u = cross(C.f, C.r);
  C.pos = {c.pos[0], c.pos[1], c.pos[2]};
  C.tx = c.tan_half_fov_x; C.w = c.film_w; C.h = c.film_h;
  C.inside = true;
  for (int a = 0; a < 3; ++a) C.inside = C.inside && axisOf(C.pos, a) > M.lo[a] && axisOf(C.pos, a) < M.hi[a];
  return true;
}

void setAxis(V &v, int a, float x) { (a == 0 ? v.x : (a == 1 ? v.y : v.z)) = x; }

bool makeRay(const Mesh &M, const Cam &C, float eps, float tx, float ty, float sx, float sy, V &ro, V &rd, float &rl) {
  const float x = ((sx / (float)C.w - 0.5f) * 2.f) * tx, y = ((sy / (float)C.h - 0.5f) * 2.f) * ty;
  const V dir = unit((C.r * x + C.u * y) + C.f);
  rd = dir;
  if (C.inside) {
    ro = C.pos;
  } else {
    float tIn = -INFINITY, tOut = INFINITY;
    int face = -1;
    for (int a = 0; a < 3; ++a) {
      const float dc = axisOf(dir, a), oc = axisOf(C.pos, a);
      if (dc == 0.f) {
        if (oc < M.lo[a] || oc > M.hi[a]) tOut = -INFINITY;
        continue;
      }
      const float t0 = (M.lo[a] - oc) / dc, t1 = (M.hi[a] - oc) / dc;
      const float tn = t0 < t1 ? t0 : t1, tf = t0 < t1 ? t1 : t0;
      if (tn > tIn) { tIn = tn; face = a; }
      if (tf < tOut) tOut = tf;
    }
    if (face < 0 || !(tIn <= tOut) || !(tIn > 0.f)) { ro = C.pos; rl = 0.f; return false; }
    ro = C.pos + dir * tIn;
    setAxis(ro, face, axisOf(dir, face) > 0.f ? M.lo[face] : M.hi[face]);
    for (int a = 0; a < 3; ++a)
      if (a != face && (axisOf(ro, a) <= M.lo[a] || axisOf(ro, a) >= M.hi[a])) { rl = 0.f; return false; }
    // blocked by a triangle before the entry face moved inwards by the grown box's margin
    const float inner = axisOf(dir, face) > 0.f ? M.lo[face] + (M.lo[face] - M.glo[face])
                                                : M.hi[face] - (M.ghi[face] - M.hi[face]);
    float b = (inner - axisOf(C.pos, face)) / axisOf(dir, face);
    if (closest(M, C.pos, dir, b, kNone) != kNone) { rl = 0.f; return false; }
  }
  rl = intersectMesh(M, ro, rd, kNone).t;
  return rl > 4.f * eps;
}

int compact1by1(uint32_t v) {
  v &= 0x55555555u;
  v = (v ^ (v >> 1)) & 0x33333333u;
  v = (v ^ (v >> 2)) & 0x0f0f0f0fu;
  v = (v ^ (v >> 4)) & 0x00ff00ffu;
  v = (v ^ (v >> 8)) & 0x0000ffffu;
  return (int)v;
}

}  // namespace

extern "C" {

// fills `out` (caller-allocated arrays of n entries) with exactly n photons; returns the light paths traced, or -1
long long mesh_ref_trace_photons(const gvpm_mesh_scene *scene, const gvpm_medium *med, size_t n, uint64_t seed,
                                 int max_depth, int rr_depth, int min_depth, gvpm_photon_soa *out) {
  return trace(scene, med, n, seed, max_depth, rr_depth, min_depth, Out{out, nullptr, n, 0, 0, false});
}
long long mesh_ref_trace_beams(const gvpm_mesh_scene *scene, const gvpm_medium *med, size_t n, uint64_t seed,
                               int max_depth, int rr_depth, int min_depth, gvpm_beam_soa *out) {
  return trace(scene, med, n, seed, max_depth, rr_depth, min_depth, Out{nullptr, out, n, 0, 0, false});
}

// k_generate_rays on the mesh: rays in the device's order (blocks row by row, pixels of a block row-major or Z-order);
// returns the number of rays, or -1
long long mesh_ref_generate_rays(const gvpm_mesh_scene *scene, const gvpm_lookat_camera *cam, uint64_t seed, int block,
                                 int y0, int y1, float eps, gvpm_ray_soa *out) {
  if (!scene || !cam || !out) return -1;
  const Mesh M = makeMesh(*scene);
  Cam C;
  if (!makeCam(*cam, M, C)) return -1;
  const bool zorder = block < 0;
  const int bs = zorder ? -block : block, w = C.w;
  const int blocksX = (w + bs - 1) / bs, blocksY = (y1 - y0 + bs - 1) / bs;
  const float tx = C.tx, ty = (tx * (float)C.h) / (float)w;
  size_t n = 0;
  const int off[4][2] = {{-1, 0}, {1, 0}, {0, 1}, {0, -1}};
  for (int b = 0; b < blocksX * blocksY; ++b) {
    const int bx = (b % blocksX) * bs, by = y0 + (b / blocksX) * bs;
    for (int i = 0; i < bs * bs; ++i) {
      const int x = bx + (zorder ? compact1by1((uint32_t)i) : i % bs), y = by + (zorder ? compact1by1((uint32_t)i >> 1) : i / bs);
      if (x >= w || y >= y1) continue;
      Rng rng(seed ^ 0x9E3779B97F4A7C15ULL, (uint64_t)y * (uint64_t)w + (uint64_t)x);
      const float sx = (float)x + rng.uniform(), sy = (float)y + rng.uniform();
      V ro, rd;
      float rl;
      const bool ok = makeRay(M, C, eps, tx, ty, sx, sy, ro, rd, rl);
      put(out->o, n, ro);
      put(out->d, n, rd);
      const_cast<float *>(out->mint)[n] = eps;
      const_cast<float *>(out->maxt)[n] = ok ? rl - eps : 0.f;
      const_cast<float *>(out->edge_len)[n] = ok ? rl : 0.f;
      put(out->eye_contrib, n, V{1, 1, 1});
      const_cast<float *>(out->xi)[n] = rng.uniform();
      const_cast<int32_t *>(out->px)[n] = x;
      const_cast<int32_t *>(out->py)[n] = y;
      const_cast<int32_t *>(out->edge_id)[n] = C.inside ? 1 : 2;
      for (int k = 0; k < 4; ++k) {
        V ko, kd;
        float kl;
        const bool kv = makeRay(M, C, eps, tx, ty, sx + (float)off[k][0], sy + (float)off[k][1], ko, kd, kl);
        const_cast<uint8_t *>(out->off_valid)[4 * n + k] = kv ? 1 : 0;
        put(out->off_o, 4 * n + k, ko);
        put(out->off_d, 4 * n + k, kd);
        const_cast<float *>(out->off_len)[4 * n + k] = kl;
        put(out->off_eye, 4 * n + k, V{1, 1, 1});
        const_cast<float *>(out->off_sensor)[4 * n + k] = 1.0f;
      }
      ++n;
    }
  }
  return (long long)n;
}

// closest hit of m rays (brute force; skip[i] = triangle to skip or 0xffffffff): t (box exit when no triangle),
// triangle index (0xffffffff: box exit), normal facing the ray
void mesh_ref_closest(const gvpm_mesh_scene *scene, const float *o, const float *d, const uint32_t *skip, size_t m,
                      float *t, uint32_t *tri, float *n) {
  const Mesh M = makeMesh(*scene);
  for (size_t i = 0; i < m; ++i) {
    const MHit h = intersectMesh(M, {o[3 * i], o[3 * i + 1], o[3 * i + 2]}, {d[3 * i], d[3 * i + 1], d[3 * i + 2]},
                                 skip ? skip[i] : kNone);
    t[i] = h.t;
    tri[i] = h.tri;
    n[3 * i] = h.n.x; n[3 * i + 1] = h.n.y; n[3 * i + 2] = h.n.z;
  }
}

// the emitter pick of u0 (and the point of u1, u2): emissive triangle index per draw
void mesh_ref_pick(const gvpm_mesh_scene *scene, const float *u0, size_t m, uint32_t *tri) {
  const Mesh M = makeMesh(*scene);
  for (size_t i = 0; i < m; ++i) {
    const float target = u0[i] * M.cdf.back();
    tri[i] = M.emit[std::min((uint32_t)(std::upper_bound(M.cdf.begin(), M.cdf.end(), target) - M.cdf.begin()), M.last)];
  }
}

}  // extern "C"
