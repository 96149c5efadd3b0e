// generate.cu — the two host stages on either side of the gather, on the device (SURVEY.md §8 rows f-1, f-2), for the
// box scene class of include/gvpm_b200.h (gvpm_box_scene) and the mesh scene class (gvpm_mesh_scene: triangles in the
// medium's box, walked through their BVH by closest_hit_bvh).  The walk, the camera rays and their kernels are
// templates on the scene (its parameter struct); the box instantiations are the code they were before the mesh existed:
//   k_generate_rays   camera-ray medium segments + 4 offset segments of a pinhole sensor: what GatherPointMap::generate
//                     (gvpm/gvpm_gatherpoint.h:259-486), ShiftGatherPoint::generate (gvpm/shift/shift_cameraPath.h:146-413)
//                     and sensorMIS (gvpm_struct.h:608-631) produce per pixel, written straight into the ray staging
//                     arrays (then packed by gvpm_commit_rays)
//   k_trace_count / k_trace_emit   the light-path random walk of GradientPhotonProcess (gvpm/gvpm_proc.cpp:125-210)
//                     + GPhotonMap::tryAppend (gvpm_accel.h:119-199): one thread per light path, two passes (count,
//                     exclusive scan over the paths, emit), so the photons land in path order whatever the launch
//                     geometry and the set is bit-reproducible; photon flux / pdf bookkeeping as libbidir's
//                     (SURVEY.md §9.1).  The same walk emits photon beams instead (EmitKind::Beams): every edge
//                     that does not escape, LTBeamMap::tryAppendLT (gvpm_beams.h:54-84).
//   k_planes_from_beams   LTPhotonPlane::transformBeam (gvpm_plane.h:53-73) of every beam of the current set: one
//                     thread per beam, photon planes written into the plane staging arrays.
//   k_vpm_count / k_vpm_emit   the camera distance samples of G-VPM (computeVolumeGradientPhoton, gvpm.cpp:1141-1175,
//                     as gvpm_synth_vpm_samples restates it) from the current ray set: one thread per ray, count ->
//                     exclusive scan over tiles of rays -> emit into the sample staging arrays, so the samples land in
//                     ray order.
// Random numbers: PCG32 keyed by (seed, pixel index) / (seed, path index) / (seed ^ constant, beam or ray index).  Arithmetic: strictly rounded fp32 in a fixed
// operation order; log, exp, sin and cos are polynomial routines (pm_*) built from +, -, *, / only, so a CPU
// restatement compiled without FMA contraction reproduces every record bit for bit (tests/test_gpu_generate.py).
#include <type_traits>

#include "gvpm_device.cuh"
#include "launch_sizing.cuh"
#include "occluder_device.cuh"
#include "warp_ops.cuh"

namespace gvpm {

// ---- counter-based RNG ---------------------------------------------------------------------------------------------
struct Pcg32 {
  unsigned long long state, inc;
  __device__ Pcg32(unsigned long long seed, unsigned long long seq) {
    state = 0;
    inc = (seq << 1u) | 1u;
    next();
    state += seed;
    next();
  }
  __device__ uint32_t next() {
    const unsigned long long old = state;
    state = old * 6364136223846793005ULL + inc;
    const uint32_t xorshifted = (uint32_t)(((old >> 18u) ^ old) >> 27u);
    const uint32_t rot = (uint32_t)(old >> 59u);
    return (xorshifted >> rot) | (xorshifted << ((0u - rot) & 31u));
  }
  __device__ float uniform() { return __fmul_rn((float)(next() >> 8), 1.0f / 16777216.0f); }  // [0,1)
};

// ---- portable elementary functions (strictly rounded, fixed order) ----------------------------------------------------
__device__ __forceinline__ float pm_log(float x) {   // x > 0, normal
  const uint32_t bits = __float_as_uint(x);
  int e = (int)(bits >> 23) - 127;
  sf m(__uint_as_float((bits & 0x007fffffu) | 0x3f800000u));   // [1, 2)
  if (m.v > 1.41421356f) { m = m * sf(0.5f); e += 1; }
  const sf s = (m - sf(1.f)) / (m + sf(1.f));
  const sf s2 = s * s;
  sf p(0.11111111f);
  p = p * s2 + sf(0.14285715f);
  p = p * s2 + sf(0.2f);
  p = p * s2 + sf(0.33333334f);
  p = p * s2 + sf(1.0f);
  return ((sf(2.f) * s) * p + sf((float)e) * sf(0.69314718f)).v;
}
__device__ __forceinline__ float pm_exp(float x) {   // x <= ~0
  if (x < -87.f) return 0.f;
  const sf n(floorf((sf(x) * sf(1.44269504f) + sf(0.5f)).v));
  sf r = sf(x) - n * sf(0.693359375f);
  r = r - n * sf(-2.12194440e-4f);
  sf p(1.0f / 720.0f);
  p = p * r + sf(1.0f / 120.0f);
  p = p * r + sf(1.0f / 24.0f);
  p = p * r + sf(1.0f / 6.0f);
  p = p * r + sf(0.5f);
  p = p * r + sf(1.0f);
  p = p * r + sf(1.0f);
  const int ni = (int)n.v;
  return (sf(__uint_as_float((uint32_t)(ni + 127) << 23)) * p).v;
}
__device__ __forceinline__ void pm_sincos2pi(float u, float &sn, float &cs) {   // sin / cos of 2 pi u, u in [0, 1)
  const sf q(floorf((sf(u) * sf(4.f) + sf(0.5f)).v));
  const sf a = (sf(u) - q * sf(0.25f)) * sf(6.2831855f);   // [-pi/4, pi/4]
  const sf a2 = a * a;
  sf p(-1.9841270e-4f);
  p = p * a2 + sf(8.3333333e-3f);
  p = p * a2 + sf(-0.16666667f);
  p = p * a2 + sf(1.0f);
  const sf s = a * p;
  sf c(2.4801587e-5f);
  c = c * a2 + sf(-1.3888889e-3f);
  c = c * a2 + sf(4.1666668e-2f);
  c = c * a2 + sf(-0.5f);
  c = c * a2 + sf(1.0f);
  switch ((int)q.v & 3) {
    case 0: sn = s.v; cs = c.v; break;
    case 1: sn = c.v; cs = -s.v; break;
    case 2: sn = -s.v; cs = -c.v; break;
    default: sn = -c.v; cs = s.v; break;
  }
}

// ---- scene ---------------------------------------------------------------------------------------------------------
struct SceneHit { sf t; v3 n, albedo; bool escaped; };
struct MeshSceneHit : SceneHit { uint32_t tri; };   // tri: the triangle hit (caller's index)
__device__ __forceinline__ float comp(const v3 &a, int axis) { return axis == 0 ? a.x.v : (axis == 1 ? a.y.v : a.z.v); }
// nearest of the five walls, the open face and the rectangles, in this order (ties keep the earlier one)
__device__ __forceinline__ SceneHit intersect_scene(const gvpm_box_scene &S, v3 o, v3 d) {
  SceneHit h;
  h.t = sf(1e30f);
  h.escaped = false;
  h.n = v3(0.f, 0.f, 0.f);
  h.albedo = v3(0.7f, 0.7f, 0.7f);
  auto plane = [&](int axis, float pos, v3 n, const float *alb, bool esc) {
    const float dc = comp(d, axis), oc = comp(o, axis);
    if (dc == 0.f) return;
    const sf t = (sf(pos) - sf(oc)) / sf(dc);
    if (t.v > 1e-6f && t < h.t) {
      h.t = t; h.n = n; h.escaped = esc;
      h.albedo = esc ? v3(0.f, 0.f, 0.f) : v3(alb[0], alb[1], alb[2]);
    }
  };
  plane(0, S.lo[0], v3(1.f, 0.f, 0.f), S.face_albedo[0], false);
  plane(0, S.hi[0], v3(-1.f, 0.f, 0.f), S.face_albedo[1], false);
  plane(1, S.lo[1], v3(0.f, 1.f, 0.f), S.face_albedo[2], false);
  plane(1, S.hi[1], v3(0.f, -1.f, 0.f), S.face_albedo[3], false);
  plane(2, S.hi[2], v3(0.f, 0.f, -1.f), S.face_albedo[4], false);
  plane(2, S.lo[2], v3(0.f, 0.f, 1.f), S.face_albedo[4], true);
  if (d.y.v != 0.f)
    for (int r = 0; r < S.n_rects; ++r) {
      const sf t = (sf(S.rect[r].y) - o.y) / d.y;
      if (t.v > 1e-6f && t < h.t) {
        const sf x = o.x + d.x * t, z = o.z + d.z * t;
        if (x.v >= S.rect[r].x0 && x.v <= S.rect[r].x1 && z.v >= S.rect[r].z0 && z.v <= S.rect[r].z1) {
          h.t = t;
          h.n = d.y.v < 0.f ? v3(0.f, 1.f, 0.f) : v3(0.f, -1.f, 0.f);
          h.albedo = v3(S.rect[r].albedo[0], S.rect[r].albedo[1], S.rect[r].albedo[2]);
          h.escaped = false;
        }
      }
    }
  return h;
}
__device__ __forceinline__ v3 unit(v3 a) { return a * (sf(1.0f) / length(a)); }
// the box has no triangles to skip
__device__ __forceinline__ SceneHit intersect_scene(const gvpm_box_scene &S, v3 o, v3 d, uint32_t) {
  return intersect_scene(S, o, d);
}

// ---- mesh scene (gvpm_set_trace_mesh) -----------------------------------------------------------------------------------
// parameter of the exit of a ray from inside the box lo / hi: the nearest of the three far planes, strictly rounded
__device__ __forceinline__ sf box_exit(const float *lo, const float *hi, v3 o, v3 d) {
  sf t(INFINITY);
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float dc = comp(d, a);
    if (dc == 0.f) continue;
    const sf ta = (sf(dc > 0.f ? hi[a] : lo[a]) - sf(comp(o, a))) / sf(dc);
    if (ta < t) t = ta;
  }
  return t;
}
// winding normal of the triangle at leaf slot s / of 9 floats
__device__ __forceinline__ v3 tri_normal(const float *p) {
  const v3 p0(p[0], p[1], p[2]), p1(p[3], p[4], p[5]), p2(p[6], p[7], p[8]);
  return unit(cross(p1 - p0, p2 - p0));
}
// the nearest triangle (closest_hit_bvh, never `skip`) up to the exit of the grown box, else the box exit (escaped):
// a triangle at t <= t_exit wins, and so does one on a face of the box that rounding puts just beyond it
__device__ __forceinline__ MeshSceneHit intersect_scene(const MeshScene &M, v3 o, v3 d, uint32_t skip) {
  const sf texit = box_exit(M.lo, M.hi, o, d);
  const MeshHit c = closest_hit_bvh(M, o, d, box_exit(M.glo, M.ghi, o, d), skip);
  MeshSceneHit h;
  h.tri = c.idx;
  if (c.slot == kMeshNone) {
    h.t = texit; h.escaped = true;
    h.n = v3(0.f, 0.f, 0.f); h.albedo = v3(0.f, 0.f, 0.f);
    return h;
  }
  h.t = sf(c.t);
  h.escaped = false;
  const v3 n = tri_normal(M.tri + 9 * (size_t)c.slot);
  h.n = dot(n, d).v > 0.f ? -n : n;   // facing the incoming ray
  const float *a = M.albedo + 3 * (size_t)c.slot;
  h.albedo = v3(a[0], a[1], a[2]);
  return h;
}

// ---- f-2: camera rays --------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool make_ray(const MeshRayGenParams &P, sf tx, sf ty, sf sx, sf sy, v3 &ro, v3 &rd, sf &rl) {
  const MeshScene &M = P.scene;
  const LookatCam &C = P.cam;
  const sf w((float)C.film_w), h((float)C.film_h);
  const sf x = ((sx / w - sf(0.5f)) * sf(2.f)) * tx, y = ((sy / h - sf(0.5f)) * sf(2.f)) * ty;
  const v3 r(C.r[0], C.r[1], C.r[2]), u(C.u[0], C.u[1], C.u[2]), f(C.f[0], C.f[1], C.f[2]);
  const v3 dir = unit((r * x + u * y) + f);
  const v3 cam(C.pos[0], C.pos[1], C.pos[2]);
  rd = dir;
  if (C.inside_medium) {
    ro = cam;
  } else {
    // slab test: the entry face is the axis of the largest near parameter (the first such axis on ties)
    sf tIn(-INFINITY), tOut(INFINITY);
    int face = -1;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float dc = comp(dir, a), oc = comp(cam, a);
      if (dc == 0.f) {
        if (oc < M.lo[a] || oc > M.hi[a]) { tOut = sf(-INFINITY); }
        continue;
      }
      const sf t0 = (sf(M.lo[a]) - sf(oc)) / sf(dc), t1 = (sf(M.hi[a]) - sf(oc)) / sf(dc);
      const sf tn = t0 < t1 ? t0 : t1, tf = t0 < t1 ? t1 : t0;
      if (tn > tIn) { tIn = tn; face = a; }
      if (tf < tOut) tOut = tf;
    }
    if (face < 0 || !(tIn <= tOut) || !(tIn.v > 0.f)) { ro = cam; rl = sf(0.f); return false; }
    ro = cam + dir * tIn;
    const float plane = comp(dir, face) > 0.f ? M.lo[face] : M.hi[face];
    if (face == 0) ro.x = sf(plane); else if (face == 1) ro.y = sf(plane); else ro.z = sf(plane);
#pragma unroll
    for (int a = 0; a < 3; ++a)
      if (a != face && (comp(ro, a) <= M.lo[a] || comp(ro, a) >= M.hi[a])) { rl = sf(0.f); return false; }
    // a triangle in front of the entry or on the entry face (up to the grown box's tolerance inside it) hides the
    // medium: the bound is where the ray crosses the face moved inwards by that tolerance
    const float inner = comp(dir, face) > 0.f ? (sf(M.lo[face]) + (sf(M.lo[face]) - sf(M.glo[face]))).v
                                              : (sf(M.hi[face]) - (sf(M.ghi[face]) - sf(M.hi[face]))).v;
    const sf tBlock = (sf(inner) - sf(comp(cam, face))) / sf(comp(dir, face));
    if (closest_hit_bvh(M, cam, dir, tBlock, kMeshNone).slot != kMeshNone) { rl = sf(0.f); return false; }
  }
  const SceneHit hit = intersect_scene(M, ro, rd, kMeshNone);
  rl = hit.t;
  return hit.t.v > (sf(4.f) * sf(P.epsilon)).v;   // a segment that reaches the box exit ends there
}
__device__ __forceinline__ bool make_ray(const RayGenParams &P, sf tx, sf ty, sf sx, sf sy, v3 &ro, v3 &rd, sf &rl) {
  const gvpm_box_scene &S = P.scene;
  const sf w((float)P.cam.film_w), h((float)P.cam.film_h);
  const v3 dir = unit(v3(((sx / w - sf(0.5f)) * sf(2.f)) * tx, ((sy / h - sf(0.5f)) * sf(2.f)) * ty, sf(1.0f)));
  const v3 cam(P.cam.pos[0], P.cam.pos[1], P.cam.pos[2]);
  rd = dir;
  if (P.cam.inside_medium) {
    ro = cam;
  } else {
    const sf tIn = (sf(S.lo[2]) - cam.z) / dir.z;
    ro = cam + dir * tIn;
    ro.z = sf(S.lo[2]);
    if (ro.x.v <= S.lo[0] || ro.x.v >= S.hi[0] || ro.y.v <= S.lo[1] || ro.y.v >= S.hi[1]) { rl = sf(0.f); return false; }
  }
  const SceneHit hit = intersect_scene(S, ro, rd);
  rl = hit.t;
  return hit.t.v > (sf(4.f) * sf(P.epsilon)).v && !hit.escaped;
}
__device__ __forceinline__ int compact1by1(uint32_t v) {
  v &= 0x55555555u;
  v = (v ^ (v >> 1)) & 0x33333333u;
  v = (v ^ (v >> 2)) & 0x0f0f0f0fu;
  v = (v ^ (v >> 4)) & 0x00ff00ffu;
  v = (v ^ (v >> 8)) & 0x0000ffffu;
  return (int)v;
}
__device__ __forceinline__ void put3(float *dst, size_t i, v3 v) { dst[3 * i] = v.x.v; dst[3 * i + 1] = v.y.v; dst[3 * i + 2] = v.z.v; }

// one CTA per block x block pixel block (block <= 32: 1024 threads); the pixels of a block that fall inside the image
// are compacted in block order (row-major or Z-order), blocks follow each other row by row
template <class Params>
__global__ void __launch_bounds__(1024) k_generate_rays(const __grid_constant__ Params P) {
  __shared__ uint32_t warpTot[32];
  const int w = P.cam.film_w, bs = P.block;
  const int blocksX = (w + bs - 1) / bs;
  const int bx = (blockIdx.x % blocksX) * bs, by = P.y0 + (blockIdx.x / blocksX) * bs;
  const int i = threadIdx.x, lane = i & 31, wp = i >> 5;
  const int x = bx + (P.zorder ? compact1by1((uint32_t)i) : i % bs), y = by + (P.zorder ? compact1by1((uint32_t)i >> 1) : i / bs);
  const bool valid = i < bs * bs && x < w && y < P.y1;
  const uint32_t vm = __ballot_sync(0xffffffffu, valid);
  if (lane == 0) warpTot[wp] = __popc(vm);
  __syncthreads();
  uint32_t before = __popc(vm & ((1u << lane) - 1u));
  for (int k = 0; k < wp; ++k) before += warpTot[k];
  if (!valid) return;
  const int rowsHere = min(bs, P.y1 - by);
  const size_t n = (size_t)w * (size_t)(by - P.y0) + (size_t)bx * (size_t)rowsHere + before;

  const sf tx(P.cam.tan_half_fov_x), ty = tx * sf((float)P.cam.film_h) / sf((float)w);
  Pcg32 rng(P.seed ^ 0x9E3779B97F4A7C15ULL, (unsigned long long)y * (unsigned long long)w + (unsigned long long)x);
  const sf sx = sf((float)x) + sf(rng.uniform()), sy = sf((float)y) + sf(rng.uniform());
  v3 ro, rd;
  sf rl;
  const bool ok = make_ray(P, tx, ty, sx, sy, ro, rd, rl);
  put3(P.o, n, ro);
  put3(P.d, n, rd);
  P.mint[n] = P.epsilon;
  P.maxt[n] = ok ? (rl - sf(P.epsilon)).v : 0.f;   // empty segment when the pixel misses the medium
  P.edge_len[n] = ok ? rl.v : 0.f;
  put3(P.eye_contrib, n, v3(1.f, 1.f, 1.f));
  P.xi[n] = rng.uniform();
  P.px[n] = x;
  P.py[n] = y;
  P.edge_id[n] = P.cam.inside_medium ? 1 : 2;
  const int off[4][2] = {{-1, 0}, {1, 0}, {0, 1}, {0, -1}};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    v3 ko, kd;
    sf kl;
    const bool kv = make_ray(P, tx, ty, sx + sf((float)off[k][0]), sy + sf((float)off[k][1]), ko, kd, kl);
    P.off_valid[4 * n + k] = kv ? 1 : 0;
    put3(P.off_o, 4 * n + k, ko);
    put3(P.off_d, 4 * n + k, kd);
    P.off_len[4 * n + k] = kl.v;
    put3(P.off_eye, 4 * n + k, v3(1.f, 1.f, 1.f));
    P.off_sensor[4 * n + k] = 1.0f;   // sensorMIS of a pinhole (gvpm_struct.h:608-631: pdf ratio x Jacobian = 1)
  }
}

// ---- f-1: light-path random walk ----------------------------------------------------------------------------------------
__device__ __forceinline__ void frame_of(v3 n, v3 &s, v3 &t) {
  if (fabsf(n.x.v) > fabsf(n.y.v)) {
    const sf il = sf(1.0f) / ssqrt(n.x * n.x + n.z * n.z);
    t = v3(n.z * il, sf(0.f), -(n.x * il));
  } else {
    const sf il = sf(1.0f) / ssqrt(n.y * n.y + n.z * n.z);
    t = v3(sf(0.f), n.z * il, -(n.y * il));
  }
  s = cross(t, n);
}
__device__ __forceinline__ v3 to_world(v3 n, v3 l) {
  v3 s, t;
  frame_of(n, s, t);
  return (s * l.x + t * l.y) + n * l.z;
}
__device__ __forceinline__ v3 cosine_hemisphere(float u1, float u2) {
  float sn, cs;
  pm_sincos2pi(u2, sn, cs);
  const sf r = ssqrt(sf(u1));
  const sf x = r * sf(cs), y = r * sf(sn);
  return v3(x, y, safe_sqrt((sf(1.f) - x * x) - y * y));
}
__device__ __forceinline__ v3 uniform_sphere(float u1, float u2) {
  float sn, cs;
  pm_sincos2pi(u2, sn, cs);
  const sf z = sf(1.f) - sf(2.f) * sf(u1);
  const sf r = safe_sqrt(sf(1.f) - z * z);
  return v3(r * sf(cs), r * sf(sn), z);
}
__device__ __forceinline__ sf hg_eval(sf g, sf cosWiWo) {   // phase/hg.cpp:107-110 with dot(wi, wo)
  const sf temp = (sf(1.0f) + g * g) + (sf(2.0f) * g) * cosWiWo;
  return (sf(GVPM_INV_FOURPI) * (sf(1.f) - g * g)) / (temp * ssqrt(temp));
}

// ---- emitter sample of the mesh scene: vertex 1 of a light path; returns the triangle it lies on --------------------
// u0 picks the first emissive triangle whose running area sum exceeds u0 * total (clamped to the last one of
// non-zero area), u1, u2 a uniform point on it (p0 + e1 (1 - sqrt u1) + e2 u2 sqrt u1); the normal is the winding
// normal, the side the triangle emits on
__device__ __forceinline__ uint32_t sample_emitter(const MeshScene &M, Pcg32 &rng, v3 &pos, v3 &n) {
  const float target = (sf(rng.uniform()) * sf(M.emit_total)).v;
  uint32_t lo = 0, hi = M.n_emit;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (M.emit_cdf[mid] > target) hi = mid; else lo = mid + 1;
  }
  const uint32_t k = min(lo, M.emit_last);
  const float u1 = rng.uniform(), u2 = rng.uniform();
  const float *p = M.emit_tri + 9 * (size_t)k;
  const v3 p0(p[0], p[1], p[2]), e1 = v3(p[3], p[4], p[5]) - p0, e2 = v3(p[6], p[7], p[8]) - p0;
  const sf su = ssqrt(sf(u1));
  pos = p0 + (e1 * (sf(1.f) - su) + e2 * (sf(u2) * su));
  n = unit(cross(e1, e2));
  return M.emit_idx[k];
}

template <class Scene> constexpr bool kIsMesh = std::is_same<Scene, MeshScene>::value;

// What a light path stores: volume photons (GPhotonMap::tryAppend) or photon beams (LTBeamMap::tryAppendLT).
enum class EmitKind { Photons, Beams };

// The walk of light path `pathIdx`.  EMIT = false: returns the number of records it would store.  EMIT = true: stores
// them at slots first, first + 1, ... (< n_total) with path id `pid`.  The RNG draws, the arithmetic and the
// termination do not depend on KIND; only which records are written does.
template <class Scene, EmitKind KIND, bool EMIT>
__device__ __forceinline__ uint32_t walk_path(const TraceParamsT<Scene> &P, unsigned long long pathIdx,
                                              unsigned long long first, uint32_t pid) {
  const Scene &S = P.scene;
  Pcg32 rng(P.seed, pathIdx);
  const sf sigS(P.sigma_s), sigT = sf(P.sigma_s) + sf(P.sigma_a);
  // vertex 0 = emitter supernode (weight = power), vertex 1 = emitter sample
  v3 curPos, curN(0.f, -1.f, 0.f), curAlbedo(0.f, 0.f, 0.f), curWeight(1.f, 1.f, 1.f), prevPos(1.f, 1.f, 1.f);
  uint32_t curTri = kMeshNone;   // the mesh triangle the current vertex lies on
  if constexpr (kIsMesh<Scene>) {
    curTri = sample_emitter(S, rng, curPos, curN);   // one more draw (the triangle pick) before the point's two
  } else {   // a point of the light rectangle, normal -y
    const float u1 = rng.uniform(), u2 = rng.uniform();
    curPos = v3(sf(S.light_x0) + (sf(S.light_x1) - sf(S.light_x0)) * sf(u1), sf(S.light_y),
                sf(S.light_z0) + (sf(S.light_z1) - sf(S.light_z0)) * sf(u2));
  }
  int curType = GVPM_PARENT_EMITTER;
  sf curRr(1.f);
  v3 dir;
  {
    const float u1 = rng.uniform(), u2 = rng.uniform();
    dir = to_world(curN, cosine_hemisphere(u1, u2));
  }
  sf pdfOmega = smax(sf(0.f), dot(dir, curN)) * sf(GVPM_INV_PI);
  v3 thr(S.light_power, S.light_power, S.light_power);
  int ci = 1;
  uint32_t appended = 0;
  const int firstStored = max(2, P.min_depth + 1), firstBeam = max(1, P.min_depth);
  for (;;) {
    const auto h = intersect_scene(S, curPos, dir, curTri);
    const sf t = (-sf(pm_log((sf(1.0f) - sf(rng.uniform())).v))) / sigT;
    const bool inMedium = t < h.t;
    const sf L = inMedium ? t : h.t;
    if (!inMedium && h.escaped) break;
    const sf T(pm_exp(((-sigT) * L).v));
    const sf edgePdf = inMedium ? sigT * T : T;
    const sf ew = T / edgePdf;
    const v3 nvPos = curPos + dir * L;
    sf pdfArea;
    int nvType;
    v3 nvN(0.f, 0.f, 0.f), nvAlbedo(0.f, 0.f, 0.f), nvWeight;
    if (inMedium) {
      nvType = GVPM_PARENT_MEDIUM;
      nvWeight = v3(sigS, sigS, sigS);
      pdfArea = pdfOmega / (L * L);
    } else {
      nvType = GVPM_PARENT_SURFACE;
      nvN = h.n;
      nvAlbedo = h.albedo;
      nvWeight = h.albedo;
      pdfArea = (pdfOmega * sf(fabsf(dot(h.n, dir).v))) / (L * L);
    }
    const v3 prefix = thr;
    const v3 step((curWeight.x * curRr) * ew, (curWeight.y * curRr) * ew, (curWeight.z * curRr) * ew);
    const v3 flux = thr * step;
    const int ni = ci + 1;
    if (KIND == EmitKind::Beams && ci >= firstBeam) {
      // beam = edge ci -> ci + 1; its flux stops before the edge's own transmittance (gvpm_beams.h:29-35)
      if (EMIT) {
        const unsigned long long slot = first + appended;
        if (slot < P.n_total) {
          put3(P.b_origin, slot, curPos); put3(P.b_end, slot, nvPos);
          put3(P.b_flux, slot, v3((thr.x * curWeight.x) * curRr, (thr.y * curWeight.y) * curRr, (thr.z * curWeight.z) * curRr));
          put3(P.b_prefix_flux, slot, prefix); put3(P.b_parent_n, slot, curN); put3(P.b_parent_albedo, slot, curAlbedo);
          put3(P.b_pred_pos, slot, ci >= 2 ? prevPos : v3(1.f, 1.f, 1.f)); put3(P.b_end_n, slot, nvN);
          P.b_parent_pdf[slot] = pdfArea.v; P.b_rr_weight[slot] = curRr.v;
          P.b_parent_type[slot] = (uint8_t)curType; P.b_end_on_surface[slot] = inMedium ? 0 : 1;
          P.b_depth[slot] = (uint8_t)ci; P.b_path_id[slot] = pid;
        }
      }
      ++appended;
    }
    if (KIND == EmitKind::Photons && inMedium && ni >= firstStored) {
      if (EMIT) {
        const unsigned long long slot = first + appended;
        if (slot < P.n_total && P.aos != nullptr) {
          // the record the gather reads (gvpm_device.cuh photon_record)
          photon_record(P.aos + slot * 8, nvPos, pack_meta((uint32_t)curType, (uint32_t)(ni - 1), pid), flux, pdfArea,
                        curPos, edgePdf, ni >= 3 ? prevPos : v3(1.f, 1.f, 1.f), curRr, curN, prefix, curAlbedo, 0u);
        } else if (slot < P.n_total) {
          put3(P.pos, slot, nvPos); put3(P.flux, slot, flux); put3(P.parent_pos, slot, curPos);
          put3(P.pred_pos, slot, ni >= 3 ? prevPos : v3(1.f, 1.f, 1.f));
          put3(P.parent_n, slot, curN); put3(P.prefix_flux, slot, prefix); put3(P.parent_albedo, slot, curAlbedo);
          P.parent_pdf[slot] = pdfArea.v; P.edge_pdf[slot] = edgePdf.v; P.rr_weight[slot] = curRr.v;
          P.parent_type[slot] = (uint8_t)curType; P.depth[slot] = (uint8_t)(ni - 1); P.path_id[slot] = pid;
        }
      }
      ++appended;
    }
    thr = flux;
    prevPos = curPos;
    curPos = nvPos; curN = nvN; curAlbedo = nvAlbedo; curWeight = nvWeight; curType = nvType; curRr = sf(1.f);
    if constexpr (kIsMesh<Scene>) curTri = inMedium ? kMeshNone : h.tri;
    ci = ni;
    if (ci >= P.max_depth) break;   // path length bound
    // russian roulette before sampling the next direction (vertex.cpp:291-302)
    if (ci - 1 >= P.rr_depth) {
      const sf m = smax(thr.x * curWeight.x, smax(thr.y * curWeight.y, thr.z * curWeight.z));
      const sf q(fminf(m.v, 0.95f));
      if (!(rng.uniform() < q.v)) break;
      curRr = sf(1.0f) / q;
    }
    const v3 inDir = dir;
    if (curType == GVPM_PARENT_MEDIUM) {
      if (P.phase_type == GVPM_PHASE_HG && fabsf(P.hg_g) > 1e-4f) {
        const sf g(P.hg_g);
        const float u = rng.uniform();
        const sf sq = (sf(1.f) - g * g) / ((sf(1.f) - g) + (sf(2.f) * g) * sf(u));
        const sf ct = ((sf(1.f) + g * g) - sq * sq) / (sf(2.f) * g);
        const sf st = safe_sqrt(sf(1.f) - ct * ct);
        float sn, cs;
        pm_sincos2pi(rng.uniform(), sn, cs);
        dir = to_world(inDir, v3(st * sf(cs), st * sf(sn), ct));
        pdfOmega = hg_eval(g, -dot(inDir, dir));   // wi = -inDir
      } else {
        const float u1 = rng.uniform(), u2 = rng.uniform();
        dir = uniform_sphere(u1, u2);
        pdfOmega = sf(GVPM_INV_FOURPI);
      }
    } else {
      const float u1 = rng.uniform(), u2 = rng.uniform();
      dir = to_world(curN, cosine_hemisphere(u1, u2));
      pdfOmega = smax(sf(0.f), dot(dir, curN)) * sf(GVPM_INV_PI);
      if (pdfOmega.v <= 0.f) break;
    }
    dir = unit(dir);
  }
  return appended;
}

// pass 1: records per path; block totals of (records, contributing paths) packed as (paths << 40 | records)
template <class Scene, EmitKind KIND>
__global__ void __launch_bounds__(256) k_trace_count(const __grid_constant__ TraceParamsT<Scene> P, uint8_t *__restrict__ counts,
                                                      unsigned long long *__restrict__ block_tot) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t c = 0;
  if (k < P.n_paths) {
    c = walk_path<Scene, KIND, false>(P, P.path_base + k, 0ull, 0u);
    counts[k] = (uint8_t)c;
  }
  const unsigned long long t = block_total<8>((unsigned long long)c | ((unsigned long long)(c ? 1u : 0u) << 40));
  if (threadIdx.x == 0) block_tot[blockIdx.x] = t;
}
// pass 2: the same walks, stored.  last_path[0] = 1 + index of the path that stored record n_total - 1.
template <class Scene, EmitKind KIND>
__global__ void __launch_bounds__(256) k_trace_emit(const __grid_constant__ TraceParamsT<Scene> P, const uint8_t *__restrict__ counts,
                                                     const unsigned long long *__restrict__ block_off,
                                                     unsigned long long *__restrict__ last_path) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t c = k < P.n_paths ? counts[k] : 0u;
  const unsigned long long excl =
      block_off[blockIdx.x] + block_exclusive<8>((unsigned long long)c | ((unsigned long long)(c ? 1u : 0u) << 40));
  if (c == 0) return;
  const unsigned long long first = P.slot_base + (excl & ((1ull << 40) - 1ull));
  const uint32_t pid = P.path_id_base + (uint32_t)(excl >> 40);
  if (first >= P.n_total) return;
  walk_path<Scene, KIND, true>(P, P.path_base + k, first, pid);
  if (first + c >= P.n_total) last_path[0] = P.path_base + k + 1ull;   // exactly one path crosses the end of the set
}

// ---- photon planes from photon beams ------------------------------------------------------------------------------------
// One thread per beam.  w0 / length0 are PhotonBeam::setEndPoint's (as k_pack_beams forms them); length1 and w1 are
// LTPhotonPlane::transformBeam's free-flight distance and phase-function direction (host mirror
// gvpm_host::transformBeam), drawn from PCG32(seed ^ kPlaneSeed, beam index) instead of the integrator's one sequential
// sampler (DESIGN.md §6).  kPlaneSeed is the constant of gvpm_synth_planes' sampler: a caller that passes the seed of
// the light paths again does not get the light paths' random numbers.
constexpr unsigned long long kPlaneSeed = 0xA0761D6478BD642FULL;
__global__ void __launch_bounds__(256) k_planes_from_beams(const __grid_constant__ PlaneGenParams P) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  const size_t i3 = 3 * (size_t)i;
  const float o0 = P.beams.origin[i3], o1 = P.beams.origin[i3 + 1], o2 = P.beams.origin[i3 + 2];
  // PhotonBeam::setEndPoint (beams_struct.h:73-81), operation for operation as k_pack_beams
  float d0 = __fsub_rn(P.beams.end[i3], o0), d1 = __fsub_rn(P.beams.end[i3 + 1], o1), d2 = __fsub_rn(P.beams.end[i3 + 2], o2);
  const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2)));
  const float rcp = __fdiv_rn(1.0f, len);
  d0 = __fmul_rn(d0, rcp); d1 = __fmul_rn(d1, rcp); d2 = __fmul_rn(d2, rcp);
  const v3 dir(d0, d1, d2);
  Pcg32 rng(P.seed ^ kPlaneSeed, i);
  // sampleDistance, EDistanceNormal, mint = Epsilon (homogeneous.cpp:293-352); sampling_weight is 1 (checked by the caller)
  const sf eps(1e-4f);
  const sf rand(rng.uniform());
  const sf length1 = (-sf(pm_log((sf(1.f) - rand).v))) / sf(P.sigma_t1) + eps;
  v3 w1;
  for (;;) {
    const float sx = rng.uniform(), sy = rng.uniform();
    if (P.phase_type == GVPM_PHASE_ISOTROPIC) {   // squareToUniformSphere (warp.cpp:25-31)
      const sf z = sf(1.f) - sf(2.f) * sf(sy);
      const sf r = safe_sqrt(sf(1.f) - z * z);
      float sn, cs;
      pm_sincos2pi(sx, sn, cs);
      w1 = v3(r * sf(cs), r * sf(sn), z);
    } else {                                      // hg.cpp:73-96 in FrameCoherent(dir)
      const sf g(P.hg_g);
      sf cosTheta;
      if (fabsf(g.v) < eps.v) {
        cosTheta = sf(1.f) - sf(2.f) * sf(sx);
      } else {
        const sf sq = (sf(1.f) - g * g) / ((sf(1.f) - g) + (sf(2.f) * g) * sf(sx));
        cosTheta = ((sf(1.f) + g * g) - sq * sq) / (sf(2.f) * g);
      }
      const sf sinTheta = safe_sqrt(sf(1.f) - cosTheta * cosTheta);
      float sn, cs;
      pm_sincos2pi(sy, sn, cs);
      const sf lx = sinTheta * sf(cs), ly = sinTheta * sf(sn), lz = cosTheta;
      // coordinateSystemCoherent (util.cpp:592-599)
      const sf sign(copysignf(1.0f, d2));
      const sf a = sf(-1.0f) / (sign + dir.z);
      const sf b = (dir.x * dir.y) * a;
      const v3 s(sf(1.f) + ((sign * dir.x) * dir.x) * a, sign * b, (-sign) * dir.x);
      const v3 t(b, sign + (dir.y * dir.y) * a, -dir.y);
      w1 = (s * lx + t * ly) + dir * lz;
    }
    if (fabsf(dot(dir, w1).v) != 1.0f) break;   // a direction parallel to the beam spans no plane
  }
  put3(P.origin, i, v3(o0, o1, o2));
  put3(P.w0, i, dir);
  P.length0[i] = len;
  put3(P.w1, i, w1);
  P.length1[i] = length1.v;
  P.flux[i3] = P.beams.flux[i3]; P.flux[i3 + 1] = P.beams.flux[i3 + 1]; P.flux[i3 + 2] = P.beams.flux[i3 + 2];
  P.edge_id[i] = (int32_t)P.beams.depth[i];
}

// ---- G-VPM camera distance samples ----------------------------------------------------------------------------------
// computeVolumeGradientPhoton's draws (gvpm.cpp:1141-1175) for a ray that is its gather point's only medium edge
// (pdfSel = 1): nb uniforms, stratified or not, each turned into a distance by HomogeneousMedium::sampleDistance with
// EDistanceAlwaysValid and the balance strategy (homogeneous.cpp:293-430), in gvpm_synth_vpm_samples' operation order.
// Ray r draws from PCG32(seed ^ kVpmSeed, r), the synth's stream.  EMIT = false: returns the number of samples the ray
// keeps.  EMIT = true: also stores them at slots first, first + 1, ... of S.
constexpr unsigned long long kVpmSeed = 0xD1B54A32D192ED03ULL;
template <bool EMIT>
__device__ __forceinline__ uint32_t vpm_draws(const VpmGenParams &P, uint32_t r, uint32_t first, const SampleStaging &S) {
  const sf eps(P.epsilon), len(P.edge_len[r]);
  if (!(len > sf(4.f) * eps)) return 0u;
  const sf mint = eps, maxt = len;
  const sf density(P.sigma_t[1]);   // the sampling channel, min(int(0.5 * 3), 2) = 1
  const sf maxDist = smax((maxt - mint) - eps, sf(0.f));
  const sf norm = sf(1.f) - sf(pm_exp(((-density) * maxDist).v));
  const sf distSurf = maxt - mint;
  sf coef[3];   // sigma_t[c] / (1 - exp(-sigma_t[c] * distSurf)): pdfSuccess' normalisation of channel c
#pragma unroll
  for (int c = 0; c < 3; ++c) coef[c] = sf(P.sigma_t[c]) / (sf(1.f) - sf(pm_exp(((-sf(P.sigma_t[c])) * distSurf).v)));
  const v3 o(P.o[3 * (size_t)r], P.o[3 * (size_t)r + 1], P.o[3 * (size_t)r + 2]);
  const v3 d(P.d[3 * (size_t)r], P.d[3 * (size_t)r + 1], P.d[3 * (size_t)r + 2]);
  const float rad = P.radius_per_ray ? P.radius_per_ray[r] : P.radius;
  const sf normalization = sf(1.f) / sf((float)P.nb);
  Pcg32 rng(P.seed ^ kVpmSeed, r);
  uint32_t kept = 0;
  for (int i = 0; i < P.nb; ++i) {
    sf rand(rng.uniform());
    if (P.stratified) rand = sf((float)i) * normalization + rand * normalization;
    const sf dist = (-sf(pm_log((sf(1.f) - rand * norm).v))) / density;
    if (!(dist < distSurf)) continue;   // "failed to sample the distance": the draw is skipped
    const sf t = dist + mint;
    const v3 p = o + d * t;
    if (p.x == o.x && p.y == o.y && p.z == o.z) continue;
    // exp(-sigma_t[c] * dist) is both pdfSuccess' factor and the transmittance: (-a) * b and a * (-b) round alike
    sf tr[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) tr[c] = sf(pm_exp(((-sf(P.sigma_t[c])) * dist).v));
    sf pdf(0.f);
#pragma unroll
    for (int c = 0; c < 3; ++c) pdf = pdf + coef[c] * tr[c];
    pdf = pdf / sf(3.f);
    if (smax(tr[0], smax(tr[1], tr[2])).v < 1e-20f) tr[0] = tr[1] = tr[2] = sf(0.f);
    if (EMIT) {
      const size_t s = (size_t)first + kept;
      const_cast<uint32_t *>(S.ray)[s] = r;
      const_cast<float *>(S.t)[s] = t.v;
      float *T = const_cast<float *>(S.transmittance) + 3 * s;
      T[0] = tr[0].v; T[1] = tr[1].v; T[2] = tr[2].v;
      const_cast<float *>(S.pdf_success)[s] = pdf.v;
      const_cast<float *>(S.pdf_sel)[s] = 1.0f;
      const_cast<float *>(S.radius)[s] = rad;
    }
    ++kept;
  }
  return kept;
}
// One thread per ray, CTAs stride over tiles of 256 rays.  Count pass: samples kept per ray and per tile.
__global__ void __launch_bounds__(256) k_vpm_count(const __grid_constant__ VpmGenParams P) {
  const uint32_t tiles = (P.n_rays + 255) / 256;
  for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const uint32_t r = tile * 256 + threadIdx.x;
    uint32_t c = 0;
    if (r < P.n_rays) {
      c = vpm_draws<false>(P, r, 0u, SampleStaging{});
      P.counts[r] = c;
    }
    const uint32_t t = block_total<8>(c);
    if (threadIdx.x == 0) P.tile_tot[tile] = t;
    __syncthreads();   // block_total's shared words are written again by the next tile
  }
}
// Emit pass: the same draws, stored at the ray's offset in the staging arrays of the set of *n_total samples, so the
// samples land ray by ray, draws in ascending order, whatever the launch geometry.
__global__ void __launch_bounds__(256) k_vpm_emit(const __grid_constant__ VpmGenParams P) {
  const uint32_t tiles = (P.n_rays + 255) / 256;
  const SampleStaging S = sample_staging_at(P.staging, *P.n_total);
  for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const uint32_t r = tile * 256 + threadIdx.x;
    const uint32_t c = r < P.n_rays ? P.counts[r] : 0u;
    const uint32_t first = P.tile_tot[tile] + block_exclusive<8>(c);
    if (c) vpm_draws<true>(P, r, first, S);
    __syncthreads();   // block_exclusive's shared words are written again by the next tile
  }
}

// ---- launchers ------------------------------------------------------------------------------------------------------
template <class Params> void generate_rays(const Params &P, cudaStream_t st) {
  const int bs = P.block;
  const int blocksX = (P.cam.film_w + bs - 1) / bs, blocksY = (P.y1 - P.y0 + bs - 1) / bs;
  if (blocksX > 0 && blocksY > 0) k_generate_rays<Params><<<blocksX * blocksY, 1024, 0, st>>>(P);
}
void launch_generate_rays(const RayGenParams &P, cudaStream_t st) { generate_rays(P, st); }
void launch_generate_rays(const MeshRayGenParams &P, cudaStream_t st) { generate_rays(P, st); }
// counts: [n_paths] bytes; block_tot: [(n_paths + 255) / 256 + 1] words; totals: [0] batch total (paths << 40 | photons)
// beams: the beam emission kind (b_* arrays) instead of photons
template <class Scene>
void trace_count(const TraceParamsT<Scene> &P, bool beams, uint8_t *counts, unsigned long long *block_tot,
                 unsigned long long *totals, cudaStream_t st) {
  const uint32_t nb = (P.n_paths + 255) / 256;
  if (nb) {
    if (beams) k_trace_count<Scene, EmitKind::Beams><<<nb, 256, 0, st>>>(P, counts, block_tot);
    else k_trace_count<Scene, EmitKind::Photons><<<nb, 256, 0, st>>>(P, counts, block_tot);
  }
  k_scan_exclusive<unsigned long long, 1><<<1, 1024, 0, st>>>(block_tot, nb, totals, 0);
}
template <class Scene>
void trace_emit(const TraceParamsT<Scene> &P, bool beams, const uint8_t *counts, const unsigned long long *block_off,
                unsigned long long *last_path, cudaStream_t st) {
  const uint32_t nb = (P.n_paths + 255) / 256;
  if (!nb) return;
  if (beams) k_trace_emit<Scene, EmitKind::Beams><<<nb, 256, 0, st>>>(P, counts, block_off, last_path);
  else k_trace_emit<Scene, EmitKind::Photons><<<nb, 256, 0, st>>>(P, counts, block_off, last_path);
}
void launch_trace_count(const TraceParams &P, bool beams, uint8_t *counts, unsigned long long *block_tot,
                        unsigned long long *totals, cudaStream_t st) {
  trace_count(P, beams, counts, block_tot, totals, st);
}
void launch_trace_count(const MeshTraceParams &P, bool beams, uint8_t *counts, unsigned long long *block_tot,
                        unsigned long long *totals, cudaStream_t st) {
  trace_count(P, beams, counts, block_tot, totals, st);
}
void launch_trace_emit(const TraceParams &P, bool beams, const uint8_t *counts, const unsigned long long *block_off,
                       unsigned long long *last_path, cudaStream_t st) {
  trace_emit(P, beams, counts, block_off, last_path, st);
}
void launch_trace_emit(const MeshTraceParams &P, bool beams, const uint8_t *counts, const unsigned long long *block_off,
                       unsigned long long *last_path, cudaStream_t st) {
  trace_emit(P, beams, counts, block_off, last_path, st);
}
void launch_planes_from_beams(const PlaneGenParams &P, cudaStream_t st) {
  if (P.n) k_planes_from_beams<<<(P.n + 255) / 256, 256, 0, st>>>(P);
}
// counts: [n_rays] words; tile_tot: [(n_rays + 255) / 256 + 1] words; total: the samples kept in all (one word, which
// P.n_total of the emit pass points to)
void launch_vpm_samples(const VpmGenParams &P, uint32_t *total, int sm_count, cudaStream_t st) {
  const uint32_t tiles = (P.n_rays + 255) / 256;
  if (tiles) k_vpm_count<<<stride_grid<k_vpm_count>(sm_count, 256, P.n_rays), 256, 0, st>>>(P);
  k_scan_exclusive<uint32_t, 8><<<1, 1024, 0, st>>>(P.tile_tot, tiles, total, 0);
  if (tiles) k_vpm_emit<<<stride_grid<k_vpm_emit>(sm_count, 256, P.n_rays), 256, 0, st>>>(P);
}

}  // namespace gvpm
