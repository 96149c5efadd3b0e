// gvpm_device.cuh — device-side data layout and arithmetic helpers shared by the kernels.
//
// Arithmetic policy (DESIGN.md §4): everything that decides WHICH photons a ray gathers or WHICH
// shift branch is taken (neighbour predicate, kernel-chord sampling, null-shift / mirror tests,
// reconnection geometry, visibility, side tests) is computed with the explicitly rounded
// intrinsics (__fadd_rn, __fmul_rn, ...) in the reference's operation order, so nvcc can neither
// contract them into FMAs nor reassociate them and the index sets are bit-identical to a
// -ffp-contract=off CPU evaluation.  The wrapper type `sf` makes that readable.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gvpm_b200.h"

namespace gvpm {

// ---- strictly rounded float -------------------------------------------------------------
struct sf {
  float v;
  __host__ __device__ sf() : v(0.f) {}
  __host__ __device__ sf(float x) : v(x) {}
};
__device__ __forceinline__ sf operator+(sf a, sf b) { return sf(__fadd_rn(a.v, b.v)); }
__device__ __forceinline__ sf operator-(sf a, sf b) { return sf(__fsub_rn(a.v, b.v)); }
__device__ __forceinline__ sf operator*(sf a, sf b) { return sf(__fmul_rn(a.v, b.v)); }
__device__ __forceinline__ sf operator/(sf a, sf b) { return sf(__fdiv_rn(a.v, b.v)); }
__device__ __forceinline__ sf operator-(sf a) { return sf(-a.v); }
__device__ __forceinline__ bool operator<(sf a, sf b) { return a.v < b.v; }
__device__ __forceinline__ bool operator>(sf a, sf b) { return a.v > b.v; }
__device__ __forceinline__ bool operator<=(sf a, sf b) { return a.v <= b.v; }
__device__ __forceinline__ bool operator>=(sf a, sf b) { return a.v >= b.v; }
__device__ __forceinline__ bool operator==(sf a, sf b) { return a.v == b.v; }
// radiometric-only quotients (never feed a decision): MUFU.RCP + FMUL, 2 ulp — the 1e-4 radiance bar is 3 orders
// of magnitude above that; __fdiv_rn costs ~8 instructions + a slow path
__device__ __forceinline__ sf fdiv(sf a, sf b) { return sf(__fdividef(a.v, b.v)); }
__device__ __forceinline__ sf frcp(sf a) { return sf(__fdividef(1.f, a.v)); }
__device__ __forceinline__ sf ssqrt(sf a) { return sf(__fsqrt_rn(a.v)); }
__device__ __forceinline__ sf smax(sf a, sf b) { return sf(fmaxf(a.v, b.v)); }
__device__ __forceinline__ sf safe_sqrt(sf a) { return ssqrt(smax(sf(0.f), a)); }

// __fdiv_rn(a, b) < 0 without the division, for |b| < 2 (the side tests' b is a dot product of two unit vectors, so
// |b| <= 1 + rounding).  The quotient is negative exactly when a and b have opposite sign bits and it is neither NaN nor
// a zero:
//   a = +-0 gives +-0 or NaN (b = +-0) and a = NaN or b = NaN gives NaN: excluded by |a| > 0 and |b| < inf;
//   b = +-inf gives +-0 or NaN: excluded by |b| < inf;
//   b = +-0 with a != 0 gives +-inf, whose sign is the xor of the sign bits (-0 counts as negative), as here;
//   a = +-inf with b finite gives +-inf, likewise;
//   finite nonzero a over finite b with |b| < 2 has |a / b| > 2^-149 / 2, so it rounds to a nonzero value of that sign.
__host__ __device__ __forceinline__ bool quotient_negative(float a, float b) {
  return fabsf(a) > 0.f && fabsf(b) < INFINITY && (signbit(a) != signbit(b));
}

struct v3 {
  sf x, y, z;
  __device__ v3() {}
  __device__ v3(sf a, sf b, sf c) : x(a), y(b), z(c) {}
  __device__ v3(float a, float b, float c) : x(a), y(b), z(c) {}
};
__device__ __forceinline__ v3 operator+(v3 a, v3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ v3 operator-(v3 a, v3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ v3 operator-(v3 a) { return v3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ v3 operator*(v3 a, sf f) { return v3(a.x * f, a.y * f, a.z * f); }
__device__ __forceinline__ v3 operator*(sf f, v3 a) { return v3(a.x * f, a.y * f, a.z * f); }
__device__ __forceinline__ v3 operator*(v3 a, v3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
// vector / scalar multiplies by the reciprocal (include/mitsuba/core/vector.h:535-542)
__device__ __forceinline__ v3 operator/(v3 a, sf f) { sf r = sf(1.f) / f; return v3(a.x * r, a.y * r, a.z * r); }
__device__ __forceinline__ sf dot(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ v3 cross(v3 a, v3 b) {
  return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ sf length_sq(v3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
__device__ __forceinline__ sf length(v3 a) { return ssqrt(length_sq(a)); }
__device__ __forceinline__ v3 normalize(v3 a) { return a / length(a); }
__device__ __forceinline__ sf max3(v3 a) { return smax(a.x, smax(a.y, a.z)); }

#define GVPM_INV_PI 0.31830988618379067154f
#define GVPM_INV_FOURPI 0.07957747154594766788f
#define GVPM_PI 3.14159265358979323846f

// ---- device record layout (DESIGN.md §3) -----------------------------------------------------
// Photons: one 128-byte record (8 float4) per photon in the caller's order (`aos`), plus the Morton-sorted
// plane P0 (`planes`) the traversal reads and `orig` (sorted slot -> caller index).
//   A0 = pos.xyz,           meta bits   (P0 is the sorted copy of this field)
//   A1 = flux.xyz,          parent_pdf
//   A2 = parent_pos.xyz,    edge_pdf
//   A3 = wiW.xyz,           rr_weight   wiW = normalize(pred_pos - parent_pos)
//   A4 = parent_n.xyz,      cosI        cosI = dot(parent_n, wiW)
//   A5 = prefix_flux.xyz,   nEdge       nEdge = dot(parent_n, -wi)
//   A6 = parent_albedo.xyz, lBase       lBase = length(pos - parent_pos)
//   A7 = whole-set index (bits; dispatched records only, else 0), wi.xyz   wi = normalize(parent_pos - pos)
// wiW, cosI, nEdge, lBase and wi depend on the photon alone: photon_record computes them once, so the shading does
// not repeat them for every (ray, photon) pair.  The predecessor position itself is not kept.
// meta: bits 0-1 parent type, bits 2-9 depth, bit 10 pathID & 1.
#define GVPM_PLANE_PLANES 6  // float4 planes per photon-plane record (plane_device.cuh)
__host__ __device__ inline uint32_t pack_meta(uint32_t type, uint32_t depth, uint32_t path_id) {
  return (type & 3u) | ((depth & 255u) << 2) | ((path_id & 1u) << 10);
}
// Writes the record of one photon to r[0..7] (shared or global memory), from its fields.  The derived terms use the
// strictly rounded operations, in the order the shading evaluated them per pair, so the stored bits are those values.
__device__ __forceinline__ void photon_record(float4 *r, v3 pos, uint32_t meta, v3 flux, sf parentPdf, v3 parent,
                                              sf edgePdf, v3 pred, sf rrW, v3 pn, v3 prefix, v3 albedo,
                                              uint32_t wholeIndex) {
  const v3 wiW = normalize(pred - parent);
  const sf cosI = dot(pn, wiW);
  const v3 wi = normalize(parent - pos);
  // normalize(pos - parent) == -wi bit for bit (negation commutes with every rounding involved)
  const sf nEdge = dot(pn, -wi);
  const sf lBase = length(pos - parent);
  r[0] = make_float4(pos.x.v, pos.y.v, pos.z.v, __uint_as_float(meta));
  r[1] = make_float4(flux.x.v, flux.y.v, flux.z.v, parentPdf.v);
  r[2] = make_float4(parent.x.v, parent.y.v, parent.z.v, edgePdf.v);
  r[3] = make_float4(wiW.x.v, wiW.y.v, wiW.z.v, rrW.v);
  r[4] = make_float4(pn.x.v, pn.y.v, pn.z.v, cosI.v);
  r[5] = make_float4(prefix.x.v, prefix.y.v, prefix.z.v, nEdge.v);
  r[6] = make_float4(albedo.x.v, albedo.y.v, albedo.z.v, lBase.v);
  r[7] = make_float4(__uint_as_float(wholeIndex), wi.x.v, wi.y.v, wi.z.v);
}

// Rays: 5 records of 64 B per ray (4 float4 each): base + offsets L,R,T,B.
//   base: q0 = o.xyz, mint | q1 = d.xyz, maxt | q2 = eye.xyz, edge_len | q3 = xi, px, py, edge_id (bits)
//   off : q0 = o.xyz, len  | q1 = d.xyz, sensor | q2 = eye.xyz, valid (bits) | q3 = unused
#define GVPM_RAY_FLOAT4 20

// raw staging layout: element offsets of each SoA array inside one contiguous device buffer
struct PhotonStaging {
  const float *pos, *flux, *parent_pos, *pred_pos, *parent_n, *prefix_flux, *parent_albedo;
  const float *parent_pdf, *edge_pdf, *rr_weight;
  const uint8_t *parent_type, *depth;
  const uint32_t *path_id;
};
// photon_record of photon s of the staging arrays
__device__ __forceinline__ void photon_record(float4 *r, const PhotonStaging &S, size_t s, uint32_t wholeIndex) {
  const size_t s3 = 3 * s;
  auto ld3 = [&](const float *p) { return v3(__ldg(p + s3), __ldg(p + s3 + 1), __ldg(p + s3 + 2)); };
  photon_record(r, ld3(S.pos), pack_meta(S.parent_type[s], S.depth[s], S.path_id[s]), ld3(S.flux),
                sf(__ldg(S.parent_pdf + s)), ld3(S.parent_pos), sf(__ldg(S.edge_pdf + s)), ld3(S.pred_pos),
                sf(__ldg(S.rr_weight + s)), ld3(S.parent_n), ld3(S.prefix_flux), ld3(S.parent_albedo), wholeIndex);
}
struct RayStaging {
  const float *o, *d, *mint, *maxt, *edge_len, *eye_contrib, *xi;
  const int32_t *px, *py, *edge_id;
  const uint8_t *off_valid;
  const float *off_o, *off_d, *off_len, *off_eye, *off_sensor;
};

struct BeamStaging {   // raw gvpm_beam_soa arrays on the device
  const float *origin, *end, *flux, *prefix_flux, *parent_n, *parent_albedo, *pred_pos, *end_n, *parent_pdf, *rr_weight;
  const uint8_t *parent_type, *end_on_surface, *depth;
  const uint32_t *path_id;
};
struct PlaneStaging {  // raw gvpm_plane_soa arrays on the device
  const float *origin, *w0, *length0, *w1, *length1, *flux;
  const int32_t *edge_id;
};
struct SampleStaging { // raw gvpm_vpm_sample_soa arrays on the device
  const uint32_t *ray;
  const float *t, *transmittance, *pdf_success, *pdf_sel, *radius;
};
// The sample staging arrays of a set of n samples inside one buffer, laid out as capi_internal.cuh's SoaLayout<SampleSoA>
// lays them out (element sizes 4, 4, 12, 4, 4, 4 bytes, each array on a 256-byte boundary).  For kernels that learn n
// on the device (the samples gvpm_generate_vpm_samples draws).
__host__ __device__ __forceinline__ SampleStaging sample_staging_at(const void *base, uint32_t n) {
  const size_t a4 = (4 * (size_t)n + 255) & ~(size_t)255, a12 = (12 * (size_t)n + 255) & ~(size_t)255;
  const char *b = (const char *)base;
  SampleStaging S;
  S.ray = (const uint32_t *)b;
  S.t = (const float *)(b + a4);
  S.transmittance = (const float *)(b + 2 * a4);
  S.pdf_success = (const float *)(b + 2 * a4 + a12);
  S.pdf_sel = (const float *)(b + 3 * a4 + a12);
  S.radius = (const float *)(b + 4 * a4 + a12);
  return S;
}

// implicit 32-ary hierarchy over Morton-sorted photons: level 0 = leaves of 32 photons,
// level l+1 node j = union of level l nodes [32j, 32j+32).  Boxes already inflated by the radius
// (+ conservative pad).  lo/hi: float4 arrays holding all levels, level l starts at off[l].
#define GVPM_MAX_LEVELS 8
struct Tree {
  const float4 *lo, *hi;
  uint32_t off[GVPM_MAX_LEVELS];
  uint32_t cnt[GVPM_MAX_LEVELS];
  int levels;       // number of levels; the top level has <= 32 nodes
  uint32_t n;       // photons
};

// Perspective ("frustum") grid over the photons, for ray sets whose supporting lines all pass through one point C
// (primary camera rays of a pinhole sensor: every medium segment of a pixel's first edge).  Directions from C are
// projected on the plane at distance 1 along the mean ray direction m (gnomonic projection, basis u, v); a photon at
// distance rho from C can only be a neighbour of rays whose projected direction lies within
//   w = tan(theta + alpha) - tan(theta),  alpha = asin((r + delta) / rho),  tan(theta) = |proj(photon)|
// of its own projection (delta = largest distance of C to a ray's line).  Photons are binned by FOOTPRINT CLASS c
// (w <= cell * 2^c) into a grid coarsened by 2^c, so that a ray finds every neighbour in the 3x3 cells around its own
// cell of every class; photons whose footprint exceeds the coarsest class go to the NEAR bucket (tested by every ray),
// photons that no ray can reach (no ray in the 3x3 cells around them) are DROPPED.  cell_start[k] = first sorted slot with key >= k.
#define GVPM_GRID_CLASSES 16
struct FrustumGrid {
  float C[3], m[3], u[3], v[3];
  float gx0, gy0;                        // plane coordinates of the grid origin
  float csize[GVPM_GRID_CLASSES];        // cell edge of class c = csize[0] * 2^c
  float xmin, xmax, ymin, ymax;          // bounds of the rays' projected directions
  float pad_r;                           // r + delta
  uint32_t nx[GVPM_GRID_CLASSES], ny[GVPM_GRID_CLASSES], base[GVPM_GRID_CLASSES];
  uint32_t n_cells;                      // cells of ONE grid (all classes)
  int classes;
  int parity_split;                      // 1: two grids, photons with even / odd pathID (the pathSet checkerboard pairs a
                                         // photon with pixels of its own parity only: half the candidates per ray);
                                         // key = parity * n_cells + cell.  NEAR = grids * n_cells, DROP = NEAR + 1
};

struct GatherParams {
  Tree tree;
  // frustum-grid variant of the point gather (tree_build.cu / gather_bre.cu k_bre_grid_traverse)
  FrustumGrid grid;
  const uint32_t *cell_start;   // [grids * n_cells + 3]
  const uint32_t *build_ovf;    // frustum build over a dispatched inbox: set when a peer's dispatch timed out or overflowed
  const float4 *planes;  // [n] sorted P0 = pos.xyz, meta (the only per-photon data the traversal reads)
  const float4 *aos;     // [n][8] full records in the caller's order (shading reads aos[orig[slot]])
  const uint32_t *orig;  // [n] original photon index of sorted slot
  const float4 *rays;    // [n_rays][20]
  uint32_t n_rays;
  float radius, radius_sq, kernel_vol;
  const float *bounds;  // device: photon AABB min[3], max[3], max |coordinate| (cull pad)
  // medium
  float sigma_s[3], sigma_t[3];
  int phase_type;
  float hg_g, sampling_weight;
  gvpm_config cfg;
  const float *tri;  // [n_tri*9]
  const float4 *tri_plane;  // [n_tri] unit plane (n, d) for the conservative cull
  const float2 *tri_aux;    // [n_tri] (rounding-slack coefficient, largest |vertex coordinate|)
  uint32_t n_tri;
  // outputs
  float *out;        // [n_rays*27]
  uint32_t *counts;  // [n_rays*2] or null
  // neighbour dump (parity aid)
  const uint64_t *nbr_offsets;
  uint32_t *nbr_idx;
  uint32_t *work_counter;
  // traversal -> shading hand-off: (ray index, sorted photon slot) pairs
  uint32_t ray_begin, ray_end;        // ray range of this launch
  uint2 *pairs;
  unsigned long long pair_cap;
  unsigned long long *pair_counter;   // pairs emitted (may exceed pair_cap: overflow)
  float packet_spread_max;            // packets wider than this are traversed ray by ray
  // G-VPM distance samples: 2 float4 per sample
  //   s0 = t, pdf_success, pdf_sel, radius | s1 = transmittance.xyz, ray index (bits)
  const float4 *samples;
  uint32_t n_samples;
  uint32_t *sample_counts;            // [n_samples*2] found / contributing, or null
  uint32_t *mvol;                     // [n_rays] sum of `found` over the ray's samples, or null
  float vpm_normalization;            // 1 / nbCameraSamples
  // G-Beams: 8 float4 per beam (DESIGN.md §3), sub-beam records sorted in Morton order (tree = hierarchy
  // over sub-beams): sub[i] = t1, t2, beam index (bits), flags (bit 0 first, bit 1 last sub-beam)
  const float4 *beams;
  const float4 *subs;
  uint32_t n_beams;
  float weight_kernel;                // 1.0 / kernelVol (double division rounded to Float)
  int sppm_beam_technique;            // gvpm_beam_technique of k_beam_shade_sppm (sppm primal beams)
  int beam_prefilter;                 // apply the depth/mode/pathSet filters already in the traversal
                                      // (when the caller does not ask for the geometric neighbour counts)
  // G-Planes: 6 float4 planes of n_planes entries in Morton order (plane_device.cuh), tree.lo/hi = leaf boxes
  const float4 *plane_rec;
  const uint32_t *plane_orig;         // [n_planes] caller's plane index of sorted slot
  uint32_t n_planes;
  // parity dump for beams: flat list of (ray, beam | contributes << 31) + its atomic cursor
  uint2 *dump_pairs;
  unsigned long long *dump_counter;
  unsigned long long dump_cap;
  // occluder BVH (occluder_device.cuh): GVPM_OCC_NODE_FLOAT4 float4 per node; null when the shadow rays use the list
  const float4 *occ_nodes;
  uint32_t n_occ_nodes;
};

// ---- photon dispatch between ranks (dispatch.cu) -----------------------------------------------------------------------
struct DispatchParams {
  PhotonStaging S;                 // this rank's staging arrays (whole-set layout)
  uint32_t begin, count;           // the slice [begin, begin + count) is dispatched
  int n_dst;
  FrustumGrid grids[GVPM_MAX_PEERS];   // the receivers' grids, by value: kernel parameters live in the constant bank, and
                                       // every thread reads the same field of the same grid at the same time
  const uint32_t *occ[GVPM_MAX_PEERS];   // local copies of the receivers' occupancy masks
  float4 *inbox[GVPM_MAX_PEERS];   // receiver d's inbox region of THIS sender (peer-mapped; local for d = self)
  uint32_t region_cap;             // records per region
  uint8_t *keepbits;               // [count]
  uint32_t *block_cnt;             // [n_dst][nb + 1]: counts, then exclusive offsets (+ total at [nb])
  uint32_t nb;
  unsigned *overflow;              // set when a region would overflow (cannot happen with region_cap >= count)
  // shared projection plane (all receivers use the frame of grids[0]): one classification per photon against the owner map
  const uint8_t *owner_map;        // kOccRes x kOccRes cells over [ux0, ux1] x [uy0, uy1], bit d = receiver d has rays there
  float ux0, uy0, ux1, uy1, uix, uiy;   // bounds, cells per unit
  float pad_r_max;                 // largest r + delta of the receivers (+ the slack for their slightly different centres)
};

struct SignalParams {
  int n_dst, self;
  uint32_t nb;
  const uint32_t *block_cnt;
  uint32_t *count_dst[GVPM_MAX_PEERS];   // receiver d's count word of THIS sender
  uint32_t *flag_dst[GVPM_MAX_PEERS];    // receiver d's "pushed" flag of THIS sender
  uint32_t gen;
};
struct FlagSetParams { int n; uint32_t value; uint32_t *dst[GVPM_MAX_PEERS]; };

// ---- on-device generators (generate.cu) -------------------------------------------------------------------------------
// The mesh scene of gvpm_set_trace_mesh on the device.  The triangles, their planes and slack terms (as the occluders'
// tri_plane / tri_aux) and the albedos are in the leaf order of the scene's BVH (occluder_device.cuh layout); perm maps
// a leaf-order slot to the caller's triangle index.  The emissive triangles are kept apart, in the caller's order.
struct MeshScene {
  const float *tri;
  const float4 *plane;
  const float2 *aux;
  const float *albedo;
  const uint32_t *perm;
  const float4 *nodes;
  uint32_t n_tri, n_nodes;
  const float *emit_tri;        // [n_emit*9]
  const uint32_t *emit_idx;     // [n_emit] caller's triangle index
  const float *emit_cdf;        // [n_emit] fp32 running sum of the areas, in index order
  uint32_t n_emit, emit_last;   // emit_last: the last emissive triangle of non-zero area
  float emit_total;             // emit_cdf[n_emit - 1]
  float lo[3], hi[3];
  // the box grown by 2e-6 of its extent on each axis (twice the tolerance of gvpm_set_trace_mesh): every triangle lies
  // inside it, so a triangle on a face of the box is found whatever the rounding of its parameter and of the exit's
  float glo[3], ghi[3];
  float light_power;
};
// gvpm_lookat_camera with its frame (right, up, forward: capi_rays.cu forms it) and the field names of
// gvpm_pinhole_camera that k_generate_rays reads
struct LookatCam {
  float pos[3], r[3], u[3], f[3];
  float tan_half_fov_x;
  int32_t film_w, film_h;
  int32_t inside_medium;
};
template <class Scene, class Cam> struct RayGenParamsT {
  Scene scene;
  Cam cam;
  unsigned long long seed;
  int block, zorder, y0, y1;
  float epsilon;
  // ray staging arrays (gvpm_ray_soa order)
  float *o, *d, *mint, *maxt, *edge_len, *eye_contrib, *xi;
  int32_t *px, *py, *edge_id;
  uint8_t *off_valid;
  float *off_o, *off_d, *off_len, *off_eye, *off_sensor;
};
using RayGenParams = RayGenParamsT<gvpm_box_scene, gvpm_pinhole_camera>;
using MeshRayGenParams = RayGenParamsT<MeshScene, LookatCam>;
template <class Scene> struct TraceParamsT {
  Scene scene;
  float sigma_s, sigma_a, hg_g;
  int phase_type, max_depth, rr_depth, min_depth;
  unsigned long long seed, path_base;
  uint32_t n_paths;             // paths of this batch
  // emit pass
  unsigned long long slot_base; // photons stored by earlier batches
  uint32_t path_id_base;        // contributing paths of earlier batches
  unsigned long long n_total;   // capacity (photons wanted)
  // staging arrays (gvpm_photon_soa order)
  float *pos, *flux, *parent_pos, *pred_pos, *parent_n, *prefix_flux, *parent_albedo, *parent_pdf, *edge_pdf, *rr_weight;
  uint8_t *parent_type, *depth;
  uint32_t *path_id;
  float4 *aos;                  // not null: write 128-byte gather records (layout above) instead of the staging arrays
  // beam staging arrays (gvpm_beam_soa order), written by the beam emission kind
  float *b_origin, *b_end, *b_flux, *b_prefix_flux, *b_parent_n, *b_parent_albedo, *b_pred_pos, *b_end_n, *b_parent_pdf,
      *b_rr_weight;
  uint8_t *b_parent_type, *b_end_on_surface, *b_depth;
  uint32_t *b_path_id;
};
using TraceParams = TraceParamsT<gvpm_box_scene>;
using MeshTraceParams = TraceParamsT<MeshScene>;
// photon planes from the current beam set (generate.cu k_planes_from_beams): one PCG32 stream per beam
struct PlaneGenParams {
  BeamStaging beams;
  uint32_t n;
  unsigned long long seed;
  float sigma_t1, hg_g;         // sampling density sigma_s[1] + sigma_a[1] (balance strategy); HG asymmetry
  int phase_type;
  // plane staging arrays (gvpm_plane_soa order)
  float *origin, *w0, *length0, *w1, *length1, *flux;
  int32_t *edge_id;
};
// G-VPM camera distance samples from the current ray set (generate.cu k_vpm_count / k_vpm_emit): one PCG32 stream per ray
struct VpmGenParams {
  const float *o, *d, *edge_len;   // ray staging arrays
  const float *radius_per_ray;     // [n_rays], or null: `radius` for every ray
  uint32_t n_rays;
  int nb, stratified;
  unsigned long long seed;
  float epsilon, radius;
  float sigma_t[3];
  uint32_t *counts;                // [n_rays] samples kept per ray (count pass writes, emit pass reads)
  uint32_t *tile_tot;              // [tiles + 1] samples per tile of 256 rays, scanned in place into tile offsets
  const uint32_t *n_total;         // device: samples kept in all (the scan's total; the emit pass's staging layout)
  void *staging;                   // the sample staging buffer
};
// ---- strictly rounded double (the reference's fp64 island: cylinderIntersection / solveQuadraticDouble,
// photonmapper/beams_3d_intersections.h:100-137, src/libcore/util.cpp:487-525) ----------------------------
struct sd {
  double v;
  __host__ __device__ sd() : v(0.0) {}
  __host__ __device__ sd(double x) : v(x) {}
};
__device__ __forceinline__ sd operator+(sd a, sd b) { return sd(__dadd_rn(a.v, b.v)); }
__device__ __forceinline__ sd operator-(sd a, sd b) { return sd(__dsub_rn(a.v, b.v)); }
__device__ __forceinline__ sd operator*(sd a, sd b) { return sd(__dmul_rn(a.v, b.v)); }
__device__ __forceinline__ sd operator/(sd a, sd b) { return sd(__ddiv_rn(a.v, b.v)); }
__device__ __forceinline__ sd dsqrt(sd a) { return sd(__dsqrt_rn(a.v)); }

#ifndef GVPM_PACKET
#define GVPM_PACKET 4  // camera rays per traversal warp
#endif

}  // namespace gvpm
