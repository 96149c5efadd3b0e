// occluder_bvh.cu — device build of the occluder BVH that the reconnection shadow rays walk (occluder_device.cuh) when the
// occluder set is large: Hilbert keys of the triangle centroids (tree_build.cu's bounds and key kernels) -> radix sort
// -> triangles permuted into key order -> a binary radix tree over groups of GVPM_OCC_LEAF consecutive triangles
// (Karras, "Maximizing parallelism in the construction of BVHs, octrees and k-d trees", HPG 2012; equal keys are told
// apart by the leaf index) -> depth-first node positions -> boxes, normal cones and slack bounds bottom-up, the second
// child to arrive at a node building it.  Replaces the reference's kd-tree over the scene's meshes for this one query
// (scene->rayIntersect, shift_volume_photon.cpp:396-402).
#include "capi_internal.cuh"
#include "bre_device.cuh"

namespace gvpm {

namespace {
constexpr uint32_t kNone = 0xffffffffu;
constexpr float kHalfPi = 1.5707963f;

__global__ void k_occ_centroids(const float *__restrict__ tri, uint32_t n, float *__restrict__ cen) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float *p = tri + 9 * (size_t)i;
#pragma unroll
  for (int a = 0; a < 3; ++a) cen[3 * (size_t)i + a] = (p[a] + p[3 + a] + p[6 + a]) * (1.f / 3.f);
}

// triangle arrays into key order
__global__ void k_occ_permute(const uint32_t *__restrict__ sorted, uint32_t n, const float *__restrict__ tri,
                              const float4 *__restrict__ plane, const float2 *__restrict__ aux, float *__restrict__ tri_o,
                              float4 *__restrict__ plane_o, float2 *__restrict__ aux_o) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = sorted[i];
#pragma unroll
  for (int a = 0; a < 9; ++a) tri_o[9 * (size_t)i + a] = tri[9 * (size_t)s + a];
  plane_o[i] = plane[s];
  aux_o[i] = aux[s];
}

// common prefix of the (key, index) pairs of leaves i and j; -1 outside [0, nL)
__device__ __forceinline__ int occ_delta(const uint32_t *keys, uint32_t nL, int i, int j) {
  if (j < 0 || j >= (int)nL) return -1;
  const unsigned long long a = ((unsigned long long)keys[(size_t)i * GVPM_OCC_LEAF] << 32) | (uint32_t)i;
  const unsigned long long b = ((unsigned long long)keys[(size_t)j * GVPM_OCC_LEAF] << 32) | (uint32_t)j;
  return __clzll(a ^ b);
}

// inner node i of the radix tree over nL leaves: its leaf range [first, last], split (left child ends at split) and
// the parent links of its two children
__global__ void k_occ_karras(const uint32_t *__restrict__ keys, uint32_t nL, uint32_t *__restrict__ first,
                             uint32_t *__restrict__ last, uint32_t *__restrict__ split, uint32_t *__restrict__ parent,
                             uint32_t *__restrict__ leaf_parent) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= (int)nL - 1) return;
  const int d = occ_delta(keys, nL, i, i + 1) > occ_delta(keys, nL, i, i - 1) ? 1 : -1;
  const int dmin = occ_delta(keys, nL, i, i - d);
  int lmax = 2;
  while (occ_delta(keys, nL, i, i + lmax * d) > dmin) lmax *= 2;
  int l = 0;
  for (int t = lmax / 2; t >= 1; t /= 2)
    if (occ_delta(keys, nL, i, i + (l + t) * d) > dmin) l += t;
  const int j = i + l * d;
  const int dnode = occ_delta(keys, nL, i, j);
  int s = 0;
  for (int div = 2;; div *= 2) {
    const int t = (l + div - 1) / div;
    if (occ_delta(keys, nL, i, i + (s + t) * d) > dnode) s += t;
    if (t <= 1) break;
  }
  const int gamma = i + s * d + min(d, 0);
  const int lo = min(i, j), hi = max(i, j);
  first[i] = lo; last[i] = hi; split[i] = gamma;
  if (lo == gamma) leaf_parent[gamma] = i; else parent[gamma] = i;
  if (hi == gamma + 1) leaf_parent[gamma + 1] = i; else parent[gamma + 1] = i;
}

// depth-first position of every node (inner 0 .. nL-2, then the leaves): the sum, over the path to the root, of 1 for a
// left child and 1 + (nodes of the left sibling's subtree) = 2 * (leaves left of the split) for a right child
__global__ void k_occ_pos(uint32_t nL, const uint32_t *__restrict__ first, const uint32_t *__restrict__ split,
                          const uint32_t *__restrict__ parent, const uint32_t *__restrict__ leaf_parent,
                          uint32_t *__restrict__ pos_inner, uint32_t *__restrict__ pos_leaf) {
  const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t nI = nL - 1;
  if (x >= nI + nL) return;
  const bool leaf = x >= nI;
  uint32_t f = leaf ? x - nI : first[x];
  uint32_t p = leaf ? leaf_parent[x - nI] : parent[x];
  uint32_t pos = 0;
  while (p != kNone) {
    const uint32_t pf = first[p];
    pos += f == pf ? 1u : 2u * (split[p] - pf + 1u);
    f = pf;
    p = parent[p];
  }
  if (leaf) pos_leaf[x - nI] = pos; else pos_inner[x] = pos;
}

// Normal cones: every normal (either sign) below a node lies within phi of +-axis; phi >= pi/2 is "no bound".  Angles
// come from atan2 (accurate to a few ulp, unlike acos near 1); every merge widens by 1e-6 rad for their rounding.
struct OccCone { float x, y, z, phi; };
__device__ __forceinline__ OccCone cone_none() { return OccCone{0.f, 0.f, 1.f, 2.f}; }
__device__ __forceinline__ float cone_angle(float ax, float ay, float az, float bx, float by, float bz) {
  const float cx = ay * bz - az * by, cy = az * bx - ax * bz, cz = ax * by - ay * bx;
  return atan2f(sqrtf(cx * cx + cy * cy + cz * cz), ax * bx + ay * by + az * bz);
}
__device__ __forceinline__ OccCone cone_of_plane(float4 pl) {
  const float l = sqrtf(pl.x * pl.x + pl.y * pl.y + pl.z * pl.z);
  if (!(l > 0.5f)) return cone_none();   // zero-area triangle (no plane): never culled on geometry
  return OccCone{pl.x / l, pl.y / l, pl.z / l, 1e-6f};
}
__device__ __forceinline__ OccCone cone_merge(OccCone A, OccCone B) {
  if (!(A.phi < kHalfPi) || !(B.phi < kHalfPi)) return cone_none();
  float dp = A.x * B.x + A.y * B.y + A.z * B.z;
  if (dp < 0.f) { B.x = -B.x; B.y = -B.y; B.z = -B.z; dp = -dp; }
  const float th = cone_angle(A.x, A.y, A.z, B.x, B.y, B.z);
  if (th + B.phi + 1e-6f <= A.phi) return A;
  if (th + A.phi + 1e-6f <= B.phi) return B;
  if (0.5f * (th + A.phi + B.phi) >= kHalfPi - 1e-3f) return cone_none();
  // axis: A's turned towards B's by half the excess, so that the cone just covers both
  OccCone C = A;
  const float px = B.x - A.x * dp, py = B.y - A.y * dp, pz = B.z - A.z * dp;
  const float pl = sqrtf(px * px + py * py + pz * pz);
  if (pl > 1e-20f) {
    const float rot = 0.5f * (th + B.phi - A.phi);
    const float c = cosf(rot), s = sinf(rot) / pl;
    C.x = A.x * c + px * s; C.y = A.y * c + py * s; C.z = A.z * c + pz * s;
    const float cl = sqrtf(C.x * C.x + C.y * C.y + C.z * C.z);
    C.x /= cl; C.y /= cl; C.z /= cl;
  }
  // whatever the axis came out as, phi covers both cones from it
  C.phi = fmaxf(cone_angle(C.x, C.y, C.z, A.x, A.y, A.z) + A.phi, cone_angle(C.x, C.y, C.z, B.x, B.y, B.z) + B.phi) + 1e-6f;
  return C.phi >= kHalfPi - 1e-3f ? cone_none() : C;
}

__device__ __forceinline__ void store_node(float4 *nodes, uint32_t pos, float lx, float ly, float lz, uint32_t word,
                                           float hx, float hy, float hz, float kappa, const OccCone &c) {
  float4 *q = nodes + (size_t)GVPM_OCC_NODE_FLOAT4 * pos;
  q[0] = make_float4(lx, ly, lz, __uint_as_float(word));
  q[1] = make_float4(hx, hy, hz, kappa);
  q[2] = make_float4(c.x, c.y, c.z, c.phi);
}

// one thread per leaf: its box, cone and kappa, then up the tree while it is the second child to arrive
__global__ void k_occ_boxes(uint32_t n, uint32_t nL, const float *__restrict__ tri, const float4 *__restrict__ plane,
                            const float2 *__restrict__ aux, const uint32_t *__restrict__ first,
                            const uint32_t *__restrict__ last, const uint32_t *__restrict__ split,
                            const uint32_t *__restrict__ parent, const uint32_t *__restrict__ leaf_parent,
                            const uint32_t *__restrict__ pos_inner, const uint32_t *__restrict__ pos_leaf,
                            uint32_t *__restrict__ arrived, float4 *nodes) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nL) return;
  const uint32_t t0 = j * GVPM_OCC_LEAF, t1 = min(t0 + GVPM_OCC_LEAF, n);
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  float kappa = 0.f;
  OccCone cone = cone_of_plane(plane[t0]);
  for (uint32_t t = t0; t < t1; ++t) {
    for (int v = 0; v < 9; ++v) {
      const float c = tri[9 * (size_t)t + v];
      lo[v % 3] = fminf(lo[v % 3], c);
      hi[v % 3] = fmaxf(hi[v % 3], c);
    }
    kappa = fmaxf(kappa, aux[t].x);
    if (t > t0) cone = cone_merge(cone, cone_of_plane(plane[t]));
  }
  store_node(nodes, pos_leaf[j], lo[0], lo[1], lo[2], GVPM_OCC_LEAF_BIT | t0, hi[0], hi[1], hi[2], kappa, cone);
  __threadfence();
  for (uint32_t p = leaf_parent[j]; p != kNone; p = parent[p]) {
    if (atomicAdd(arrived + p, 1u) == 0u) return;   // the sibling is not done yet: it continues from here
    const uint32_t pp = pos_inner[p], f = first[p];
    // both children, written by this thread or (fenced) by the sibling's: read through L2
    const float4 *L = nodes + (size_t)GVPM_OCC_NODE_FLOAT4 * (pp + 1);
    const float4 *R = nodes + (size_t)GVPM_OCC_NODE_FLOAT4 * (pp + 2u * (split[p] - f + 1u));
    const float4 l0 = __ldcg(L), l1 = __ldcg(L + 1), l2 = __ldcg(L + 2);
    const float4 r0 = __ldcg(R), r1 = __ldcg(R + 1), r2 = __ldcg(R + 2);
    const OccCone c = cone_merge(OccCone{l2.x, l2.y, l2.z, l2.w}, OccCone{r2.x, r2.y, r2.z, r2.w});
    const uint32_t escape = pp + 2u * (last[p] - f + 1u) - 1u;
    store_node(nodes, pp, fminf(l0.x, r0.x), fminf(l0.y, r0.y), fminf(l0.z, r0.z), escape, fmaxf(l1.x, r1.x),
               fmaxf(l1.y, r1.y), fmaxf(l1.z, r1.z), fmaxf(l1.w, r1.w), c);
    __threadfence();
  }
}

template <bool BVH>
__global__ void k_occluded(const __grid_constant__ GatherParams P, const float *__restrict__ o,
                           const float *__restrict__ d, const float *__restrict__ mint, const float *__restrict__ maxt,
                           uint32_t n, uint8_t *__restrict__ hit) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const v3 ro(o[3 * (size_t)i], o[3 * (size_t)i + 1], o[3 * (size_t)i + 2]);
  const v3 rd(d[3 * (size_t)i], d[3 * (size_t)i + 1], d[3 * (size_t)i + 2]);
  hit[i] = occluded<BVH>(P, ro, rd, sf(mint[i]), sf(maxt[i])) ? 1 : 0;
}
}  // namespace
}  // namespace gvpm

void launch_occluded(const GatherParams &P, bool bvh, const float *o, const float *d, const float *mint, const float *maxt,
                     uint32_t n, uint8_t *hit, cudaStream_t st) {
  if (n == 0) return;
  if (bvh) k_occluded<true><<<(n + 127) / 128, 128, 0, st>>>(P, o, d, mint, maxt, n, hit);
  else k_occluded<false><<<(n + 127) / 128, 128, 0, st>>>(P, o, d, mint, maxt, n, hit);
}

// The list up to 32 triangles (the per-pair near mask of occluder_device.cuh covers that many), the BVH above.
bool occluder_use_bvh(const gvpm_ctx *ctx) {
  if (ctx->n_tri == 0) return false;
  return ctx->occ_accel == GVPM_OCC_BVH || (ctx->occ_accel == GVPM_OCC_AUTO && ctx->n_tri > 32u);
}

void occluder_params(const gvpm_ctx *ctx, GatherParams &P) {
  P.tri = ctx->tri.as<float>();
  P.tri_plane = ctx->tri_plane.as<float4>();
  P.tri_aux = ctx->tri_aux.as<float2>();
  P.n_tri = ctx->n_tri;
  const bool bvh = occluder_use_bvh(ctx) && ctx->occ_built;
  P.occ_nodes = bvh ? ctx->occ_nodes.as<float4>() : nullptr;
  P.n_occ_nodes = bvh ? ctx->n_occ_nodes : 0u;
}

// The build of one triangle set in place: tri / plane / aux (n entries) are permuted into leaf order, the nodes written
// to `nodes` (*n_nodes of them); perm, when given, receives the permutation (leaf slot -> index the set had before).
// The occluders and the mesh scene each call it on their own arrays.
int build_tri_bvh(gvpm_ctx *ctx, DevBuf &tri, DevBuf &plane, DevBuf &aux, uint32_t n, DevBuf &nodes, uint32_t *n_nodes,
                  DevBuf *perm) {
  const uint32_t nL = (n + GVPM_OCC_LEAF - 1) / GVPM_OCC_LEAF, nI = nL - 1, nNodes = 2 * nL - 1;
  cudaStream_t st = ctx->stream;
  // scratch: centroids, keys / values in and out, sort scratch, bounds, permuted triangles, the radix tree
  size_t off = 0;
  auto carve = [&](size_t bytes) { const size_t o = off; off += align256(bytes); return o; };
  const size_t o_cen = carve(12ull * n), o_kin = carve(4ull * n), o_vin = carve(4ull * n), o_kout = carve(4ull * n),
               o_vout = carve(4ull * n), o_part = carve(6ull * 4 * bounds_blocks(n)), o_bounds = carve(64),
               o_tri = carve(36ull * n), o_plane = carve(16ull * n), o_aux = carve(8ull * n),
               o_first = carve(4ull * nL), o_last = carve(4ull * nL), o_split = carve(4ull * nL),
               o_parent = carve(4ull * nL), o_lparent = carve(4ull * nL), o_pin = carve(4ull * nL),
               o_pleaf = carve(4ull * nL), o_arrived = carve(4ull * nL);
  const size_t sort_bytes = sort_temp_bytes(n);
  const size_t o_sort = carve(sort_bytes);
  CK(ctx->occ_scratch.reserve(off));
  CK(nodes.reserve((size_t)nNodes * GVPM_OCC_NODE_FLOAT4 * sizeof(float4)));
  if (perm) CK(perm->reserve(4ull * n));
  char *S = ctx->occ_scratch.as<char>();
  auto u32 = [&](size_t o) { return (uint32_t *)(S + o); };
  float *cen = (float *)(S + o_cen);
  const unsigned b = 256, g = (n + b - 1) / b;
  k_occ_centroids<<<g, b, 0, st>>>(tri.as<float>(), n, cen);
  launch_bounds(cen, n, (float *)(S + o_part), (float *)(S + o_bounds), st, 3);
  launch_morton(cen, n, (float *)(S + o_bounds), u32(o_kin), u32(o_vin), st, 3);
  CK(run_sort_bits(S + o_sort, sort_bytes, u32(o_kin), u32(o_kout), u32(o_vin), u32(o_vout), n, kHilbertBits, st));
  k_occ_permute<<<g, b, 0, st>>>(u32(o_vout), n, tri.as<float>(), plane.as<float4>(), aux.as<float2>(),
                                 (float *)(S + o_tri), (float4 *)(S + o_plane), (float2 *)(S + o_aux));
  CK(cudaMemcpyAsync(tri.p, S + o_tri, 36ull * n, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(plane.p, S + o_plane, 16ull * n, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(aux.p, S + o_aux, 8ull * n, cudaMemcpyDeviceToDevice, st));
  if (perm) CK(cudaMemcpyAsync(perm->p, S + o_vout, 4ull * n, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemsetAsync(S + o_parent, 0xff, 4ull * nL, st));
  CK(cudaMemsetAsync(S + o_lparent, 0xff, 4ull * nL, st));
  CK(cudaMemsetAsync(S + o_arrived, 0, 4ull * nL, st));
  if (nI) k_occ_karras<<<(nI + b - 1) / b, b, 0, st>>>(u32(o_kout), nL, u32(o_first), u32(o_last), u32(o_split),
                                                       u32(o_parent), u32(o_lparent));
  k_occ_pos<<<(nI + nL + b - 1) / b, b, 0, st>>>(nL, u32(o_first), u32(o_split), u32(o_parent), u32(o_lparent),
                                                 u32(o_pin), u32(o_pleaf));
  k_occ_boxes<<<(nL + b - 1) / b, b, 0, st>>>(n, nL, tri.as<float>(), plane.as<float4>(), aux.as<float2>(), u32(o_first),
                                             u32(o_last), u32(o_split), u32(o_parent), u32(o_lparent), u32(o_pin),
                                             u32(o_pleaf), u32(o_arrived), nodes.as<float4>());
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(st));
  ctx->launches += 8 + (nI ? 1 : 0);
  *n_nodes = nNodes;
  return GVPM_OK;
}

int build_occluder_bvh(gvpm_ctx *ctx) {
  const int rc = build_tri_bvh(ctx, ctx->tri, ctx->tri_plane, ctx->tri_aux, ctx->n_tri, ctx->occ_nodes,
                               &ctx->n_occ_nodes, nullptr);
  if (rc) return rc;
  ctx->occ_built = true;
  return GVPM_OK;
}

// the mesh scene's albedos into the leaf order of its BVH
namespace gvpm {
namespace {
__global__ void k_mesh_albedo(const uint32_t *__restrict__ perm, uint32_t n, const float *__restrict__ in,
                              float *__restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = perm[i];
#pragma unroll
  for (int a = 0; a < 3; ++a) out[3 * (size_t)i + a] = in[3 * (size_t)s + a];
}
}  // namespace
}  // namespace gvpm

int build_mesh_bvh(gvpm_ctx *ctx) {
  gvpm_ctx::TraceMesh &M = ctx->mesh;
  int rc = build_tri_bvh(ctx, M.tri, M.plane, M.aux, M.n_tri, M.nodes, &M.n_nodes, &M.perm);
  if (rc) return rc;
  k_mesh_albedo<<<(M.n_tri + 255) / 256, 256, 0, ctx->stream>>>(M.perm.as<uint32_t>(), M.n_tri,
                                                                  M.albedo_in.as<float>(), M.albedo.as<float>());
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->launches += 1;
  return GVPM_OK;
}
