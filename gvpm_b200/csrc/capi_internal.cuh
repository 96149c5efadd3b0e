// capi_internal.cuh — what the capi_*.cu units of the C ABI (include/gvpm_b200.h) share: the context, its device
// buffers, error reporting, the staged SoA layouts, the kernel launchers they call and the helpers more than one
// unit uses.  Private to the library.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <utility>
#include <vector>

#include "gvpm_device.cuh"

namespace gvpm {
size_t sort_temp_bytes(uint32_t n);
cudaError_t run_sort_bits(void *temp, size_t temp_bytes, const uint32_t *kin, uint32_t *kout, const uint32_t *vin,
                          uint32_t *vout, uint32_t n, int bits, cudaStream_t st);
constexpr int kHilbertBits = 30;   // width of the keys of launch_morton / launch_keys_kept (and of sort_temp_bytes' sort)
int bounds_blocks(uint32_t n);
void launch_bounds(const float *pos, uint32_t n, float *partial, float *bounds, cudaStream_t st, uint32_t stride = 3);
void launch_morton(const float *pos, uint32_t n, const float *bounds, uint32_t *keys, uint32_t *vals,
                   cudaStream_t st, uint32_t stride = 3);
int pinhole_blocks(uint32_t n);
void launch_pinhole_fit(const float4 *rays, uint32_t n, double *partial, float *fit, unsigned *stats, cudaStream_t st,
                        const float *view_dir);
size_t frustum_occ_bytes();
void launch_frustum_keys(const float *pos, uint32_t stride, const uint32_t *par_src, uint32_t par_stride, uint32_t par_shift,
                         uint32_t n, const FrustumGrid &G, const uint32_t *occ, uint32_t *keys, uint32_t *vals,
                         unsigned *coord_mag, uint32_t *keepmask, uint32_t *cell_count, uint32_t region_cap,
                         const uint32_t *region_count, cudaStream_t st);
void launch_frustum_pack(const PhotonStaging &S, uint32_t n, const FrustumGrid &G, const uint32_t *occ, uint32_t *keys,
                         uint32_t *vals, unsigned *coord_mag, uint32_t *keepmask, uint32_t *cell_count, float4 *aos,
                         float4 *plane_src, cudaStream_t st);
size_t cell_scan_temp_bytes(uint32_t n_keys);
cudaError_t launch_cell_scan(void *temp, size_t temp_bytes, const uint32_t *cell_count, uint32_t *cell_start, uint32_t n_keys,
                             cudaStream_t st);
void launch_scatter_gather(uint32_t n, const uint32_t *keepmask, const uint32_t *keys, const uint32_t *rank,
                           const uint32_t *cell_start, const float4 *src, uint32_t stride, const uint32_t *kept_dev,
                           float4 *planes, uint32_t *orig, int sm_count, cudaStream_t st);
void launch_frustum_mark(const float4 *rays, uint32_t n_rays, const FrustumGrid &G, uint32_t *occ, int sm_count, cudaStream_t st);
void launch_dispatch(const DispatchParams &P, cudaStream_t st, int ctas);
void launch_dispatch_signal(const SignalParams &P, cudaStream_t st);
void launch_flag_wait(const uint32_t *flags, int n, uint32_t target, unsigned *timeout, cudaStream_t st);
void launch_flag_set(const FlagSetParams &P, cudaStream_t st);
void launch_or_flag(uint32_t *dst, const uint32_t *src, cudaStream_t st);
void launch_l2_read(const void *p, size_t bytes, int reps, unsigned *sink, int sm_count, cudaStream_t st);
void launch_translate_idx(uint32_t *idx, unsigned long long n, const float4 *aos, cudaStream_t st);
void launch_compact_kept(const uint32_t *keepmask, const uint32_t *block_off, uint32_t n, uint32_t *vals_c, cudaStream_t st);
void launch_pack_sorted_kept(const PhotonStaging &S, uint32_t n, const uint32_t *keepmask, const uint32_t *sorted, uint32_t m,
                             float4 *aos, float4 *planes, uint32_t *orig, cudaStream_t st);
void launch_scan_u32(uint32_t *vals, uint32_t nb, uint32_t *total, cudaStream_t st);
size_t ray_grid_bytes();
size_t ray_mask_bytes();
void launch_ray_region(const float4 *rays, uint32_t nRays, float radius, float *box, void *grid, uint32_t *mask,
                       float *bounds, int sm_count, cudaStream_t st);
void launch_keep_pruned(const float *pos, uint32_t n, const void *grid, const uint32_t *mask, uint32_t *keepmask,
                        uint32_t *block_kept, cudaStream_t st);
void launch_keys_kept(const float *pos, const uint32_t *vals, uint32_t m, const void *grid, uint32_t *keys, cudaStream_t st);
void launch_pack_sorted(const PhotonStaging &S, float4 *aos, const uint32_t *sorted, uint32_t n, float4 *planes,
                        uint32_t *orig, cudaStream_t st, bool records_ready = false);
void launch_leaf_boxes(const float4 *p0, uint32_t n, uint32_t nLeaves, float radius, float4 *lo, float4 *hi,
                       cudaStream_t st);
void launch_level_boxes(const float4 *clo, const float4 *chi, uint32_t nChild, uint32_t nParent, float4 *plo,
                        float4 *phi, cudaStream_t st);
void launch_pack_rays(const RayStaging &S, uint32_t n, float4 *rays, cudaStream_t st);
void launch_pack_rays_range(const RayStaging &S, uint32_t r0, uint32_t r1, float4 *rays, cudaStream_t st);
cudaError_t launch_bre_traverse(const GatherParams &P, bool dump, int sm_count, cudaStream_t stream);
cudaError_t launch_bre_shade(const GatherParams &P, unsigned long long total, int sm_count, cudaStream_t stream);
void launch_sub_gather(const float4 *raw, const uint32_t *sorted, uint32_t n, float4 *out, cudaStream_t st);
void launch_subbeam_leaf_boxes(const float4 *subs, const float4 *beams, uint32_t n, uint32_t nLeaves, float radius,
                               float4 *lo, float4 *hi, cudaStream_t st);
cudaError_t launch_beam_traverse(const GatherParams &P, int sm_count, cudaStream_t stream);
cudaError_t launch_beam_shade(const GatherParams &P, unsigned long long total, int sm_count, cudaStream_t stream);
cudaError_t launch_beam_shade_sppm(const GatherParams &P, unsigned long long total, int sm_count, cudaStream_t stream);
void launch_plane_pack_sorted(const float4 *raw, const uint32_t *sorted, uint32_t n, float4 *planes, uint32_t *orig,
                              cudaStream_t st);
void launch_plane_leaf_boxes(const float4 *planes, uint32_t n, uint32_t nLeaves, float4 *lo, float4 *hi, cudaStream_t st);
cudaError_t launch_plane_gather(const GatherParams &P, bool dump, int sm_count, cudaStream_t stream);
cudaError_t launch_vpm_traverse(const GatherParams &P, bool dump, int sm_count, cudaStream_t stream);
cudaError_t launch_vpm_shade(const GatherParams &P, unsigned long long total, int sm_count, cudaStream_t stream);
void launch_gradient(const float *acc, int w, int h, int use_abs, float *thr, float *gx, float *gy,
                     cudaStream_t st, int reuse = 0, float inv_emitted = 1.f);
void launch_generate_rays(const RayGenParams &P, cudaStream_t st);
void launch_generate_rays(const MeshRayGenParams &P, cudaStream_t st);
void launch_trace_count(const TraceParams &P, bool beams, uint8_t *counts, unsigned long long *block_tot,
                        unsigned long long *totals, cudaStream_t st);
void launch_trace_count(const MeshTraceParams &P, bool beams, uint8_t *counts, unsigned long long *block_tot,
                        unsigned long long *totals, cudaStream_t st);
void launch_trace_emit(const TraceParams &P, bool beams, const uint8_t *counts, const unsigned long long *block_off,
                       unsigned long long *last_path, cudaStream_t st);
void launch_trace_emit(const MeshTraceParams &P, bool beams, const uint8_t *counts, const unsigned long long *block_off,
                       unsigned long long *last_path, cudaStream_t st);
void launch_planes_from_beams(const PlaneGenParams &P, cudaStream_t st);
void launch_pack_beams(const BeamStaging &S, uint32_t n, float4 *rec, float *len, cudaStream_t st);
void launch_beam_subsize_seq(const float *len, uint32_t n, float *subsize, cudaStream_t st);
void launch_sub_count(const float *len, uint32_t n, const float *subsize, uint32_t *block_tot, uint32_t *total, cudaStream_t st);
void launch_sub_emit(const float4 *rec, const float *len, uint32_t n, const float *subsize, const uint32_t *block_off,
                     uint32_t cap, float *sub_pos, float4 *sub_raw, cudaStream_t st);
void launch_pack_planes(const PlaneStaging &S, uint32_t n, float4 *rec, float *centre, uint32_t *flag, cudaStream_t st);
void launch_pack_samples(const void *staging, uint32_t n, const uint32_t *n_dev, uint32_t n_rays, float4 *packed,
                         uint32_t *stats, cudaStream_t st);
void launch_vpm_samples(const VpmGenParams &P, uint32_t *total, int sm_count, cudaStream_t st);
size_t poisson_workspace_floats(size_t n);
long long poisson_solve_device(const float *tp, const float *dx, const float *dy, const float *direct, int W, int H,
                               float alpha, int irlsIterMax, float irlsRegInit, float irlsRegIter, int cgIterMax,
                               int cgIterCheck, float cgTolerance, float *ws, float *host_rz, float *rec,
                               cudaStream_t st);
void launch_accum_scatter(const float *out, uint32_t stride, const int32_t *px, const int32_t *py, uint32_t n, int w,
                          int h, int C, float *dst, uint8_t *smoke, int sm_count, cudaStream_t st);
void launch_accum_keys(const int32_t *px, const int32_t *py, uint32_t n, int w, int h, uint32_t *keys, uint32_t *vals,
                       cudaStream_t st);
void launch_accum_runs(const float *out, uint32_t stride, const uint32_t *skeys, const uint32_t *svals, uint32_t n,
                       uint32_t npix, int C, float *dst, uint8_t *smoke, int sm_count, cudaStream_t st);
void launch_accum_fold(float *acc, float *pix, size_t count, float itm1, float rnb, float rit, int sm_count,
                       cudaStream_t st);
}  // namespace gvpm

using namespace gvpm;

struct DevBuf {  // grow-only device allocation, freed with its owner
  void *p = nullptr;
  size_t cap = 0;
  bool pinned = false;  // exported to peers (CUDA IPC): the allocation must not move any more
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept { swap(o); }
  DevBuf &operator=(DevBuf &&o) noexcept { swap(o); return *this; }
  ~DevBuf() { if (p) cudaFree(p); }
  void swap(DevBuf &o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); std::swap(pinned, o.pinned); }
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (pinned) return cudaErrorInvalidValue;
    // the old block stays valid until the new one exists; if memory is too tight for both, give the old one up
    // first and leave the buffer empty (cap = 0) when the allocation still fails
    const size_t want = bytes + bytes / 8 + 256;
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, want);
    if (e != cudaSuccess) {
      cudaGetLastError();
      if (p) cudaFree(p);
      p = nullptr;
      cap = 0;
      e = cudaMalloc(&q, want);
      if (e != cudaSuccess) return e;
    } else if (p) {
      cudaFree(p);
    }
    p = q;
    cap = want;
    return cudaSuccess;
  }
  template <typename T> T *as() const { return (T *)p; }
};

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct gvpm_ctx {
  int device = 0, sm_count = 0;
  cudaStream_t stream = nullptr, copy_in = nullptr, copy_out = nullptr;  // compute, H2D, D2H
  cudaEvent_t pipe_ev[2 * 32 + 1] = {};  // per chunk: inputs landed / results ready; [64]: staging free
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  std::string err;
  uint64_t launches = 0;

  gvpm_medium medium{};
  bool have_medium = false;
  gvpm_config cfg{};
  bool have_cfg = false;

  DevBuf tri, tri_plane, tri_aux;   // in leaf order of the occluder BVH once it is built
  uint32_t n_tri = 0;
  int occ_accel = GVPM_OCC_AUTO;     // gvpm_set_occluder_accel
  bool occ_built = false;            // occ_nodes holds the BVH of the current set
  uint32_t n_occ_nodes = 0;
  DevBuf occ_nodes, occ_scratch, occ_query;   // BVH nodes; build scratch; gvpm_occluded's rays and hits

  // mesh scene of gvpm_set_trace_mesh (capi_photons.cu): triangles, planes, slack terms, albedos and the caller's index
  // of each, in the leaf order of its BVH (build_mesh_bvh); emit = the emissive triangles' vertices, triangle indices
  // and area running sum, back to back
  struct TraceMesh {
    bool ready = false;
    uint32_t n_tri = 0, n_nodes = 0, n_emit = 0, emit_last = 0;
    float emit_total = 0.f, lo[3] = {}, hi[3] = {}, light_power = 0.f;
    size_t emit_idx_off = 0, emit_cdf_off = 0;
    DevBuf tri, plane, aux, albedo, perm, nodes, emit, albedo_in;
  } mesh;

  DevBuf ph_staging, ph_staging_alt;  // the selected photon staging buffer and the other one (double buffering)
  int ph_staging_sel = 0;
  // peer exchange over NVLink copy engines (gvpm_peer_*): interprocess events + peer mappings of the staging buffers
  cudaEvent_t ev_free[2] = {nullptr, nullptr};   // staging buffer b has been consumed by this context's last build
  cudaEvent_t ev_pushed[2] = {nullptr, nullptr}; // this context's slice has landed in every peer's staging buffer b
  cudaStream_t push_streams[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaStream_t push_kernel_stream = nullptr;  // highest priority: the SM push kernel takes its CTA slots as soon as they free
  int push_ctas = 32;                         // 0: copy engines (cudaMemcpyAsync per field and peer)
  cudaEvent_t push_ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // [0..3] push stream done, [4] slice ready
  int n_peers = 0, peer_self = -1;
  std::vector<void *> peer_staging[2];
  std::vector<cudaEvent_t> peer_free[2], peer_pushed[2];
  void *staging_ptr(int which) const { return which == ph_staging_sel ? ph_staging.p : ph_staging_alt.p; }
  uint32_t n_photons = 0;
  bool photons_loaded = false;
  bool photons_direct = false;   // gvpm_trace_photons_direct: the 128-byte records in `aos` ARE the photon set (no staging, no packing)
  // dispatched photon set (gvpm_build_dispatched): the records live in an inbox the peers wrote; one region of
  // region_cap records per sender, region_count[s] (device) of them filled
  const uint32_t *build_ovf = nullptr;   // device flag of the last frustum build (a peer's dispatch timed out or overflowed)
  float4 *aos_override = nullptr;
  uint32_t region_cap = 0;
  const uint32_t *region_count = nullptr;
  float4 *records() { return aos_override ? aos_override : aos.as<float4>(); }
  struct RayFit { bool concurrent = false; float C[3], m[3], u[3], v[3], delta, cosmin, xmin, xmax, ymin, ymax, count; };
  // photon dispatch between ranks (dispatch.cu, gvpm_dispatch_*)
  struct Dispatch {
    int n_peers = 0, self = -1;
    uint32_t region_cap = 0;
    bool connected = false;
    DevBuf inbox[2], ctrl, occ_all, grids_dev[2], keepbits, block_cnt, owner_map;
    bool shared_frame = false;                  // every rank projects on the same plane: one classification per photon
    float ux0 = 0.f, uy0 = 0.f, ux1 = 0.f, uy1 = 0.f;   // bounds of the owner map (union of the ranks' ray bounds)
    RayFit fit[GVPM_MAX_PEERS];
    char *peer_inbox[2][GVPM_MAX_PEERS] = {};   // mapped (or, same process, raw) pointers; [self] = own
    uint32_t *peer_ctrl[GVPM_MAX_PEERS] = {};
    bool peer_mapped[GVPM_MAX_PEERS] = {};      // opened through CUDA IPC (to be closed)
    FrustumGrid *grids_host[2] = {nullptr, nullptr};   // pinned
    uint32_t gen_push[2] = {0, 0}, gen_build[2] = {0, 0}, gen_collect[2] = {0, 0};
    std::vector<void *> shared_owned, shared_opened;   // gvpm_shared_buffer_create / _open
    cudaEvent_t ev_src = nullptr;
  } disp;
  DevBuf aos, keys_in, keys_out, vals_in, vals_out, sort_temp, planes, orig, box_lo, box_hi, bounds_partial, bounds;
  Tree tree{};
  float radius = 0.f;
  bool built = false;
  float extent_hint = 1.f;  // diagonal of the photon AABB (host copy, refreshed lazily)
  // gvpm_build_points_for_rays: occupancy grid of the uploaded rays; the hierarchy then holds only the photons they can
  // reach and is valid for that ray set (rays_gen) alone
  DevBuf ray_region;        // [0,32): ray box, [32,..): RayGrid, the 32 KB cell mask, one keep bit per photon
  uint64_t rays_gen = 0, pruned_for_gen = 0;
  bool pruned = false;
  uint32_t n_kept = 0;
  // frustum grid (gvpm_device.cuh FrustumGrid): chosen by gvpm_build_points_for_rays when the uploaded rays are concurrent
  enum { ACCEL_BVH = 0, ACCEL_FRUSTUM = 1 };
  int accel = ACCEL_BVH;
  bool force_bvh = false;            // GVPM_ACCEL=bvh: A/B switch for kernel experiments
  FrustumGrid grid{};
  DevBuf cell_start, grid_occ, pin_scratch, trace_scratch, keepmask, cell_count;
  DevBuf plane_src;                  // first float4 of each kept photon's record, caller's order (staged frustum builds)
  bool occ_ready = false;            // grid_occ holds the occupancy mask of the current RayFit (analyse_rays)
  double trace_photons_per_path = 0.0;   // running estimate (sizes the first batch of gvpm_trace_photons)
  double trace_beams_per_path = 0.0;     // the same for gvpm_trace_beams
  // pin_scratch: [0,64) fit floats, [64,96) stats words, [128,..) block partials (doubles)
  uint64_t pin_gen = ~0ull;          // rays_gen the ray analysis below belongs to
  bool have_view_dir = false;        // gvpm_set_view_direction: axis of the perspective grid's projection plane
  float view_dir[3] = {0.f, 0.f, 1.f};
  RayFit pin;
  float *pin_host = nullptr;         // pinned: 16 fit floats + 8 stats words

  DevBuf ray_staging, rays;
  uint32_t n_rays = 0;
  bool rays_loaded = false;

  DevBuf out, counts, nbr_offsets, nbr_idx, work_counter, pairs;
  unsigned long long pair_cap = 0;         // capacity of `pairs` in entries
  unsigned long long *pair_count_host = nullptr;  // pinned read-back of the pair counter
  unsigned long long last_pairs = 0;
  // asynchronous BRE gathers in flight (pending_check): pair count slot = pair_count_host[8 + index]
  struct AsyncGather { cudaEvent_t done = nullptr; uint64_t gen = 0; float *out = nullptr; uint32_t *counts = nullptr; unsigned long long cap = 0; };
  static constexpr int kRing = 8;
  AsyncGather ring[kRing];
  int ring_tail = 0, ring_n = 0;
  uint64_t state_gen = 0;   // bumped by everything a gather's result depends on (photons, build, rays, medium, config)
  // G-Beams
  DevBuf beams, beam_bounds, sub_pos, sub_raw, subs, beam_box_lo, beam_box_hi;
  DevBuf beam_staging, beam_len, beam_aux;  // raw gvpm_beam_soa arrays; beam lengths; [0] subbeamSize, [1] sub-beam total, [16..] block offsets
  float beam_subsize = 0.f;                 // avgLength / 10 (summed on the host by gvpm_upload_beams, read back by gvpm_trace_beams)
  uint32_t n_subs = 0;                      // sub-beams of the uploaded beam set
  uint32_t n_beams = 0;
  bool beams_loaded = false, beams_built = false;
  Tree beam_tree{};
  float beam_radius = 0.f;
  // G-Planes
  DevBuf plane_raw, plane_pos, plane_rec, plane_orig, plane_box_lo, plane_box_hi, plane_bounds;
  DevBuf plane_staging;                     // raw gvpm_plane_soa arrays
  uint32_t n_planes = 0;
  bool planes_loaded = false, planes_built = false;
  DevBuf samples, sample_counts, mvol, sample_staging;  // G-VPM distance samples (+ their raw SoA arrays)
  DevBuf sample_scratch;                  // gvpm_generate_vpm_samples: samples per ray, then per tile of 256 rays
  uint32_t *sample_stats_host = nullptr;  // pinned: [2] plane flag; [4] sub-beam size (float bits), [5] sub-beam count of
                                          // traced beams; [8..10] the sample pack's stats (commit_samples)
  uint32_t n_samples = 0;
  bool samples_loaded = false;
  float sample_radius_max = 0.f;
  bool samples_drawn = false;             // the samples were drawn by gvpm_generate_vpm_samples, for ray set samples_rays_gen
  uint64_t samples_rays_gen = 0;
  // what `out` holds for gvpm_accum_add: OUT_READY = the per-ray results (out_stride floats per ray) of the last gather,
  // run on ray set out_gen; OUT_ADDED = the same, already added; OUT_ELSEWHERE = the last gather wrote to caller memory
  enum { OUT_NONE = 0, OUT_READY, OUT_ADDED, OUT_ELSEWHERE };
  int out_state = OUT_NONE;
  uint64_t out_gen = 0;
  uint32_t out_stride = GVPM_OUT_FLOATS;
  uint64_t pixel_rays_gen = ~0ull;   // rays_gen of a gvpm_generate_rays set: one ray per pixel of its rows
  // per-pixel accumulators (gvpm_accum_*, capi_accum.cu): acc [w*h*channels], pix the iteration sum (APA mode),
  // smoke one byte per pixel, keys four arrays of n_rays words + sort scratch (uploaded rays)
  struct Accum {
    bool ready = false, apa = false;
    int w = 0, h = 0, channels = 0;
    uint64_t total = 0;   // emitted paths (non-APA mode)
    DevBuf acc, pix, smoke, keys;
  } accum;
  DevBuf grad_in, grad_out;
  DevBuf poisson_io, poisson_ws;   // device copies of the four input planes + the result; solver workspace
  float poisson_ms = 0.f;
  float build_ms = 0.f, gather_ms = 0.f;
  bool timed_build = false, timed_gather = false;
  bool split_timed = false;   // the last gather recorded ev[4] / ev[5] around its traversal kernel
};

inline int fail(gvpm_ctx *c, int code, const std::string &msg) {
  if (c) c->err = msg;
  return code;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(ctx, GVPM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));        \
  } while (0)

// ---- staged SoAs --------------------------------------------------------------------------------------------------------
// Every SoA the ABI stages (gvpm_*_soa) is a struct of N pointers whose arrays go into one device buffer back to back,
// each starting on a 256-byte boundary; the device view (*Staging) holds the same N pointers in the same order.  elt[]
// is the one statement of each array's element size: offsets, sizes, views and copies all follow from it.
struct PhotonSoA {
  static constexpr int N = 13;
  static constexpr size_t elt[N] = {12, 12, 12, 12, 12, 12, 12, 4, 4, 4, 1, 1, 4};
  using Host = gvpm_photon_soa;
  using Staging = PhotonStaging;
  static constexpr const char *name = "gvpm_photon_soa";
};
struct RaySoA {
  static constexpr int N = 16;
  static constexpr size_t elt[N] = {12, 12, 4, 4, 4, 12, 4, 4, 4, 4, 4, 48, 48, 16, 48, 16};
  using Host = gvpm_ray_soa;
  using Staging = RayStaging;
  static constexpr const char *name = "gvpm_ray_soa";
};
struct BeamSoA {
  static constexpr int N = 14;
  static constexpr size_t elt[N] = {12, 12, 12, 12, 12, 12, 12, 12, 4, 4, 1, 1, 1, 4};
  using Host = gvpm_beam_soa;
  using Staging = BeamStaging;
  static constexpr const char *name = "gvpm_beam_soa";
};
struct PlaneSoA {
  static constexpr int N = 7;
  static constexpr size_t elt[N] = {12, 12, 4, 12, 4, 12, 4};
  using Host = gvpm_plane_soa;
  using Staging = PlaneStaging;
  static constexpr const char *name = "gvpm_plane_soa";
};
struct SampleSoA {
  static constexpr int N = 6;
  static constexpr size_t elt[N] = {4, 4, 12, 4, 4, 4};
  using Host = gvpm_vpm_sample_soa;
  using Staging = SampleStaging;
  static constexpr const char *name = "gvpm_vpm_sample_soa";
};

// sample_staging_at (gvpm_device.cuh) states this layout for the device
static_assert(SampleSoA::elt[0] == 4 && SampleSoA::elt[1] == 4 && SampleSoA::elt[2] == 12 && SampleSoA::elt[3] == 4 &&
                  SampleSoA::elt[4] == 4 && SampleSoA::elt[5] == 4, "sample_staging_at");

template <class S> struct SoaLayout {  // offsets of the arrays of n elements inside the staging buffer
  size_t off[S::N], bytes = 0;
  explicit SoaLayout(size_t n) {
    for (int i = 0; i < S::N; ++i) { off[i] = bytes; bytes += align256(S::elt[i] * n); }
  }
};

// the pointers of a struct that holds nothing but N pointers, in declaration order, and back
template <int N, class T> void struct_to_ptrs(const T &s, const void *(&p)[N]) {
  static_assert(sizeof(T) == N * sizeof(void *), "a struct of N pointers");
  memcpy(p, &s, sizeof(T));
}
template <int N, class T> void ptrs_to_struct(const void *const (&p)[N], T &s) {
  static_assert(sizeof(T) == N * sizeof(void *), "a struct of N pointers");
  memcpy(&s, p, sizeof(T));
}

template <class S> typename S::Staging staging_ptrs(const void *base, size_t n) {
  const SoaLayout<S> L(n);
  const void *p[S::N];
  for (int i = 0; i < S::N; ++i) p[i] = (const char *)base + L.off[i];
  typename S::Staging st;
  ptrs_to_struct<S::N>(p, st);
  return st;
}

// The writable view of a staging buffer a generator kernel fills (RayGenParams o .. off_sensor, TraceParams pos ..
// path_id and b_origin .. b_path_id, PlaneGenParams origin .. edge_id): the Staging pointers, in their order, without
// const.
static_assert(offsetof(RayGenParams, off_sensor) - offsetof(RayGenParams, o) == (RaySoA::N - 1) * sizeof(void *), "view");
static_assert(offsetof(TraceParams, path_id) - offsetof(TraceParams, pos) == (PhotonSoA::N - 1) * sizeof(void *), "view");
static_assert(offsetof(TraceParams, b_path_id) - offsetof(TraceParams, b_origin) == (BeamSoA::N - 1) * sizeof(void *), "view");
static_assert(offsetof(PlaneGenParams, edge_id) - offsetof(PlaneGenParams, origin) == (PlaneSoA::N - 1) * sizeof(void *), "view");
template <class S, class Field> void writable_view(Field *&first, const typename S::Staging &st) { memcpy(&first, &st, sizeof(st)); }

// Copies elements [src_first, src_first + count) of every array of `h` to elements [dst_first, dst_first + count) of
// the same array in a staging buffer laid out for n_total elements.  A null array is an error (nothing is copied).
template <class S>
int copy_soa(gvpm_ctx *ctx, const typename S::Host &h, void *staging, size_t n_total, size_t src_first, size_t dst_first,
             size_t count, cudaStream_t st) {
  const void *src[S::N];
  struct_to_ptrs<S::N>(h, src);
  for (const void *a : src)
    if (!a) return fail(ctx, GVPM_ERR_INVALID, std::string("null array in ") + S::name);
  const SoaLayout<S> L(n_total);
  for (int i = 0; i < S::N; ++i)
    CK(cudaMemcpyAsync((char *)staging + L.off[i] + dst_first * S::elt[i], (const char *)src[i] + src_first * S::elt[i],
                       count * S::elt[i], cudaMemcpyHostToDevice, st));
  return GVPM_OK;
}

// ---- helpers shared between the units ----------------------------------------------------------------------------------
// pair count a gather reports when its perspective grid is incomplete (build_ovf: a peer's dispatch timed out or overflowed)
constexpr unsigned long long kBuildOverflow = 1ull << 62;

// a gather has queued its per-ray results for the current ray set into ctx->out, `stride` floats per ray
inline void out_written(gvpm_ctx *ctx, uint32_t stride = GVPM_OUT_FLOATS) {
  ctx->out_state = gvpm_ctx::OUT_READY;
  ctx->out_gen = ctx->rays_gen;
  ctx->out_stride = stride;
}
int grid_incomplete(gvpm_ctx *ctx);                                   // the failure a gather reports then
// the checks and fields every gather shares: medium and config, its structure built, rays, counter block
int gather_params(gvpm_ctx *ctx, GatherParams &P, bool built, const char *not_built);
int fill_params(gvpm_ctx *ctx, GatherParams &P, float *out_dev, uint32_t *counts_dev);   // G-BRE / G-VPM
int reserve_pairs(gvpm_ctx *ctx, size_t entries);
// "run the traversal, read back the pair count, grow the list, retry" (capi_gather.cu)
int traverse_growing(gvpm_ctx *ctx, GatherParams &P, int attempts, const char *overflow_msg, bool within_budget,
                     const std::function<int()> &clear, const std::function<int()> &traverse,
                     unsigned long long *total);
// CSR neighbour dump (gvpm_dump_neighbours_*): counts -> offsets -> capacity check -> fill -> copy back -> canonical order
int dump_neighbours(gvpm_ctx *ctx, size_t rows, uint64_t *offsets, uint32_t *idx, size_t cap, bool pair_list,
                    const std::function<int(uint32_t *counts)> &count, const std::function<int(uint64_t total)> &fill);
// blocking copy of a gather's results to the host (bytes 0: nothing to copy)
int copy_back(gvpm_ctx *ctx, float *out, size_t out_bytes, uint32_t *counts, size_t counts_bytes, bool wait = true);
int pending_check(gvpm_ctx *ctx, bool block);
int reserve_sort(gvpm_ctx *ctx, uint32_t n);                          // radix-sort keys, values and scratch for n
int bvh_levels(gvpm_ctx *ctx, Tree &T, uint32_t n, const char *too_many, uint32_t *nodes);
void replace_photon_set(gvpm_ctx *ctx, size_t n, bool direct, float4 *records = nullptr, uint32_t region_cap = 0,
                        const uint32_t *region_count = nullptr);
int analyse_rays(gvpm_ctx *ctx);
FrustumGrid make_frustum_grid(const gvpm_ctx::RayFit &F, float radius, bool parity_split);
int build_frustum(gvpm_ctx *ctx, float radius, uint32_t *n_kept);
int build_pruned_bvh(gvpm_ctx *ctx, float radius, uint32_t *n_kept);
int check_scene(gvpm_ctx *ctx, const gvpm_box_scene *s);
// occluder BVH (occluder_bvh.cu): whether the gathers walk it, building it for the current set (n_tri > 0), the
// occluder fields of a gather's parameters, and the any-hit of gvpm_occluded on rays already on the device
bool occluder_use_bvh(const gvpm_ctx *ctx);
int build_tri_bvh(gvpm_ctx *ctx, DevBuf &tri, DevBuf &plane, DevBuf &aux, uint32_t n, DevBuf &nodes, uint32_t *n_nodes,
                  DevBuf *perm);
int build_occluder_bvh(gvpm_ctx *ctx);
// the mesh scene's BVH over ctx->mesh.tri / plane / aux (n_tri set, in the caller's order), then its albedos
// (ctx->mesh.albedo_in, the caller's order) into leaf order
int build_mesh_bvh(gvpm_ctx *ctx);
MeshScene mesh_view(const gvpm_ctx *ctx);   // the device view of ctx->mesh (capi_photons.cu)
// plane (unit normal, offset; zeros for a zero-area triangle) and rounding-slack terms (coefficient, largest |vertex
// coordinate|) of each triangle, as the BVH walks and their culls read them
void triangle_planes(const float *tri, size_t n_tri, std::vector<float> &planes, std::vector<float> &aux);
void occluder_params(const gvpm_ctx *ctx, GatherParams &P);
void launch_occluded(const GatherParams &P, bool bvh, const float *o, const float *d, const float *mint, const float *maxt,
                     uint32_t n, uint8_t *hit, cudaStream_t st);
// a new beam set of n beams (staging sized, the old set and its build dropped); then fill the staging arrays and
// commit_beams: records packed, sub-beam size and count known (host: the caller's arrays, for the host-side length sum;
// nullptr: the beams exist on the device only and the sum runs there)
int begin_beam_set(gvpm_ctx *ctx, size_t n);
int commit_beams(gvpm_ctx *ctx, const gvpm_beam_soa *host);
// computeGradient / computeGradient + Poisson on [h*w*27] accumulators: host memory (uploaded first) or, acc_on_device,
// device memory of this context read where it is (capi_image.cu)
int compute_gradient_impl(gvpm_ctx *ctx, const float *acc, bool acc_on_device, int w, int h, int use_abs, int reuse,
                          float inv_emitted, float *throughput, float *gx, float *gy);
int reconstruct_impl(gvpm_ctx *ctx, const float *acc, bool acc_on_device, int w, int h, int use_abs, const float *direct,
                     const gvpm_poisson_params *params, float *throughput, float *gx, float *gy, float *reconstruction);
