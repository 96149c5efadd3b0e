// capi_photons.cu — photon staging and upload, peer exchange of photon slices, on-device photon and beam tracing.
#include <type_traits>

#include "capi_internal.cuh"

// A new photon set replaces the old one: staged (direct = false), traced straight into the gather records, or
// dispatched by the peers into an inbox (records = the inbox, region_cap records per sender, region_count[s] filled).
void replace_photon_set(gvpm_ctx *ctx, size_t n, bool direct, float4 *records, uint32_t region_cap,
                        const uint32_t *region_count) {
  ctx->n_photons = (uint32_t)n;
  ctx->photons_loaded = true;
  ctx->photons_direct = direct;
  ctx->aos_override = records;
  ctx->region_cap = region_cap;
  ctx->region_count = region_count;
  ctx->built = false;
  ++ctx->state_gen;
}

int check_scene(gvpm_ctx *ctx, const gvpm_box_scene *s) {
  if (s->n_rects < 0 || s->n_rects > 4) return fail(ctx, GVPM_ERR_INVALID, "gvpm_box_scene: n_rects must be in [0, 4]");
  for (int a = 0; a < 3; ++a)
    if (!(s->lo[a] < s->hi[a])) return fail(ctx, GVPM_ERR_INVALID, "gvpm_box_scene: empty box");
  return GVPM_OK;
}

extern "C" {

int gvpm_photon_staging(gvpm_ctx *ctx, size_t n, void **dev, size_t *bytes) {
  if (!ctx || n > 0xfffffff0u) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const SoaLayout<PhotonSoA> L(n);
  if (ctx->ph_staging.pinned && (L.bytes ? L.bytes : 256) > ctx->ph_staging.cap)
    return fail(ctx, GVPM_ERR_INVALID, "the photon staging buffers were exported to peers (gvpm_peer_export) and cannot grow: "
                                        "size them for the largest iteration before exporting");
  CK(ctx->ph_staging.reserve(L.bytes ? L.bytes : 256));
  replace_photon_set(ctx, n, false);
  if (dev) *dev = ctx->ph_staging.p;
  if (bytes) *bytes = L.bytes;
  return GVPM_OK;
}

int gvpm_photon_staging_select(gvpm_ctx *ctx, int which) {
  if (!ctx || (which != 0 && which != 1)) return GVPM_ERR_INVALID;
  if (which != ctx->ph_staging_sel) {
    std::swap(ctx->ph_staging, ctx->ph_staging_alt);
    ctx->ph_staging_sel = which;
    ctx->built = false;
    ++ctx->state_gen;
  }
  return GVPM_OK;
}

int gvpm_photon_staging_layout(size_t n, size_t field_offset[13], size_t field_elem_bytes[13]) {
  const SoaLayout<PhotonSoA> L(n);
  for (int i = 0; i < PhotonSoA::N; ++i) {
    if (field_offset) field_offset[i] = L.off[i];
    if (field_elem_bytes) field_elem_bytes[i] = PhotonSoA::elt[i];
  }
  return GVPM_OK;
}

int gvpm_upload_photons_slice(gvpm_ctx *ctx, const gvpm_photon_soa *p, size_t n_total, size_t begin, size_t count,
                              void *stream) {
  if (!ctx || (count && !p) || begin + count > n_total) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (ctx->n_photons != n_total || !ctx->ph_staging.p || ctx->ph_staging.cap < SoaLayout<PhotonSoA>(n_total).bytes)
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_photon_staging(n_total) must be called first for the selected buffer");
  if (count == 0) return GVPM_OK;
  return copy_soa<PhotonSoA>(ctx, *p, ctx->ph_staging.p, n_total, 0, begin, count,
                             stream ? (cudaStream_t)stream : ctx->stream);
}

// ---- peer exchange of photon slices over NVLink copy engines ------------------------------------------------------
struct IpcBlob {  // what gvpm_peer_export writes (GVPM_PEER_BLOB_BYTES)
  cudaIpcMemHandle_t staging[2];
  cudaIpcEventHandle_t free_ev[2], pushed_ev[2];
};
static_assert(sizeof(IpcBlob) == GVPM_PEER_BLOB_BYTES, "blob size");

int gvpm_peer_export(gvpm_ctx *ctx, void *blob) {
  if (!ctx || !blob) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (!ctx->ph_staging.p || !ctx->ph_staging_alt.p)
    return fail(ctx, GVPM_ERR_INVALID, "size both photon staging buffers (gvpm_photon_staging) before exporting them");
  IpcBlob *B = (IpcBlob *)blob;
  ctx->ph_staging.pinned = ctx->ph_staging_alt.pinned = true;
  for (int b = 0; b < 2; ++b) {
    CK(cudaIpcGetMemHandle(&B->staging[b], ctx->staging_ptr(b)));
    CK(cudaIpcGetEventHandle(&B->free_ev[b], ctx->ev_free[b]));
    CK(cudaIpcGetEventHandle(&B->pushed_ev[b], ctx->ev_pushed[b]));
    // make both events "recorded" so that a first wait on them is well defined
    CK(cudaEventRecord(ctx->ev_free[b], ctx->stream));
    CK(cudaEventRecord(ctx->ev_pushed[b], ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return GVPM_OK;
}

int gvpm_peer_connect(gvpm_ctx *ctx, const void *blobs, int n_peers, int self_index) {
  if (!ctx || !blobs || n_peers < 1 || self_index < 0 || self_index >= n_peers) return GVPM_ERR_INVALID;
  if (ctx->n_peers) return fail(ctx, GVPM_ERR_INVALID, "peers already connected");
  cudaSetDevice(ctx->device);
  const IpcBlob *B = (const IpcBlob *)blobs;
  for (int b = 0; b < 2; ++b) {
    ctx->peer_staging[b].assign(n_peers, nullptr);
    ctx->peer_free[b].assign(n_peers, nullptr);
    ctx->peer_pushed[b].assign(n_peers, nullptr);
  }
  ctx->n_peers = n_peers;
  ctx->peer_self = self_index;
  for (int p = 0; p < n_peers; ++p) {
    if (p == self_index) continue;
    for (int b = 0; b < 2; ++b) {
      CK(cudaIpcOpenMemHandle(&ctx->peer_staging[b][p], B[p].staging[b], cudaIpcMemLazyEnablePeerAccess));
      CK(cudaIpcOpenEventHandle(&ctx->peer_free[b][p], B[p].free_ev[b]));
      CK(cudaIpcOpenEventHandle(&ctx->peer_pushed[b][p], B[p].pushed_ev[b]));
    }
  }
  return GVPM_OK;
}

// SM push: one kernel reads this rank's slice of the 13 field arrays once (128-bit loads) and stores every word into
// the same place of every peer's staging buffer over NVLink (peer-mapped pointers), so the 7 outgoing streams of an
// 8-GPU box are fed in parallel.  It runs on a highest-priority stream with a small grid: the copy engines top out
// near 220 GB/s per GPU on this many-small-copies pattern (13 fields x 7 peers), a few SMs' worth of stores do not.
struct PushParams {
  const char *src;
  char *dst[8];
  int n_dst;
  unsigned long long off[13];   // byte offset of each field's slice inside a staging buffer
  unsigned long long cum[14];   // prefix sums of the slice sizes in 16-byte words
};
__global__ void __launch_bounds__(512) k_peer_push(const __grid_constant__ PushParams P) {
  const unsigned long long total = P.cum[13], stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long w0 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; w0 < total; w0 += 4 * stride) {
    uint4 v[4];
    unsigned long long byte[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const unsigned long long w = w0 + u * stride;
      byte[u] = ~0ull;
      if (w < total) {
        int f = 0;
        while (w >= P.cum[f + 1]) ++f;
        byte[u] = P.off[f] + (w - P.cum[f]) * 16ull;
        v[u] = __ldcs((const uint4 *)(P.src + byte[u]));
      }
    }
    for (int d = 0; d < P.n_dst; ++d)
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (byte[u] != ~0ull) __stcs((uint4 *)(P.dst[d] + byte[u]), v[u]);
  }
}

int gvpm_peer_push_mode(gvpm_ctx *ctx, int sm_ctas) {
  if (!ctx || sm_ctas < 0 || sm_ctas > 1024) return GVPM_ERR_INVALID;
  ctx->push_ctas = sm_ctas;
  return GVPM_OK;
}

int gvpm_peer_push_photon_slice(gvpm_ctx *ctx, int which, size_t n_total, size_t begin, size_t count, void *after_stream) {
  if (!ctx || (which != 0 && which != 1) || begin + count > n_total) return GVPM_ERR_INVALID;
  if (!ctx->n_peers) return fail(ctx, GVPM_ERR_INVALID, "gvpm_peer_connect has not been called");
  cudaSetDevice(ctx->device);
  const SoaLayout<PhotonSoA> L(n_total);
  const size_t *elt = PhotonSoA::elt;
  const char *mine = (const char *)ctx->staging_ptr(which);
  // the slice must be complete on this rank (work queued on after_stream, e.g. its H2D upload) ...
  cudaEvent_t src_ready = ctx->push_ev[4];
  CK(cudaEventRecord(src_ready, after_stream ? (cudaStream_t)after_stream : ctx->stream));
  bool aligned = ctx->n_peers <= 9;
  for (int f = 0; f < PhotonSoA::N; ++f) aligned = aligned && (begin * elt[f]) % 16 == 0 && (count * elt[f]) % 16 == 0;
  if (ctx->push_ctas > 0 && aligned && count > 0) {
    PushParams PP{};
    PP.src = mine;
    cudaStream_t ks = ctx->push_kernel_stream;
    CK(cudaStreamWaitEvent(ks, src_ready, 0));
    for (int p = 0; p < ctx->n_peers; ++p) {
      if (p == ctx->peer_self) continue;
      CK(cudaStreamWaitEvent(ks, ctx->peer_free[which][p], 0));
      PP.dst[PP.n_dst++] = (char *)ctx->peer_staging[which][p];
    }
    for (int f = 0; f < PhotonSoA::N; ++f) {
      PP.off[f] = L.off[f] + begin * elt[f];
      PP.cum[f + 1] = PP.cum[f] + count * elt[f] / 16;
    }
    k_peer_push<<<ctx->push_ctas, 512, 0, ks>>>(PP);
    CK(cudaGetLastError());
    ctx->launches += 1;
    CK(cudaEventRecord(ctx->ev_pushed[which], ks));
    return GVPM_OK;
  }
  int si = 0;
  for (int p = 0; p < ctx->n_peers; ++p) {
    if (p == ctx->peer_self) continue;
    cudaStream_t ps = ctx->push_streams[si++ & 3];
    CK(cudaStreamWaitEvent(ps, src_ready, 0));
    // ... and the peer must have consumed what its buffer held (its last build from it)
    CK(cudaStreamWaitEvent(ps, ctx->peer_free[which][p], 0));
    char *dst = (char *)ctx->peer_staging[which][p];
    for (int f = 0; f < PhotonSoA::N; ++f)
      CK(cudaMemcpyAsync(dst + L.off[f] + begin * elt[f], mine + L.off[f] + begin * elt[f], count * elt[f],
                         cudaMemcpyDeviceToDevice, ps));
  }
  // ev_pushed[which] = all push streams done: funnel them through stream 0
  for (int i = 1; i < 4; ++i) {
    CK(cudaEventRecord(ctx->push_ev[i], ctx->push_streams[i]));
    CK(cudaStreamWaitEvent(ctx->push_streams[0], ctx->push_ev[i], 0));
  }
  CK(cudaEventRecord(ctx->ev_pushed[which], ctx->push_streams[0]));
  return GVPM_OK;
}

int gvpm_peer_wait_photons(gvpm_ctx *ctx, int which) {
  if (!ctx || (which != 0 && which != 1)) return GVPM_ERR_INVALID;
  if (!ctx->n_peers) return fail(ctx, GVPM_ERR_INVALID, "gvpm_peer_connect has not been called");
  cudaSetDevice(ctx->device);
  for (int p = 0; p < ctx->n_peers; ++p)
    if (p != ctx->peer_self) CK(cudaStreamWaitEvent(ctx->stream, ctx->peer_pushed[which][p], 0));
  return GVPM_OK;
}

int gvpm_upload_photons(gvpm_ctx *ctx, const gvpm_photon_soa *p, size_t n) {
  if (!ctx || (n && !p)) return GVPM_ERR_INVALID;
  int rc = gvpm_photon_staging(ctx, n, nullptr, nullptr);
  if (rc) return rc;
  if (n == 0) return GVPM_OK;
  return copy_soa<PhotonSoA>(ctx, *p, ctx->ph_staging.p, n, 0, 0, n, ctx->stream);
}

// ---- on-device generators (SURVEY.md 8 rows f-1, f-2; csrc/generate.cu) -----------------------------------------------------
int gvpm_box_scene_default(gvpm_box_scene *s) {
  if (!s) return GVPM_ERR_INVALID;
  memset(s, 0, sizeof(*s));
  for (int a = 0; a < 3; ++a) { s->lo[a] = 0.f; s->hi[a] = 1.f; }
  const float alb[5][3] = {{0.63f, 0.065f, 0.05f}, {0.14f, 0.45f, 0.091f}, {0.7f, 0.7f, 0.7f}, {0.7f, 0.7f, 0.7f}, {0.7f, 0.7f, 0.7f}};
  memcpy(s->face_albedo, alb, sizeof(alb));
  s->n_rects = 1;   // the shelf
  s->rect[0].y = 0.5f; s->rect[0].x0 = 0.3f; s->rect[0].x1 = 0.7f; s->rect[0].z0 = 0.4f; s->rect[0].z1 = 0.8f;
  s->rect[0].albedo[0] = s->rect[0].albedo[1] = s->rect[0].albedo[2] = 0.6f;
  s->light_y = 0.999f; s->light_x0 = 0.35f; s->light_x1 = 0.65f; s->light_z0 = 0.35f; s->light_z1 = 0.65f;
  s->light_power = 100.f;
  return GVPM_OK;
}

}  // extern "C"

// The checks every tracer shares and the walk parameters of the medium: a non-zero return is the error to report.
// `scene` is the box (Params = TraceParams) or null (the mesh scene of gvpm_set_trace_mesh).
template <class Params>
static int trace_setup(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth, int rr_depth,
                       int min_depth, Params &P) {
  constexpr bool mesh = std::is_same<Params, MeshTraceParams>::value;
  if (!ctx || (!mesh && !scene) || n > 0xfffffff0u) return GVPM_ERR_INVALID;
  if (!ctx->have_medium) return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_medium first");
  cudaSetDevice(ctx->device);
  P = Params{};
  if constexpr (mesh) {
    if (!ctx->mesh.ready) return fail(ctx, GVPM_ERR_INVALID, "no mesh scene: gvpm_set_trace_mesh first");
    P.scene = mesh_view(ctx);
  } else {
    int rc = check_scene(ctx, scene);
    if (rc) return rc;
    P.scene = *scene;
  }
  P.sigma_s = ctx->medium.sigma_s[0];
  P.sigma_a = ctx->medium.sigma_a[0];
  P.hg_g = ctx->medium.hg_g;
  P.phase_type = ctx->medium.phase_type;
  P.max_depth = max_depth > 0 ? max_depth : 64;
  P.rr_depth = rr_depth;
  P.min_depth = min_depth;
  P.seed = seed;
  P.n_total = n;
  return GVPM_OK;
}

// Batches of light paths (count -> scan -> emit, in path order) until P.n_total records exist.  The first batch is
// sized from the records-per-path ratio seen so far (`per_path`, updated); `barren` is the error when 64 batches do not
// fill the set.  n_paths: paths up to and including the
// one that stored the last record.
template <class Params>
static int trace_batches(gvpm_ctx *ctx, Params &P, bool beams, double &per_path, const char *barren,
                         uint64_t *n_paths) {
  const unsigned long long n = P.n_total;
  cudaStream_t st = ctx->stream;
  unsigned long long filled = 0, pathBase = 0, *host = ctx->pair_count_host;   // host[0] batch total, host[1] last path
  uint32_t pidBase = 0;
  host[1] = 0;
  for (int batch = 0; filled < n; ++batch) {
    if (batch > 64) return fail(ctx, GVPM_ERR_INVALID, barren);
    const double ratio = per_path > 0.0 ? per_path : 1.0;
    double want = (double)(n - filled) / ratio * 1.03 + 4096.0;
    if (want > 2.0e9) want = 2.0e9;
    const uint32_t np = (uint32_t)want;
    const uint32_t nb = (np + 255) / 256;
    const size_t offCounts = 64, offBlocks = align256(offCounts + np);
    CK(ctx->trace_scratch.reserve(offBlocks + ((size_t)nb + 1) * 8));
    char *sc = ctx->trace_scratch.as<char>();
    unsigned long long *totals = (unsigned long long *)sc;   // [0] batch total, [1] last path
    if (batch == 0) CK(cudaMemsetAsync(sc, 0, 64, st));
    P.path_base = pathBase;
    P.n_paths = np;
    P.slot_base = filled;
    P.path_id_base = pidBase;
    launch_trace_count(P, beams, (uint8_t *)(sc + offCounts), (unsigned long long *)(sc + offBlocks), totals, st);
    launch_trace_emit(P, beams, (const uint8_t *)(sc + offCounts), (const unsigned long long *)(sc + offBlocks), totals + 1, st);
    ctx->launches += 3;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(host, totals, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const unsigned long long records = host[0] & ((1ull << 40) - 1ull), paths = host[0] >> 40;
    filled += records;
    pidBase += (uint32_t)paths;
    pathBase += np;
    per_path = (double)filled / (double)pathBase;
  }
  if (n_paths) *n_paths = host[1];
  return GVPM_OK;
}

template <class Params>
static int trace_impl(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth, int rr_depth,
                      int min_depth, uint64_t *n_paths, bool direct) {
  Params P;
  int rc = trace_setup(ctx, scene, n, seed, max_depth, rr_depth, min_depth, P);
  if (rc) return rc;
  void *dev = nullptr;
  PhotonStaging S{};
  if (direct) {
    // no staging: the records are written where the gather reads them
    CK(ctx->aos.reserve(128 * std::max<size_t>(n, 1)));
    replace_photon_set(ctx, n, true);
  } else {
    rc = gvpm_photon_staging(ctx, n, &dev, nullptr);
    if (rc) return rc;
    S = staging_ptrs<PhotonSoA>(dev, n);
  }
  if (n_paths) *n_paths = 0;
  if (n == 0) return GVPM_OK;
  P.aos = direct ? ctx->aos.as<float4>() : nullptr;
  writable_view<PhotonSoA>(P.pos, S);
  return trace_batches(ctx, P, false, ctx->trace_photons_per_path,
                       "gvpm_trace_photons: the light paths store (almost) no photon in this scene", n_paths);
}

template <class Params>
static int trace_beams_impl(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth,
                            int rr_depth, int min_depth, uint64_t *n_paths) {
  if (ctx && max_depth > 255)   // per-path counts are bytes: a path stores at most max_depth - 1 beams
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_trace_beams: max_depth must be <= 255");
  if (n > 0x0ffffff0u) return GVPM_ERR_INVALID;   // the bound of gvpm_upload_beams
  Params P;
  int rc = trace_setup(ctx, scene, n, seed, max_depth, rr_depth, min_depth, P);
  if (rc) return rc;
  rc = begin_beam_set(ctx, n);
  if (rc) return rc;
  if (n_paths) *n_paths = 0;
  if (n == 0) return GVPM_OK;
  const BeamStaging S = staging_ptrs<BeamSoA>(ctx->beam_staging.p, n);
  writable_view<BeamSoA>(P.b_origin, S);
  rc = trace_batches(ctx, P, true, ctx->trace_beams_per_path,
                     "gvpm_trace_beams: the light paths store (almost) no beam in this scene", n_paths);
  if (rc) return rc;
  return commit_beams(ctx, nullptr);
}

// ---- mesh scene (gvpm_set_trace_mesh) -------------------------------------------------------------------------------
// the box grown by 2e-6 of its extent (MeshScene::glo / ghi), each operation rounded on its own
__attribute__((optimize("fp-contract=off"))) static void grown_box(float lo, float hi, float &glo, float &ghi) {
  const float m = 2e-6f * (hi - lo);
  glo = lo - m;
  ghi = hi + m;
}

MeshScene mesh_view(const gvpm_ctx *ctx) {
  const gvpm_ctx::TraceMesh &M = ctx->mesh;
  MeshScene V{};
  V.tri = M.tri.as<float>();
  V.plane = M.plane.as<float4>();
  V.aux = M.aux.as<float2>();
  V.albedo = M.albedo.as<float>();
  V.perm = M.perm.as<uint32_t>();
  V.nodes = M.nodes.as<float4>();
  V.n_tri = M.n_tri;
  V.n_nodes = M.n_nodes;
  V.emit_tri = M.emit.as<float>();
  V.emit_idx = (const uint32_t *)(M.emit.as<char>() + M.emit_idx_off);
  V.emit_cdf = (const float *)(M.emit.as<char>() + M.emit_cdf_off);
  V.n_emit = M.n_emit;
  V.emit_last = M.emit_last;
  V.emit_total = M.emit_total;
  for (int a = 0; a < 3; ++a) { V.lo[a] = M.lo[a]; V.hi[a] = M.hi[a]; grown_box(M.lo[a], M.hi[a], V.glo[a], V.ghi[a]); }
  V.light_power = M.light_power;
  return V;
}

// area of a triangle in fp32, each operation rounded on its own in this order (the CPU restatement forms the same)
__attribute__((optimize("fp-contract=off"))) static float triangle_area(const float *p) {
  const float e1x = p[3] - p[0], e1y = p[4] - p[1], e1z = p[5] - p[2];
  const float e2x = p[6] - p[0], e2y = p[7] - p[1], e2z = p[8] - p[2];
  const float cx = e1y * e2z - e1z * e2y, cy = e1z * e2x - e1x * e2z, cz = e1x * e2y - e1y * e2x;
  return 0.5f * std::sqrt((cx * cx + cy * cy) + cz * cz);
}

static int set_trace_mesh(gvpm_ctx *ctx, const gvpm_mesh_scene *s) {
  if (!s) return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: null scene");
  const size_t n = s->n_tri;
  if (n > GVPM_MAX_OCCLUDERS) return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: more than 2^24 triangles");
  if (n && (!s->tri || !s->albedo || !s->emissive))
    return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: null tri, albedo or emissive array");
  float tol[3];
  for (int a = 0; a < 3; ++a) {
    if (!std::isfinite(s->lo[a]) || !std::isfinite(s->hi[a]))
      return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: the box is not finite");
    if (!(s->lo[a] < s->hi[a])) return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: empty box");
    tol[a] = 1e-6f * (s->hi[a] - s->lo[a]);
  }
  if (!std::isfinite(s->light_power)) return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: light_power is not finite");
  std::vector<float> etri;
  std::vector<uint32_t> eidx;
  std::vector<float> ecdf;
  float total = 0.f;
  uint32_t last = 0;
  bool any = false;
  for (size_t t = 0; t < n; ++t) {
    const float *p = s->tri + 9 * t;
    for (int k = 0; k < 9; ++k) {
      const int a = k % 3;
      if (!std::isfinite(p[k]))
        return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: triangle " + std::to_string(t) + " has a non-finite coordinate");
      if (p[k] < s->lo[a] - tol[a] || p[k] > s->hi[a] + tol[a])
        return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: triangle " + std::to_string(t) + " lies outside the box");
    }
    for (int c = 0; c < 3; ++c)
      if (!std::isfinite(s->albedo[3 * t + c]))
        return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: triangle " + std::to_string(t) + " has a non-finite albedo");
    if (!s->emissive[t]) continue;
    const float area = triangle_area(p);
    total = total + area;
    if (area > 0.f) { last = (uint32_t)eidx.size(); any = true; }
    etri.insert(etri.end(), p, p + 9);
    eidx.push_back((uint32_t)t);
    ecdf.push_back(total);
  }
  if (!any) return fail(ctx, GVPM_ERR_INVALID, "gvpm_set_trace_mesh: no emissive triangle of positive area");
  gvpm_ctx::TraceMesh &M = ctx->mesh;
  std::vector<float> planes, aux;
  triangle_planes(s->tri, n, planes, aux);
  cudaStream_t st = ctx->stream;
  CK(M.tri.reserve(36 * n));
  CK(M.plane.reserve(16 * n));
  CK(M.aux.reserve(8 * n));
  CK(M.albedo.reserve(12 * n));
  CK(M.albedo_in.reserve(12 * n));
  const size_t m = eidx.size();
  M.emit_idx_off = align256(36 * m);
  M.emit_cdf_off = M.emit_idx_off + align256(4 * m);
  CK(M.emit.reserve(M.emit_cdf_off + 4 * m));
  CK(cudaMemcpyAsync(M.tri.p, s->tri, 36 * n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(M.plane.p, planes.data(), 16 * n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(M.aux.p, aux.data(), 8 * n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(M.albedo_in.p, s->albedo, 12 * n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(M.emit.p, etri.data(), 36 * m, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(M.emit.as<char>() + M.emit_idx_off, eidx.data(), 4 * m, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(M.emit.as<char>() + M.emit_cdf_off, ecdf.data(), 4 * m, cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  M.n_tri = (uint32_t)n;
  const int rc = build_mesh_bvh(ctx);
  if (rc) return rc;
  M.n_emit = (uint32_t)m;
  M.emit_last = last;
  M.emit_total = total;
  for (int a = 0; a < 3; ++a) { M.lo[a] = s->lo[a]; M.hi[a] = s->hi[a]; }
  M.light_power = s->light_power;
  M.ready = true;
  return GVPM_OK;
}

extern "C" {

int gvpm_trace_photons(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth, int rr_depth,
                       int min_depth, uint64_t *n_paths) {
  return trace_impl<TraceParams>(ctx, scene, n, seed, max_depth, rr_depth, min_depth, n_paths, false);
}
int gvpm_trace_photons_direct(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth,
                              int rr_depth, int min_depth, uint64_t *n_paths) {
  return trace_impl<TraceParams>(ctx, scene, n, seed, max_depth, rr_depth, min_depth, n_paths, true);
}
int gvpm_trace_beams(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth, int rr_depth,
                     int min_depth, uint64_t *n_paths) {
  return trace_beams_impl<TraceParams>(ctx, scene, n, seed, max_depth, rr_depth, min_depth, n_paths);
}

int gvpm_set_trace_mesh(gvpm_ctx *ctx, const gvpm_mesh_scene *scene) {
  if (!ctx) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  ctx->mesh.ready = false;   // a failed call leaves no mesh scene
  return set_trace_mesh(ctx, scene);
}
int gvpm_trace_photons_mesh(gvpm_ctx *ctx, size_t n, uint64_t seed, int max_depth, int rr_depth, int min_depth,
                            uint64_t *n_paths) {
  return trace_impl<MeshTraceParams>(ctx, nullptr, n, seed, max_depth, rr_depth, min_depth, n_paths, false);
}
int gvpm_trace_photons_direct_mesh(gvpm_ctx *ctx, size_t n, uint64_t seed, int max_depth, int rr_depth, int min_depth,
                                   uint64_t *n_paths) {
  return trace_impl<MeshTraceParams>(ctx, nullptr, n, seed, max_depth, rr_depth, min_depth, n_paths, true);
}
int gvpm_trace_beams_mesh(gvpm_ctx *ctx, size_t n, uint64_t seed, int max_depth, int rr_depth, int min_depth,
                          uint64_t *n_paths) {
  return trace_beams_impl<MeshTraceParams>(ctx, nullptr, n, seed, max_depth, rr_depth, min_depth, n_paths);
}

}  // extern "C"
