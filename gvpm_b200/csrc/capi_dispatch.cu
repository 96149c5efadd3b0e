// capi_dispatch.cu — photon dispatch between ranks (dispatch.cu kernels), shared buffers and result collection.
#include <unistd.h>

#include "capi_internal.cuh"

extern "C" {

// ---- photon dispatch between ranks (dispatch.cu; include/gvpm_b200.h gvpm_dispatch_*) -----------------------------------
// Control block of a rank (its own device memory; the peers write into it, only the owner reads it), in 32-bit words:
enum {
  DC_PUSHED = 0,                           // [2][MAX_PEERS] generation of sender s's last dispatch into my inbox b
  DC_COUNT = 2 * GVPM_MAX_PEERS,           // [2][MAX_PEERS] records sender s wrote into its region of my inbox b
  DC_FREED = 4 * GVPM_MAX_PEERS,           // [2][MAX_PEERS] generation up to which RECEIVER d has released its inbox b
  DC_COLLECTED = 6 * GVPM_MAX_PEERS,       // [2][MAX_PEERS] generation of rank s's last result copy into MY image buffer b
  DC_TIMEOUT = 8 * GVPM_MAX_PEERS,         // set by k_flag_wait when a peer never signalled
  DC_OVERFLOW = 8 * GVPM_MAX_PEERS + 1,
  DC_OCC = 8 * GVPM_MAX_PEERS + 16,        // my ray-occupancy mask (frustum_occ_bytes), copied by the peers at connect
};
struct DispatchBlob {   // what gvpm_dispatch_export writes (GVPM_DISPATCH_BLOB_BYTES)
  long long pid;
  int device, n_peers;
  unsigned long long region_cap;
  void *raw_inbox[2], *raw_ctrl;           // valid inside the exporting process
  cudaIpcMemHandle_t inbox[2], ctrl;
  gvpm_ctx::RayFit fit;
};
static_assert(sizeof(DispatchBlob) <= GVPM_DISPATCH_BLOB_BYTES, "blob size");

int gvpm_dispatch_export(gvpm_ctx *ctx, int n_peers, size_t region_cap, void *blob) {
  if (!ctx || !blob || n_peers < 1 || n_peers > GVPM_MAX_PEERS || region_cap == 0 ||
      (unsigned long long)n_peers * region_cap > 0xfffffff0ull)
    return GVPM_ERR_INVALID;
  if (!ctx->rays_loaded) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_export needs this rank's rays first (gvpm_upload_rays)");
  if (ctx->disp.n_peers) return fail(ctx, GVPM_ERR_INVALID, "dispatch buffers already exported");
  cudaSetDevice(ctx->device);
  int rc = analyse_rays(ctx);
  if (rc) return rc;
  if (!ctx->pin.concurrent)
    return fail(ctx, GVPM_ERR_UNSUPPORTED, "photon dispatch needs concurrent rays (a pinhole's primary rays); use the all-gather exchange");
  gvpm_ctx::Dispatch &D = ctx->disp;
  const size_t ctrl_bytes = (size_t)DC_OCC * 4 + frustum_occ_bytes();
  for (int b = 0; b < 2; ++b) {
    CK(D.inbox[b].reserve((size_t)n_peers * region_cap * 128));
    D.inbox[b].pinned = true;
    CK(D.grids_dev[b].reserve(sizeof(FrustumGrid) * GVPM_MAX_PEERS));
    if (!D.grids_host[b]) CK(cudaHostAlloc((void **)&D.grids_host[b], sizeof(FrustumGrid) * GVPM_MAX_PEERS, cudaHostAllocDefault));
  }
  CK(D.ctrl.reserve(ctrl_bytes));
  D.ctrl.pinned = true;
  CK(D.occ_all.reserve(frustum_occ_bytes() * (size_t)n_peers));
  if (!D.ev_src) CK(cudaEventCreateWithFlags(&D.ev_src, cudaEventDisableTiming));
  CK(cudaMemsetAsync(D.ctrl.p, 0, ctrl_bytes, ctx->stream));
  // the occupancy mask depends on the rays alone (projection basis and bounds of the fit), not on the radius
  const FrustumGrid G = make_frustum_grid(ctx->pin, 1.f, false);
  launch_frustum_mark(ctx->rays.as<float4>(), ctx->n_rays, G, D.ctrl.as<uint32_t>() + DC_OCC, ctx->sm_count, ctx->stream);
  ctx->launches += 1;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream));
  DispatchBlob B{};
  B.pid = (long long)getpid();
  B.device = ctx->device;
  B.n_peers = n_peers;
  B.region_cap = region_cap;
  for (int b = 0; b < 2; ++b) {
    B.raw_inbox[b] = D.inbox[b].p;
    CK(cudaIpcGetMemHandle(&B.inbox[b], D.inbox[b].p));
  }
  B.raw_ctrl = D.ctrl.p;
  CK(cudaIpcGetMemHandle(&B.ctrl, D.ctrl.p));
  B.fit = ctx->pin;
  memset(blob, 0, GVPM_DISPATCH_BLOB_BYTES);
  memcpy(blob, &B, sizeof(B));
  D.n_peers = n_peers;
  D.region_cap = (uint32_t)region_cap;
  return GVPM_OK;
}

int gvpm_dispatch_connect(gvpm_ctx *ctx, const void *blobs, int n_peers, int self_index) {
  if (!ctx || !blobs || self_index < 0 || self_index >= n_peers) return GVPM_ERR_INVALID;
  gvpm_ctx::Dispatch &D = ctx->disp;
  if (D.n_peers != n_peers) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_export first, with the same number of peers");
  if (D.connected) return fail(ctx, GVPM_ERR_INVALID, "dispatch peers already connected");
  cudaSetDevice(ctx->device);
  const long long me = (long long)getpid();
  for (int p = 0; p < n_peers; ++p) {
    DispatchBlob B;
    memcpy(&B, (const char *)blobs + (size_t)p * GVPM_DISPATCH_BLOB_BYTES, sizeof(B));
    if (B.n_peers != n_peers || B.region_cap != D.region_cap)
      return fail(ctx, GVPM_ERR_INVALID, "dispatch blobs disagree on the number of peers / the region size");
    D.fit[p] = B.fit;
    if (B.pid == me) {   // same process (several contexts, tests): the pointers are valid as they are
      if (B.device != ctx->device) {
        int can = 0;
        CK(cudaDeviceCanAccessPeer(&can, ctx->device, B.device));
        if (!can) return fail(ctx, GVPM_ERR_UNSUPPORTED, "no peer access between two devices of this process");
        cudaError_t e = cudaDeviceEnablePeerAccess(B.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
        cudaGetLastError();
      }
      for (int b = 0; b < 2; ++b) D.peer_inbox[b][p] = (char *)B.raw_inbox[b];
      D.peer_ctrl[p] = (uint32_t *)B.raw_ctrl;
    } else {
      for (int b = 0; b < 2; ++b) CK(cudaIpcOpenMemHandle((void **)&D.peer_inbox[b][p], B.inbox[b], cudaIpcMemLazyEnablePeerAccess));
      CK(cudaIpcOpenMemHandle((void **)&D.peer_ctrl[p], B.ctrl, cudaIpcMemLazyEnablePeerAccess));
      D.peer_mapped[p] = true;
    }
    // the receiver's occupancy mask, read once: the classification then touches local memory only
    CK(cudaMemcpyAsync(D.occ_all.as<char>() + frustum_occ_bytes() * (size_t)p, D.peer_ctrl[p] + DC_OCC, frustum_occ_bytes(),
                       cudaMemcpyDeviceToDevice, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  D.self = self_index;
  D.connected = true;
  // Do all ranks project on the same plane (same axis and basis - gvpm_set_view_direction - and, up to rounding, the same
  // centre)?  Then a photon is classified ONCE: its footprint box is looked up in an owner map - kOccRes^2 cells over the
  // union of the ranks' ray bounds, one bit per rank whose own occupancy mask has a ray under the cell (dilated by a cell)
  // - instead of one key evaluation per receiver.
  D.shared_frame = n_peers <= 8;
  float cmag = 0.f;
  for (int k = 0; k < 3; ++k) cmag = std::max(cmag, std::fabs(D.fit[0].C[k]));
  for (int p = 1; p < n_peers && D.shared_frame; ++p)
    for (int k = 0; k < 3; ++k)
      D.shared_frame = D.shared_frame && D.fit[p].m[k] == D.fit[0].m[k] && D.fit[p].u[k] == D.fit[0].u[k] &&
                       D.fit[p].v[k] == D.fit[0].v[k] && std::fabs(D.fit[p].C[k] - D.fit[0].C[k]) <= 1e-5f * (1.f + cmag);
  if (D.shared_frame) {
    const int R = (int)std::lround(std::sqrt((double)frustum_occ_bytes() * 8.0));   // kOccRes
    D.ux0 = D.uy0 = 3.4e38f; D.ux1 = D.uy1 = -3.4e38f;
    for (int p = 0; p < n_peers; ++p) {
      D.ux0 = std::min(D.ux0, D.fit[p].xmin); D.ux1 = std::max(D.ux1, D.fit[p].xmax);
      D.uy0 = std::min(D.uy0, D.fit[p].ymin); D.uy1 = std::max(D.uy1, D.fit[p].ymax);
    }
    const double uw = std::max((double)D.ux1 - D.ux0, 1e-20), uh = std::max((double)D.uy1 - D.uy0, 1e-20);
    std::vector<uint32_t> occ(frustum_occ_bytes() / 4 * (size_t)n_peers);
    CK(cudaMemcpy(occ.data(), D.occ_all.p, occ.size() * 4, cudaMemcpyDeviceToHost));
    std::vector<uint8_t> map((size_t)R * R, 0);
    for (int p = 0; p < n_peers; ++p) {
      const gvpm_ctx::RayFit &F = D.fit[p];
      const double wx = std::max((double)F.xmax - F.xmin, 1e-20) / R, wy = std::max((double)F.ymax - F.ymin, 1e-20) / R;
      const uint32_t *o = occ.data() + (frustum_occ_bytes() / 4) * (size_t)p;
      for (int j = 0; j < R; ++j)
        for (int i = 0; i < R; ++i) {
          if (!(o[(j * R + i) >> 5] >> ((j * R + i) & 31) & 1u)) continue;
          const int i0 = (int)std::floor((F.xmin + i * wx - D.ux0) / uw * R) - 1, i1 = (int)std::floor((F.xmin + (i + 1) * wx - D.ux0) / uw * R) + 1;
          const int j0 = (int)std::floor((F.ymin + j * wy - D.uy0) / uh * R) - 1, j1 = (int)std::floor((F.ymin + (j + 1) * wy - D.uy0) / uh * R) + 1;
          for (int jj = std::max(j0, 0); jj <= std::min(j1, R - 1); ++jj)
            for (int ii = std::max(i0, 0); ii <= std::min(i1, R - 1); ++ii) map[(size_t)jj * R + ii] |= (uint8_t)(1u << p);
        }
    }
    CK(D.owner_map.reserve(map.size()));
    CK(cudaMemcpy(D.owner_map.p, map.data(), map.size(), cudaMemcpyHostToDevice));
  }
  return GVPM_OK;
}

int gvpm_dispatch_photons(gvpm_ctx *ctx, int which, size_t n_total, size_t begin, size_t count, float radius, void *after_stream) {
  if (!ctx || (which != 0 && which != 1) || begin + count > n_total || !(radius > 0.f)) return GVPM_ERR_INVALID;
  gvpm_ctx::Dispatch &D = ctx->disp;
  if (!D.connected) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_connect has not been called");
  if (count > D.region_cap) return fail(ctx, GVPM_ERR_INVALID, "slice larger than the exported region size");
  if (!ctx->ph_staging.p || ctx->ph_staging.cap < SoaLayout<PhotonSoA>(n_total).bytes)
    return fail(ctx, GVPM_ERR_INVALID, "size the selected photon staging buffer for n_total first (gvpm_photon_staging)");
  cudaSetDevice(ctx->device);
  // after_stream == the context's own stream: the dispatch runs IN that stream (between a build and its gather, say: a
  // side stream only gets CTA slots as the persistent gather kernels retire theirs, and every rank's next build waits for
  // the slowest rank's dispatch); any other stream / NULL: on the internal highest-priority stream, after that work
  cudaStream_t ks = ctx->push_kernel_stream;
  if (after_stream == (void *)ctx->stream) {
    ks = ctx->stream;
  } else {
    CK(cudaEventRecord(D.ev_src, after_stream ? (cudaStream_t)after_stream : ctx->stream));
    CK(cudaStreamWaitEvent(ks, D.ev_src, 0));
  }
  const uint32_t gen = ++D.gen_push[which];
  uint32_t *ctrl = D.ctrl.as<uint32_t>();
  // every receiver must have released its inbox `which` gen - 1 times (flags the receivers write into MY control block)
  if (gen > 1) {
    launch_flag_wait(ctrl + DC_FREED + which * GVPM_MAX_PEERS, D.n_peers, gen - 1, ctrl + DC_TIMEOUT, ks);
    ctx->launches += 1;
  }
  const bool parity = ctx->have_cfg && ctx->cfg.path_set && !ctx->cfg.sppm_primal;
  const uint32_t nb = (uint32_t)((count + 255) / 256);
  CK(D.keepbits.reserve(std::max<size_t>(count, 256)));
  CK(D.block_cnt.reserve((size_t)GVPM_MAX_PEERS * (nb + 2) * 4));
  static_assert(sizeof(DispatchParams) <= 4000, "kernel parameter space");
  DispatchParams P{};
  P.S = staging_ptrs<PhotonSoA>(ctx->ph_staging.p, n_total);
  P.begin = (uint32_t)begin;
  P.count = (uint32_t)count;
  P.n_dst = D.n_peers;
  for (int d = 0; d < D.n_peers; ++d) P.grids[d] = make_frustum_grid(D.fit[d], radius, parity);
  P.region_cap = D.region_cap;
  P.keepbits = D.keepbits.as<uint8_t>();
  P.block_cnt = D.block_cnt.as<uint32_t>();
  P.nb = nb;
  P.overflow = ctrl + DC_OVERFLOW;
  SignalParams Sg{};
  Sg.n_dst = D.n_peers;
  Sg.self = D.self;
  Sg.nb = nb;
  Sg.block_cnt = P.block_cnt;
  Sg.gen = gen;
  for (int d = 0; d < D.n_peers; ++d) {
    P.occ[d] = D.occ_all.as<uint32_t>() + (frustum_occ_bytes() / 4) * (size_t)d;
    P.inbox[d] = (float4 *)(D.peer_inbox[which][d] + (size_t)D.self * D.region_cap * 128);
    Sg.count_dst[d] = D.peer_ctrl[d] + DC_COUNT + which * GVPM_MAX_PEERS + D.self;
    Sg.flag_dst[d] = D.peer_ctrl[d] + DC_PUSHED + which * GVPM_MAX_PEERS + D.self;
  }
  P.owner_map = D.shared_frame ? D.owner_map.as<uint8_t>() : nullptr;
  if (D.shared_frame) {
    P.ux0 = D.ux0; P.uy0 = D.uy0;
    P.uix = (float)(std::sqrt((double)frustum_occ_bytes() * 8.0) / std::max((double)D.ux1 - D.ux0, 1e-20));
    P.uiy = (float)(std::sqrt((double)frustum_occ_bytes() * 8.0) / std::max((double)D.uy1 - D.uy0, 1e-20));
    P.ux1 = D.ux1; P.uy1 = D.uy1;
    P.pad_r_max = 0.f;
    for (int d = 0; d < D.n_peers; ++d) P.pad_r_max = std::max(P.pad_r_max, P.grids[d].pad_r);
    P.pad_r_max += 2e-5f * (1.f + std::fabs(P.grids[0].C[0]) + std::fabs(P.grids[0].C[1]) + std::fabs(P.grids[0].C[2]));   // the centres agree to 1e-5
  }
  // on the side stream: a persistent grid of one CTA per SM (N = 8, cfg5: 32 CTAs 1.96 ms / step, 96: 1.11, one per
  // chunk: 1.13); in-stream: one CTA per chunk
  launch_dispatch(P, ks, ks == ctx->stream ? 0 : ctx->sm_count);
  launch_dispatch_signal(Sg, ks);
  ctx->launches += 4;
  CK(cudaGetLastError());
  return GVPM_OK;
}

int gvpm_build_dispatched(gvpm_ctx *ctx, int which, float radius, uint32_t *n_kept) {
  if (!ctx || (which != 0 && which != 1) || !(radius > 0.f)) return GVPM_ERR_INVALID;
  gvpm_ctx::Dispatch &D = ctx->disp;
  if (!D.connected) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_connect has not been called");
  if (!ctx->rays_loaded) return fail(ctx, GVPM_ERR_INVALID, "no rays uploaded");
  cudaSetDevice(ctx->device);
  int rc = analyse_rays(ctx);
  if (rc) return rc;
  const gvpm_ctx::RayFit &Fa = ctx->pin, &Fb = D.fit[D.self];
  bool same = Fa.concurrent && Fb.concurrent && Fa.delta == Fb.delta && Fa.xmin == Fb.xmin && Fa.xmax == Fb.xmax &&
              Fa.ymin == Fb.ymin && Fa.ymax == Fb.ymax && Fa.count == Fb.count;
  for (int k = 0; k < 3; ++k) same = same && Fa.C[k] == Fb.C[k] && Fa.m[k] == Fb.m[k] && Fa.u[k] == Fb.u[k] && Fa.v[k] == Fb.v[k];
  if (!same)
    return fail(ctx, GVPM_ERR_INVALID, "the rays changed since gvpm_dispatch_export: the peers dispatch for the exported ray set");
  const uint32_t gen = ++D.gen_build[which];
  uint32_t *ctrl = D.ctrl.as<uint32_t>();
  launch_flag_wait(ctrl + DC_PUSHED + which * GVPM_MAX_PEERS, D.n_peers, gen, ctrl + DC_TIMEOUT, ctx->stream);
  ctx->launches += 1;
  replace_photon_set(ctx, (size_t)D.n_peers * D.region_cap, true, D.inbox[which].as<float4>(), D.region_cap,
                     ctrl + DC_COUNT + which * GVPM_MAX_PEERS);
  rc = build_frustum(ctx, radius, n_kept);
  if (rc) return rc;
  // a peer that never signalled (k_flag_wait timed out) or a region overflow: the grid is incomplete, and the gather says
  // so (through the build's overflow flag, which the BRE traversal reads); gvpm_dispatch_status names the cause
  if (ctx->build_ovf) {
    launch_or_flag(const_cast<uint32_t *>(ctx->build_ovf), ctrl + DC_TIMEOUT, ctx->stream);
    launch_or_flag(const_cast<uint32_t *>(ctx->build_ovf), ctrl + DC_OVERFLOW, ctx->stream);
    ctx->launches += 2;
    CK(cudaGetLastError());
  }
  return GVPM_OK;
}

int gvpm_dispatch_release(gvpm_ctx *ctx, int which) {
  if (!ctx || (which != 0 && which != 1)) return GVPM_ERR_INVALID;
  gvpm_ctx::Dispatch &D = ctx->disp;
  if (!D.connected) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_connect has not been called");
  cudaSetDevice(ctx->device);
  FlagSetParams F{};
  F.n = D.n_peers;
  F.value = D.gen_build[which];
  for (int s = 0; s < D.n_peers; ++s) F.dst[s] = D.peer_ctrl[s] + DC_FREED + which * GVPM_MAX_PEERS + D.self;
  launch_flag_set(F, ctx->stream);
  ctx->launches += 1;
  CK(cudaGetLastError());
  return GVPM_OK;
}


// ---- result collection over the copy engines (rank 0's image buffer, written by every rank) -------------------------------
int gvpm_shared_buffer_create(gvpm_ctx *ctx, size_t bytes, void **dev, void *handle) {
  if (!ctx || !dev || !handle || bytes == 0) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  void *p = nullptr;
  CK(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); CK(e); }
  ctx->disp.shared_owned.push_back(p);
  static_assert(sizeof(cudaIpcMemHandle_t) + 16 <= GVPM_SHARED_HANDLE_BYTES, "handle size");
  memset(handle, 0, GVPM_SHARED_HANDLE_BYTES);
  memcpy(handle, &h, sizeof(h));
  const long long pid = (long long)getpid();
  memcpy((char *)handle + sizeof(h), &pid, 8);
  memcpy((char *)handle + sizeof(h) + 8, &p, 8);
  *dev = p;
  return GVPM_OK;
}

int gvpm_shared_buffer_open(gvpm_ctx *ctx, const void *handle, void **dev) {
  if (!ctx || !dev || !handle) return GVPM_ERR_INVALID;
  cudaSetDevice(ctx->device);
  cudaIpcMemHandle_t h;
  long long pid = 0;
  void *raw = nullptr;
  memcpy(&h, handle, sizeof(h));
  memcpy(&pid, (const char *)handle + sizeof(h), 8);
  memcpy(&raw, (const char *)handle + sizeof(h) + 8, 8);
  if (pid == (long long)getpid()) { *dev = raw; return GVPM_OK; }   // same process: the pointer is valid as it is
  void *p = nullptr;
  CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  ctx->disp.shared_opened.push_back(p);
  *dev = p;
  return GVPM_OK;
}

int gvpm_collect_signal(gvpm_ctx *ctx, int which, int root, void *stream) {
  if (!ctx || (which != 0 && which != 1)) return GVPM_ERR_INVALID;
  gvpm_ctx::Dispatch &D = ctx->disp;
  if (!D.connected || root < 0 || root >= D.n_peers) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_connect has not been called");
  cudaSetDevice(ctx->device);
  FlagSetParams F{};
  F.n = 1;
  F.value = ++D.gen_collect[which];
  F.dst[0] = D.peer_ctrl[root] + DC_COLLECTED + which * GVPM_MAX_PEERS + D.self;
  launch_flag_set(F, stream ? (cudaStream_t)stream : ctx->stream);
  ctx->launches += 1;
  CK(cudaGetLastError());
  return GVPM_OK;
}

int gvpm_collect_wait(gvpm_ctx *ctx, int which) {
  if (!ctx || (which != 0 && which != 1)) return GVPM_ERR_INVALID;
  gvpm_ctx::Dispatch &D = ctx->disp;
  if (!D.connected) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_connect has not been called");
  cudaSetDevice(ctx->device);
  uint32_t *ctrl = D.ctrl.as<uint32_t>();
  // every rank signals once per iteration and buffer: wait until all have caught up with this rank's own count
  launch_flag_wait(ctrl + DC_COLLECTED + which * GVPM_MAX_PEERS, D.n_peers, D.gen_collect[which], ctrl + DC_TIMEOUT, ctx->stream);
  ctx->launches += 1;
  CK(cudaGetLastError());
  return GVPM_OK;
}

int gvpm_dispatch_join(gvpm_ctx *ctx) {
  if (!ctx) return GVPM_ERR_INVALID;
  gvpm_ctx::Dispatch &D = ctx->disp;
  if (!D.connected) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_connect has not been called");
  cudaSetDevice(ctx->device);
  CK(cudaEventRecord(D.ev_src, ctx->push_kernel_stream));
  CK(cudaStreamWaitEvent(ctx->stream, D.ev_src, 0));
  return GVPM_OK;
}

int gvpm_dispatch_status(gvpm_ctx *ctx, uint32_t counts[GVPM_MAX_PEERS], int which) {
  if (!ctx || (which != 0 && which != 1)) return GVPM_ERR_INVALID;
  gvpm_ctx::Dispatch &D = ctx->disp;
  if (!D.connected) return fail(ctx, GVPM_ERR_INVALID, "gvpm_dispatch_connect has not been called");
  cudaSetDevice(ctx->device);
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaStreamSynchronize(ctx->push_kernel_stream));
  uint32_t h[DC_OCC];
  CK(cudaMemcpy(h, D.ctrl.p, sizeof(h), cudaMemcpyDeviceToHost));
  if (counts) for (int s = 0; s < GVPM_MAX_PEERS; ++s) counts[s] = s < D.n_peers ? h[DC_COUNT + which * GVPM_MAX_PEERS + s] : 0u;
  if (h[DC_TIMEOUT]) return fail(ctx, GVPM_ERR_CUDA, "photon dispatch: a peer never signalled (flag wait timed out)");
  if (h[DC_OVERFLOW]) return fail(ctx, GVPM_ERR_INVALID, "photon dispatch: inbox region overflow");
  return GVPM_OK;
}

}  // extern "C"
