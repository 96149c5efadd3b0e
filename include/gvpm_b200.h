/* gvpm_b200.h — C ABI of the B200-native density-estimation gather.
 *
 * This is the drop-in boundary for ONE path of gradientpm/gvpm: the per-iteration volumetric
 * gather (primal + 4 offset-path gradient contributions per camera-ray medium segment) that
 * the `gvpm` / `sppm` integrator plugins run on CPU threads.  The C++ integrator stays host
 * code; the bodies of the reference's gather drivers become calls into this library.
 * Every entry point cites the reference interface it replaces (paths relative to the
 * reference root, src/integrators/photonmapper/...).
 *
 * Conventions
 *   - every function returns 0 on success, a negative gvpm_status otherwise; the message is
 *     available from gvpm_last_error().  No exception crosses this boundary (the reference
 *     throws from SLog(EError), the host shim re-raises).
 *   - host arrays are caller-owned and only read during the call; device buffers belong to
 *     the context and are reused (grow-only) across iterations.
 *   - Float is fp32 (north-star), Spectrum is 3 floats (SPECTRUM_SAMPLES=3).
 *   - offsets are ordered {Left(-1,0), Right(+1,0), Top(0,+1), Bottom(0,-1)} as
 *     generateOffsetPos, gvpm/shift/shift_utilities.h:255-261 / EPixel gvpm_struct.h:354-359.
 *   - there is no CPU fallback: without a CUDA device gvpm_ctx_create fails.
 */
#ifndef GVPM_B200_H
#define GVPM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GVPM_ABI_VERSION 1

typedef struct gvpm_ctx gvpm_ctx; /* opaque, one per device, externally synchronised */

enum gvpm_status {
  GVPM_OK = 0,
  GVPM_ERR_INVALID = -1,  /* bad argument / call order */
  GVPM_ERR_CUDA = -2,     /* CUDA runtime error (text in gvpm_last_error) */
  GVPM_ERR_NO_DEVICE = -3,/* no sm_100 device: the product path has no CPU fallback */
  GVPM_ERR_UNSUPPORTED = -4
};

/* Parent-vertex type of a photon / beam (PathVertex::EVertexType of vertex c-1 on the light
 * path; gvpm/shift/operation/shift_diffuse.cpp:18-88).  GVPM_PARENT_OTHER marks a glossy or
 * specular surface parent: the reference routes those to the manifold shift
 * (shift_utilities.h:112-136), which is out of scope; the gather treats it as the reference
 * does with useManifold=false (shift fails, weight 1). */
enum gvpm_parent_type {
  GVPM_PARENT_EMITTER = 0,
  GVPM_PARENT_SURFACE = 1,
  GVPM_PARENT_MEDIUM = 2,
  GVPM_PARENT_OTHER = 3
};

enum gvpm_phase_type { GVPM_PHASE_ISOTROPIC = 0, GVPM_PHASE_HG = 1 };

/* ELightingEffects bits, src/integrators/volume_utils.h:95-103 */
enum gvpm_lighting_mode {
  GVPM_SURF2MEDIA = 1 << 2,
  GVPM_MEDIA2MEDIA = 1 << 4,
  GVPM_ALL2MEDIA = (1 << 2) | (1 << 4)
};

/* Homogeneous medium + phase function: src/medium/homogeneous.cpp:432-513 (balance strategy,
 * equal sigma_t across channels is required by the reference, :188-201), phase/isotropic.cpp:76,
 * phase/hg.cpp:107-110. */
typedef struct gvpm_medium {
  float sigma_s[3];
  float sigma_a[3];
  int32_t phase_type;      /* gvpm_phase_type */
  float hg_g;
  float sampling_weight;   /* mediumSamplingWeight; 1 for volume-only renders (gvpm.cpp:135-141) */
} gvpm_medium;

/* The subset of GPMConfig (gvpm/gvpm_struct.h:106-333) the gather reads. */
typedef struct gvpm_config {
  int32_t max_depth;        /* maxDepth (-1/0 = unbounded; test is maxDepth > 0) */
  int32_t min_depth;        /* minDepth */
  int32_t lighting_mode;    /* lightingInteractionMode bits (gvpm_lighting_mode) */
  int32_t use_mis;          /* useMIS == "area" */
  int32_t use_shift_null;   /* useShiftNull (mixed shift / spatial relaxation) */
  int32_t path_set;         /* pathSet checkerboard (shift_volume_photon.cpp:689-697) */
  int32_t power_heuristic;  /* powerHeuristic */
  int32_t kernel_3d;        /* 1: bre3d (default "bre"), 0: bre2d */
  int32_t film_w, film_h;   /* film size, for the right/top border rule (:843-846) */
  float shadow_maxt_scale;  /* the reference passes maxt = lProj*ShadowEpsilon (=1e-3f) to the
                               reconnection shadow ray, shift_volume_photon.cpp:396; kept as a
                               parameter so the quirk is visible.  Default 1e-3f. */
  float epsilon;            /* Epsilon (include/mitsuba/core/constants.h:24-30, 1e-4f in single
                               precision): mint of the offset rays and of the shadow ray */
  int32_t long_beams;       /* photon beams were converted to long beams (convertLong, gvpm.cpp:884-887) */
  uint32_t rng_seed;        /* G-Beams-3D draws two uniforms per (camera ray, beam) from the integrator's
                               sampler in traversal order (shift_volume_beams.h:224,245), which no parallel
                               gather can reproduce; they are replaced by a counter-based hash of
                               (rng_seed, px, py, edge, beam index, dimension) — DESIGN.md §6 */
  int32_t beam_kernel_1d;   /* G-Beams: 0 = "beam3d" (EBeamBeam3D_Optimized), 1 = "beam1d" (EBeamBeam1D, for which
                               GPMIntegrator forces newShiftBeam = true, gvpm.cpp:96-98) */
  int32_t sppm_primal;      /* 1: the point gather runs sppm's primal BeamRadianceEstimator::query
                               (photonmapper/bre.cpp:167-259) instead of gvpm's gradient functor: see gvpm_gather_sppm_bre */
} gvpm_config;

/* Volume photons, flattened from GPhotonNodeData + its light Path
 * (gvpm/gvpm_accel.h:17-65,119-199).  c = vertexId of the photon on its light path. */
typedef struct gvpm_photon_soa {
  const float *pos;           /* [n*3] vertex(c).position */
  const float *flux;          /* [n*3] running importance weight (gvpm_accel.h:134-148) */
  const float *parent_pos;    /* [n*3] vertex(c-1).position; wi = normalize(parent - pos) */
  const float *pred_pos;      /* [n*3] vertex(c-2).position, or (1,1,1) when c < 3
                                        (shift_volume_photon.cpp:431) */
  const float *parent_n;      /* [n*3] geometric normal of a surface / emitter parent */
  const float *prefix_flux;   /* [n*3] prod_{i<c-1} weight*rr*edgeWeight (:415-422) */
  const float *parent_albedo; /* [n*3] diffuse reflectance of a surface parent */
  const float *parent_pdf;    /* [n] vertex(c-1).pdf[EImportance], area measure */
  const float *edge_pdf;      /* [n] edge(c-1).pdf[EImportance] */
  const float *rr_weight;     /* [n] vertex(c-1).rrWeight */
  const uint8_t *parent_type; /* [n] gvpm_parent_type */
  const uint8_t *depth;       /* [n] c-1 = number of preceding interactions */
  const uint32_t *path_id;    /* [n] GPhotonNodeData::pathID */
} gvpm_photon_soa;

/* Camera-ray medium segments with their four offset segments: what
 * computeVolumeGradientPhotonBRE builds per (gather point, medium edge), gvpm.cpp:1008-1042,
 * plus the per-offset data ShiftGatherPoint caches (shift_cameraPath.h:29-140,
 * gvpm_struct.h:585-631). */
typedef struct gvpm_ray_soa {
  const float *o;           /* [n*3] vertex(e).position */
  const float *d;           /* [n*3] unit direction */
  const float *mint;        /* [n]   Epsilon */
  const float *maxt;        /* [n]   beamDist - Epsilon */
  const float *edge_len;    /* [n]   edge(e).length */
  const float *eye_contrib; /* [n*3] getWeightBeam(e-1)*getWeightVertex(e) */
  const float *xi;          /* [n]   the sampler->next1D() of gvpm.cpp:1042 */
  const int32_t *px;        /* [n]   int(samplePosition.x) */
  const int32_t *py;        /* [n] */
  const int32_t *edge_id;   /* [n]   e (currEdge) */
  const uint8_t *off_valid; /* [n*4] validVolumeEdge(e, medium) */
  const float *off_o;       /* [n*4*3] */
  const float *off_d;       /* [n*4*3] -edge_k(e).d */
  const float *off_len;     /* [n*4]   edge_k(e).length */
  const float *off_eye;     /* [n*4*3] eyeShiftContrib */
  const float *off_sensor;  /* [n*4]   sensorMIS(e, base, .,.) */
} gvpm_ray_soa;

/* G-VPM distance samples: what computeVolumeGradientPhoton draws on the host per gather point
 * (gvpm.cpp:1141-1175: edge selection by the discrete CDF, then
 * HomogeneousMedium::sampleDistance(ray, mRec, sampler, EDistanceAlwaysValid), homogeneous.cpp:293-430).
 * One entry per (pixel, camera sample); `ray` indexes the gvpm_ray_soa record of the chosen medium edge.
 * Uploaded, the distance is sampled on the host (it consumes the integrator's sampler and libm's logf), so the
 * query points are bit-identical inputs for the gather; gvpm_generate_vpm_samples draws them on the device. */
typedef struct gvpm_vpm_sample_soa {
  const uint32_t *ray;         /* [n]   index into the uploaded rays */
  const float *t;              /* [n]   mRec.t (the query point is o + t*d) */
  const float *transmittance;  /* [n*3] mRec.transmittance */
  const float *pdf_success;    /* [n]   mRec.pdfSuccess (baseDistPDF) */
  const float *pdf_sel;        /* [n]   selBeam[sampleIndex] (pdfSelSection) */
  const float *radius;         /* [n]   BBPourcentageCONST * gp.scaleVol of the pixel (gvpm.cpp:1131) */
} gvpm_vpm_sample_soa;

/* Photon beams, flattened from LTPhotonBeam + its light Path (gvpm/gvpm_beams.h:18-84,
 * photonmapper/beams_struct.h:25-110).  A beam is the light-path edge i = edgeID from vertex(i) (the
 * beam origin, which is also the PARENT vertex of the diffuse reconnection, shift_volume_beams.cpp:430-436)
 * to vertex(i+1). */
typedef struct gvpm_beam_soa {
  const float *origin;        /* [n*3] vertex(i).position (p1) */
  const float *end;           /* [n*3] vertex(i+1).position (p2); dir and length are derived as setEndPoint does */
  const float *flux;          /* [n*3] prod_{k<i} rr*weight*edgeWeight * vertex(i).weight * rr_i, without the
                                        transmittance of edge i (gvpm_beams.h:29-35) */
  const float *prefix_flux;   /* [n*3] prod_{k<=i-1} weight*rr*edgeWeight (shift_volume_beams.cpp:442-449) */
  const float *parent_n;      /* [n*3] geometric normal of a surface / emitter origin vertex */
  const float *parent_albedo; /* [n*3] diffuse reflectance of a surface origin vertex */
  const float *pred_pos;      /* [n*3] vertex(i-1).position, or (1,1,1) when i < 2 (:457) */
  const float *end_n;         /* [n*3] geometric normal of vertex(i+1) when it lies on a surface */
  const float *parent_pdf;    /* [n]   vertex(i).pdf[EImportance] (area measure) */
  const float *rr_weight;     /* [n]   vertex(i).rrWeight */
  const uint8_t *parent_type; /* [n]   gvpm_parent_type of vertex(i) */
  const uint8_t *end_on_surface; /* [n] vertex(i+1).isOnSurface() */
  const uint8_t *depth;       /* [n]   beam->depth = i */
  const uint32_t *path_id;    /* [n]   LTPhotonBeam::pathID */
} gvpm_beam_soa;

/* Photon planes (0D kernel), flattened from LTPhotonPlane (gvpm/gvpm_plane.h:18-46, photonmapper/plane_struct.h:18-58):
 * the photon beam of light-path edge i extended by a second sampled direction/length on the host
 * (LTPhotonPlane::transformBeam, gvpm_plane.h:53-73; mirrored by gvpm_host::transformBeam).  The plane functor
 * reads no parent-vertex data (its shift keeps origin and w0, shift_volume_planes.h:263-416). */
typedef struct gvpm_plane_soa {
  const float *origin;    /* [n*3] _ori = vertex(i).position */
  const float *w0;        /* [n*3] _w0 = edge(i).d (unit) */
  const float *length0;   /* [n]   _length0 = edge(i).length */
  const float *w1;        /* [n*3] _w1 = sampled scattering direction (unit) */
  const float *length1;   /* [n]   _length1 = sampled distance */
  const float *flux;      /* [n*3] _flux, as the beam flux (gvpm_plane.h:36-44) */
  const int32_t *edge_id; /* [n]   edgeID = i (the t0 Jacobian factor is skipped for i == 1, :357-359) */
} gvpm_plane_soa;

/* Occluder triangles for the reconnection shadow ray (scene->rayIntersect,
 * shift_volume_photon.cpp:396-402), tested as Triangle::rayIntersect
 * (include/mitsuba/core/triangle.h:109-145). */

/* Floats per ray in the gather output: mediumFlux[3], shiftedMediumFlux[4][3],
 * weightedMediumFlux[4][3] (AbstractVolumeGradientRecord, shift_volume_photon.h:17-20). */
#define GVPM_OUT_FLOATS 27

/* ---- context ------------------------------------------------------------------------- */
int gvpm_abi_version(void);
int gvpm_ctx_create(int device, gvpm_ctx **out);
int gvpm_ctx_destroy(gvpm_ctx *ctx);
const char *gvpm_last_error(const gvpm_ctx *ctx); /* ctx may be NULL: last create error */
int gvpm_sync(gvpm_ctx *ctx);
/* the CUDA stream (cudaStream_t) all work of this context is enqueued on */
void *gvpm_stream(gvpm_ctx *ctx);

/* ---- scene constants ----------------------------------------------------------------- */
int gvpm_set_medium(gvpm_ctx *ctx, const gvpm_medium *m);
int gvpm_set_config(gvpm_ctx *ctx, const gvpm_config *c);
/* Occluders: the triangles the reconnection shadow rays test, typically every triangle of the
 * scene (flattenOccluders).  n_tri = 0 clears them; more than GVPM_MAX_OCCLUDERS fails with
 * GVPM_ERR_INVALID.  When the selected path (gvpm_set_occluder_accel) is the BVH, the call builds
 * it on the device once for the set; the gathers then use it until the next call. */
#define GVPM_MAX_OCCLUDERS (1u << 24)
int gvpm_set_occluders(gvpm_ctx *ctx, const float *tri_xyz /* [n_tri*9] */, size_t n_tri);
/* Path of the shadow-ray any-hit.  AUTO (the default): the flat list up to 32 triangles, the BVH
 * above.  LIST and BVH force one path; both give the same answer for every ray.  Any other value
 * fails with GVPM_ERR_INVALID.  Selecting the BVH for the current set builds it if needed. */
enum gvpm_occluder_accel { GVPM_OCC_AUTO = 0, GVPM_OCC_LIST = 1, GVPM_OCC_BVH = 2 };
int gvpm_set_occluder_accel(gvpm_ctx *ctx, int mode);
/* the path the gathers take for the current set: GVPM_OCC_LIST or GVPM_OCC_BVH (0 for ctx = NULL) */
int gvpm_occluder_accel_kind(const gvpm_ctx *ctx);
/* Any-hit of n rays (host arrays: o, d [n*3], mint, maxt [n]) against the occluders, through the
 * path the gathers take and the same device code as their shadow rays; hit[i] = 0 or 1.  A parity
 * and timing aid; blocking. */
int gvpm_occluded(gvpm_ctx *ctx, const float *o, const float *d, const float *mint, const float *maxt, size_t n,
                  uint8_t *hit);

/* ---- photon points: replaces GPhotonMap::tryAppend/build (gvpm_accel.h:119-203,
 *      include/mitsuba/core/kdtree.h:326-378) and the GradientBeamRadianceEstimator
 *      constructor + buildHierarchy (gvpm_accel.cpp:10-55) ---------------------------------- */
int gvpm_upload_photons(gvpm_ctx *ctx, const gvpm_photon_soa *p, size_t n);
/* Device-resident variant for multi-GPU: returns the context's raw staging buffer sized for n
 * photons (the 13 SoA arrays back to back, each 256-byte aligned, in the field order of
 * gvpm_photon_soa).  Rank 0 fills it with gvpm_upload_photons, the host broadcasts `bytes`
 * bytes at `dev` over NCCL, and every rank then calls gvpm_build_points. */
int gvpm_photon_staging(gvpm_ctx *ctx, size_t n, void **dev, size_t *bytes);
/* Multi-GPU / pipelined use.  The context owns TWO photon staging buffers; gvpm_photon_staging_select chooses the
 * one that gvpm_photon_staging, gvpm_upload_photons(_slice) and gvpm_build_points work on, so that the photon set
 * of iteration k+1 can be uploaded / all-gathered into one buffer while iteration k is built and gathered from the
 * other.  gvpm_upload_photons_slice copies `count` photons (the host arrays point at the slice's first element)
 * into elements [begin, begin+count) of the selected buffer, sized for n_total by a previous gvpm_photon_staging
 * call, asynchronously on `stream` (a cudaStream_t; NULL = the context's stream): every rank uploads 1/G of the set
 * over its own PCIe link and the ranks all-gather the 13 field arrays in place over NVLink.
 * gvpm_photon_staging_layout gives each field's byte offset in the staging buffer and its bytes per photon. */
int gvpm_photon_staging_select(gvpm_ctx *ctx, int which /* 0 or 1 */);
int gvpm_photon_staging_layout(size_t n, size_t field_offset[13], size_t field_elem_bytes[13]);
int gvpm_upload_photons_slice(gvpm_ctx *ctx, const gvpm_photon_soa *p, size_t n_total, size_t begin, size_t count,
                              void *stream);
/* Peer exchange of the photon slices over NVLink COPY ENGINES (no SMs: the transfers overlap the gather kernels,
 * which an SM-based collective cannot while persistent kernels fill the machine).  For contexts in different
 * processes (one per GPU) the staging buffers and four events are shared through CUDA IPC:
 *   gvpm_peer_export   writes this context's GVPM_PEER_BLOB_BYTES-byte blob (both staging buffers must have been
 *                      sized with gvpm_photon_staging for the largest iteration: once exported they cannot grow, and a
 *                      gvpm_photon_staging / gvpm_upload_photons call that needs more fails with GVPM_ERR_INVALID);
 *   gvpm_peer_connect  takes the blobs of all n_peers contexts (rank order, own one included) and maps them;
 *   gvpm_peer_push_photon_slice  copies photons [begin, begin+count) of staging buffer `which` into the same place of
 *                      every peer's buffer `which` with cudaMemcpyAsync on internal streams, after the work queued
 *                      on `after_stream` (NULL = the context's stream; e.g. the slice's H2D upload) and after each
 *                      peer's last build from that buffer;
 *   gvpm_peer_wait_photons       makes the context's stream wait until every peer's slice has landed in buffer
 *                      `which`.
 * Interprocess events order work only with respect to records already ISSUED: the host processes must pass a
 * barrier once per iteration between a rank's push / build calls and the other ranks' waits on them (bench.py). */
#define GVPM_PEER_BLOB_BYTES 384
int gvpm_peer_export(gvpm_ctx *ctx, void *blob /* [GVPM_PEER_BLOB_BYTES] */);
int gvpm_peer_connect(gvpm_ctx *ctx, const void *blobs /* [n_peers * GVPM_PEER_BLOB_BYTES] */, int n_peers,
                      int self_index);
int gvpm_peer_push_photon_slice(gvpm_ctx *ctx, int which, size_t n_total, size_t begin, size_t count,
                                void *after_stream);
int gvpm_peer_wait_photons(gvpm_ctx *ctx, int which);
/* How gvpm_peer_push_photon_slice moves the bytes: sm_ctas > 0 (default 32) = one kernel of that many CTAs on a
 * highest-priority stream that reads the slice once and stores it into every peer's buffer through the peer mappings;
 * 0 = cudaMemcpyAsync per field and peer on the copy engines (also the fallback for slices that are not 16-byte
 * aligned in every field). */
int gvpm_peer_push_mode(gvpm_ctx *ctx, int sm_ctas);
/* Photon DISPATCH between ranks: the scalable form of the exchange for image-sharded G-BRE iterations (SURVEY.md §8e;
 * replaces what the reference does with one shared-memory photon map, gvpm.cpp:453 + the BlockScheduler of :999-1052,
 * when the gather points are split over several GPUs).  Instead of copying every photon to every rank, each rank
 * classifies the photons of ITS slice against every receiver's perspective grid and ray-occupancy mask (the keep test
 * of the receiver's own gvpm_build_points_for_rays) and writes the 128-byte gather records of the photons a receiver
 * can reach straight into that receiver's inbox over NVLink (peer-mapped stores; one fused pack + exchange kernel).
 * A photon crosses the link once per rank that needs it, and a receiver builds over what it was sent only.
 *   gvpm_dispatch_export   after gvpm_upload_rays (the rank's own tile rays; they must be concurrent, i.e. a pinhole's
 *                          primary rays, else GVPM_ERR_UNSUPPORTED - use the gvpm_peer_* exchange): allocates two
 *                          inboxes of n_peers regions x region_cap records (region_cap >= the largest slice any rank
 *                          dispatches), publishes the ray fit and the occupancy mask, writes the rank's blob;
 *   gvpm_dispatch_connect  takes the blobs of all ranks (rank order, own one included).  Contexts of one process (tests,
 *                          one host thread driving several GPUs) are wired directly, others through CUDA IPC;
 *   gvpm_dispatch_photons  classifies photons [begin, begin+count) of the selected staging buffer (sized for n_total by
 *                          gvpm_photon_staging) for search radius `radius` and writes them into inbox `which` of every
 *                          rank, on an internal highest-priority stream, after the work queued on `after_stream`
 *                          (NULL = the context's stream) and after every receiver's release of that inbox; with
 *                          after_stream = gvpm_stream(ctx) itself the dispatch is queued IN the context's stream (e.g.
 *                          between a build and its gather, where no persistent gather kernel holds the SMs);
 *   gvpm_build_dispatched  waits (on the context's stream) until every rank's records for inbox `which` have landed,
 *                          then builds the perspective grid over them: the gathers (gvpm_gather_bre*) run as after
 *                          gvpm_build_points_for_rays, with identical neighbour sets and results;
 *   gvpm_dispatch_release  stream-ordered: the gathers from inbox `which` are done, the senders may refill it;
 *   gvpm_dispatch_join     the context's stream waits for this rank's dispatches issued so far (end of a timed region);
 *   gvpm_dispatch_status   synchronises and reports the records received per sender for inbox `which`
 *                          (counts[GVPM_MAX_PEERS], may be NULL) and any protocol failure (a peer that never signalled).
 * No host barrier is needed: ordering between ranks goes through generation flags in device memory.  Every rank calls
 * dispatch / build / release once per iteration and inbox, in the same order. */
#define GVPM_MAX_PEERS 8
#define GVPM_DISPATCH_BLOB_BYTES 512
int gvpm_dispatch_export(gvpm_ctx *ctx, int n_peers, size_t region_cap, void *blob /* [GVPM_DISPATCH_BLOB_BYTES] */);
int gvpm_dispatch_connect(gvpm_ctx *ctx, const void *blobs /* [n_peers * GVPM_DISPATCH_BLOB_BYTES] */, int n_peers,
                          int self_index);
int gvpm_dispatch_photons(gvpm_ctx *ctx, int which, size_t n_total, size_t begin, size_t count, float radius,
                          void *after_stream);
int gvpm_build_dispatched(gvpm_ctx *ctx, int which, float radius, uint32_t *n_kept);
int gvpm_dispatch_release(gvpm_ctx *ctx, int which);
int gvpm_dispatch_join(gvpm_ctx *ctx);
int gvpm_dispatch_status(gvpm_ctx *ctx, uint32_t counts[GVPM_MAX_PEERS], int which);
/* Result collection ("the primal and gradient buffers gathered at the end of each iteration"): a device buffer that other
 * ranks can write (CUDA IPC).  The root creates it, the ranks open it and copy their rows in with a plain device-to-device
 * copy on a side stream - copy engines over NVLink, no SMs taken from the gather kernels - then signal; the root waits for
 * every rank's signal on its stream before it reads the image.  (Needs gvpm_dispatch_connect: the signals are generation
 * flags in the root's control block, one set per buffer `which`.) */
#define GVPM_SHARED_HANDLE_BYTES 96
int gvpm_shared_buffer_create(gvpm_ctx *ctx, size_t bytes, void **dev, void *handle /* [GVPM_SHARED_HANDLE_BYTES] */);
int gvpm_shared_buffer_open(gvpm_ctx *ctx, const void *handle, void **dev);
int gvpm_collect_signal(gvpm_ctx *ctx, int which, int root, void *stream /* the stream the copy was queued on */);
int gvpm_collect_wait(gvpm_ctx *ctx, int which);
/* Hilbert sort + implicit 32-ary AABB hierarchy for search radius `radius`
 * (= bsphereR*globalScaleVolume*0.01, gvpm.cpp:989) */
int gvpm_build_points(gvpm_ctx *ctx, float radius);

/* gvpm_build_points restricted to the photons the currently uploaded rays can reach (call gvpm_upload_rays first).
 * Meant for image-tile sharding over GPUs (SURVEY.md §8e): a rank that gathers only its own tiles' rays sorts and
 * boxes only the part of the photon set those rays cross.  The ray segments, dilated by `radius`, mark the cells of a
 * 64^3 occupancy grid over their bounding box; photons in unmarked cells are left out.  Conservative: the left-out
 * photons fail the neighbour predicate (gvpm_accel.h:297-301) of every uploaded ray, so every gather returns what
 * it returns after gvpm_build_points.  The hierarchy is valid for this ray set only - the gathers fail with
 * GVPM_ERR_INVALID once other rays are uploaded, until the next build.  n_kept (may be NULL): photons kept. */
int gvpm_build_points_for_rays(gvpm_ctx *ctx, float radius, uint32_t *n_kept);
/* When the lines of ALL uploaded rays pass through one point (the primary rays of a pinhole sensor: the first medium
 * edge of every pixel), gvpm_build_points_for_rays builds a PERSPECTIVE GRID instead of a box hierarchy: photons are
 * binned by the direction in which that point sees them, in cells about one pixel wide (coarser cells for photons
 * close to the point, whose search sphere covers many pixels), and a ray finds all its neighbours in the 3x3 cells
 * around its own direction - no traversal.  Same neighbour sets, same results.  n_kept (photons some ray can reach)
 * then costs one device read-back: pass NULL when it is not needed.  gvpm_accel_kind: 0 = box hierarchy, 1 = grid. */
int gvpm_accel_kind(const gvpm_ctx *ctx);
/* Read-only view of the perspective grid the last build made (diagnostics, e.g. tools/trav_census.py): the grid's
 * parameters as the device sees them (struct FrustumGrid of gvpm_device.cuh, all 4-byte fields; grid_bytes must be its
 * size) and, when cell_start is not NULL, its cell_start array (first sorted slot of every key, NEAR and DROP included,
 * then the end: *n_entries values; cap = room in cell_start).  Either output may be NULL.  Fails when the last build
 * made a box hierarchy. */
int gvpm_frustum_grid(gvpm_ctx *ctx, void *grid, size_t grid_bytes, uint32_t *cell_start, size_t cap, size_t *n_entries);
/* Optional: the axis of the perspective grid's projection plane (default: the mean direction of the uploaded rays).
 * The sensor's viewing direction is the natural choice; ranks of a sharded image that all pass the same vector project
 * on the same plane, which lets gvpm_dispatch_photons classify a photon once for all receivers.  NULL: back to the
 * default.  Any direction within ~69 degrees of every ray works; results do not depend on it. */
int gvpm_set_view_direction(gvpm_ctx *ctx, const float dir[3]);

/* ---- camera rays --------------------------------------------------------------------- */
int gvpm_upload_rays(gvpm_ctx *ctx, const gvpm_ray_soa *r, size_t n);
/* same idea for rays: staging buffer (16 SoA arrays, 256-byte aligned, field order of
 * gvpm_ray_soa) to be filled on the device, then gvpm_commit_rays packs it. */
int gvpm_ray_staging(gvpm_ctx *ctx, size_t n, void **dev, size_t *bytes);
int gvpm_commit_rays(gvpm_ctx *ctx);

/* ---- gathers: replace bre->query(ray, medium, gRec, xi) over all gather points,
 *      gvpm.cpp:999-1052 + gvpm_accel.h:268-312 + shift_volume_photon.cpp:658-856 ------------ */
/* out: [n_rays*27] host floats (un-normalised: the caller divides by nbPathVolume and folds
 * into the APA running mean, gvpm.cpp:1054-1069).  counts (may be NULL): [n_rays*2] =
 * {geometric neighbours, contributing neighbours} per ray. */
int gvpm_gather_bre(gvpm_ctx *ctx, float *out, uint32_t *counts);
/* same, results left on the device (pointers owned by the context, valid until the next call) */
int gvpm_gather_bre_device(gvpm_ctx *ctx, const float **out_dev, const uint32_t **counts_dev);
/* same, written to caller-provided device memory (e.g. a peer-mapped / NCCL buffer) */
int gvpm_gather_bre_into(gvpm_ctx *ctx, float *out_dev, uint32_t *counts_dev);
/* gvpm_gather_bre_device and gvpm_gather_bre_into are ASYNCHRONOUS: the traversal and shading kernels are queued on the
 * context's stream with no host round trip in between.  The (ray, photon) pair list between the two kernels is grow-only
 * and sized from earlier gathers; if it overflows (first iteration of a render, or a sudden growth of the neighbour
 * count) the gather is incomplete: gvpm_sync() detects that and re-runs it, so results are final once gvpm_sync has
 * returned GVPM_OK.  Consuming them earlier on the stream is safe whenever an earlier gather of similar size has
 * completed.  The host-returning gathers (gvpm_gather_bre, _host, gvpm_gather_sppm_bre) do this check themselves. */

/* The whole per-iteration tail in one call: gvpm_upload_rays + gvpm_gather_bre, pipelined - rays go up in chunks on a
 * copy stream while earlier chunks are traversed and shaded and their results stream back, so both PCIe directions
 * and the SMs are busy at once.  r and out should be page-locked (cudaHostAlloc / cudaHostRegister) for the copies
 * to overlap; pageable memory works but serialises.  out: [n*27] host floats, un-normalised. */
int gvpm_gather_bre_host(gvpm_ctx *ctx, const gvpm_ray_soa *r, size_t n, float *out);

/* ---- sppm primal BRE: replaces `new BeamRadianceEstimator(photonMap, 120, breInitSize, true)` + bre->query(ray, medium,
 *      maxDepth - beam.depth, use3DKernel, sampler) * beam.weight over all gather-point beams, sppm.cpp:926-981 +
 *      bre.cpp:29-55,167-259.  Requires gvpm_config.sppm_primal = 1 (checked).  Inputs are the same containers:
 *      photons: pos, flux = photon.getPower(), parent_pos = pos - photon.getDirection() (so that wi = -direction),
 *      depth = photon.getDepth(); the other arrays are not read.  rays: o = beam.p1, d, mint = Epsilon, maxt =
 *      distTotal - Epsilon, eye_contrib = beam.weight, edge_id = beam.depth (maxDepth - beam.depth is formed from
 *      gvpm_config.max_depth; -1 = unbounded); offsets are ignored.  edge_len is not part of sppm's predicate: the
 *      traversal is bounded by max(edge_len, maxt), so it may be left at 0.  The 3-D kernel's per-PHOTON sampler->next1D()
 *      (bre.cpp:217) is replaced by the counter-based hash of (rng_seed, px, py, edge, photon index).
 *      out: [n_rays*3] = sum of the query results * beam.weight WITHOUT m_scaleFactor (the caller multiplies by
 *      1 / shotParticles, sppm.cpp:922).  counts (may be NULL): [n_rays*2] = {photons passing the geometric tests,
 *      same after the depth filter}. */
int gvpm_gather_sppm_bre(gvpm_ctx *ctx, float *out, uint32_t *counts);

/* ---- sppm primal photon beams: replaces beamMap->build(EBVHAccel) + BeamRadianceQuery + beamMap->query(bRadQuery) over
 *      all gather-point beams, sppm.cpp:803,823-860 + photonmapper/beams.h:29-223 + beams_accel.h:90-243, for the four
 *      beam x beam techniques of EVolumeTechnique (volTechnique = beam1d | beam3d_naive | beam3d_egsr | beam3d).
 *      Call order: gvpm_upload_beams (origin, end, flux, depth are read; the parent arrays may hold anything),
 *      gvpm_build_beams(radius), gvpm_upload_rays (o = beam.p1, d, mint = Epsilon, maxt = distTotal - Epsilon,
 *      edge_len = distTotal, eye_contrib = beam.weight, edge_id = camera beam.depth; offsets ignored).  The depth
 *      window is formed like sppm.cpp:853-854 from gvpm_config.max_depth (-1 = unbounded) and min_depth.  The
 *      sampler->next1D() draws are replaced by the counter-based hash of (rng_seed, px, py, edge, beam index, dimension);
 *      the naive technique samples per sub-beam (dimension = 2 + 2*sub-beam ordinal, +1).
 *      out: [n_rays*3] = sum of bRadQuery.Li * beam.weight, WITHOUT the 1 / shotParticles normalisation (:863).
 *      counts (may be NULL): [n_rays*2] = {accepted (ray, beam) pairs - (ray, sub-beam) for the naive technique -,
 *      same after the depth filters}. */
enum gvpm_beam_technique {
  GVPM_BEAM_1D = 0,          /* EBeamBeam1D */
  GVPM_BEAM_3D_NAIVE = 1,    /* EBeamBeam3D_Naive */
  GVPM_BEAM_3D_EGSR = 2,     /* EBeamBeam3D_EGSR */
  GVPM_BEAM_3D_OPTIMIZED = 3 /* EBeamBeam3D_Optimized */
};
int gvpm_gather_sppm_beams(gvpm_ctx *ctx, int technique, float *out, uint32_t *counts);
/* per-ray lists of accepted beam indices (bit 31 = passes the depth filters; one entry per accepted sub-beam for the
 * naive technique), CSR like gvpm_dump_neighbours_bre */
int gvpm_dump_neighbours_sppm_beams(gvpm_ctx *ctx, int technique, uint64_t *offsets, uint32_t *idx, size_t cap);

/* Parity aid: neighbour index sets in CSR form.  offsets: [n_rays+1]; idx: capacity `cap`
 * entries, original photon index with bit 31 set when the photon also passes the depth /
 * interaction-mode / pathSet filters; every ray's entries in ascending photon index order (this and the
 * other gvpm_dump_neighbours_* calls).  Returns GVPM_ERR_INVALID when cap is too small
 * (offsets[n_rays] then holds the needed size). */
int gvpm_dump_neighbours_bre(gvpm_ctx *ctx, uint64_t *offsets, uint32_t *idx, size_t cap);

/* ---- G-Beams ("beam3d", or "beam1d" with gvpm_config.beam_kernel_1d): replaces beamMap->build(EBVHAccel) + beamMap->query(radQuery) over all gather
 *      points, gvpm.cpp:880-986 + beams_accel.h:90-243 + shift_volume_beams.cpp:139-539,748-786 ---------------
 * gvpm_build_beams cuts the beams into sub-beams of averageLength/10 and builds the hierarchy for beam radius
 * `radius` (= bsphereR*globalScaleVolume*0.01, gvpm.cpp:881).  out: [n_rays*27], un-normalised (the caller
 * divides by nbPathBeams, gvpm.cpp:958-964); counts (may be NULL, faster): [n_rays*2] = {(ray, beam) pairs
 * with a valid kernel record, pairs that also pass the depth/mode/pathSet filters}. */
int gvpm_upload_beams(gvpm_ctx *ctx, const gvpm_beam_soa *b, size_t n);
int gvpm_build_beams(gvpm_ctx *ctx, float radius);
/* number of sub-beams the uploaded beam set is cut into (SubBeamBVH's m_beamCount, beams_accel.h:107-110) */
uint64_t gvpm_beam_subbeam_count(const gvpm_ctx *ctx);
int gvpm_gather_beams(gvpm_ctx *ctx, float *out, uint32_t *counts);
/* same, results left on the device (pointers owned by the context, valid until the next gather; the work is queued on the
 * context's stream, call gvpm_sync before reading them from another stream).  counts_dev NULL: no counts (faster). */
int gvpm_gather_beams_device(gvpm_ctx *ctx, const float **out_dev, const uint32_t **counts_dev);
/* per-ray sets of beam indices (bit 31 = contributes), CSR like gvpm_dump_neighbours_bre */
int gvpm_dump_neighbours_beams(gvpm_ctx *ctx, uint64_t *offsets, uint32_t *idx, size_t cap);

/* ---- G-Planes 0D ("plane0d"): replaces PhotonPlaneBVH construction + planeBVH->query(radQuery) over all gather
 *      points, gvpm.cpp:782-878 + plane_accel.h:84-211 + plane_struct.h:104-192 + shift_volume_planes.h:57-101,
 *      263-453 ----------------------------------------------------------------------------------------------
 * Rays as for the other gathers (the camera must be inside the medium, gvpm.cpp:785-787; ray.maxt = edge length
 * - Epsilon, :833-837).  The functor uses neither eyeContrib nor the depth / mode / pathSet filters, and has no
 * right/top border rule (shift_volume_planes.h:57-101) - restated as is.  out: [n_rays*27], un-normalised (the
 * caller divides by nbPathBeams, :850-856); counts (may be NULL): [n_rays*2] = {planes intersected, same}. */
int gvpm_upload_planes(gvpm_ctx *ctx, const gvpm_plane_soa *p, size_t n);
int gvpm_build_planes(gvpm_ctx *ctx);
int gvpm_gather_planes(gvpm_ctx *ctx, float *out, uint32_t *counts);
int gvpm_gather_planes_device(gvpm_ctx *ctx, const float **out_dev, const uint32_t **counts_dev); /* as gvpm_gather_beams_device */
/* per-ray sets of plane indices (bit 31 always set: every intersected plane contributes), CSR */
int gvpm_dump_neighbours_planes(gvpm_ctx *ctx, uint64_t *offsets, uint32_t *idx, size_t cap);

/* ---- G-VPM: replaces gradientPhotonMap->evaluate(gRec, p, querySize) over all camera distance
 *      samples, gvpm.cpp:1141-1185 + kdtree.h:675-731 + shift_volume_photon.cpp:489-655 ----------------
 * Call order: gvpm_upload_photons, gvpm_build_points(radius >= every sample radius), gvpm_upload_rays
 * (one record per (gather point, medium edge)), gvpm_upload_vpm_samples (or gvpm_generate_vpm_samples, below),
 * gvpm_gather_vpm.
 * out: [n_rays*27] with the reference's 1/nbCameraSamples normalisation applied (gvpm.cpp:1177-1182);
 * mvol (may be NULL): [n_rays] the MVol of gvpm.cpp:1175 = photons found by the range queries of the
 * ray's samples (drives the per-pixel radius update :1191-1195, which stays on the host);
 * sample_counts (may be NULL): [n_samples*2] = {found, contributing}. */
int gvpm_upload_vpm_samples(gvpm_ctx *ctx, const gvpm_vpm_sample_soa *s, size_t n);
int gvpm_gather_vpm(gvpm_ctx *ctx, int nb_camera_samples, float *out, uint32_t *mvol, uint32_t *sample_counts);
int gvpm_gather_vpm_device(gvpm_ctx *ctx, int nb_camera_samples, const float **out_dev, const uint32_t **mvol_dev);
/* per-SAMPLE neighbour index sets, same CSR convention as gvpm_dump_neighbours_bre */
int gvpm_dump_neighbours_vpm(gvpm_ctx *ctx, int nb_camera_samples, uint64_t *offsets, uint32_t *idx, size_t cap);
/* The distance samples drawn on the device from the context's current ray set, in place of gvpm_upload_vpm_samples:
 * what gvpm_synth_vpm_samples (the host restatement of gvpm.cpp:1141-1175 + HomogeneousMedium::sampleDistance with
 * EDistanceAlwaysValid) draws, for rays that are each their gather point's only medium edge (pdf_sel = 1; the rays of
 * gvpm_generate_rays are).  A ray draws only if edge_len > 4 * epsilon.  Ray r draws from
 * PCG32(seed ^ 0xD1B54A32D192ED03, r), the synth's stream; draw i takes u (stratified: i * (1/nb) + u * (1/nb)) to
 *   d = -log(1 - u * (1 - exp(-sigma_t[1] * max(edge_len - 2 epsilon, 0)))) / sigma_t[1],
 * skipped unless d < edge_len - epsilon and o + (d + epsilon) * dir != o; t = d + epsilon,
 * pdf_success = sum_c sigma_t[c] / (1 - exp(-sigma_t[c] (edge_len - epsilon))) * exp(-sigma_t[c] d) / 3,
 * transmittance[c] = exp(-sigma_t[c] d) (all zero when all are below 1e-20), radius = radius_per_ray_dev[r] (device
 * memory, n_rays floats) or, when that is NULL, `radius`.  Samples are stored ray by ray, draws in ascending order.
 * Arithmetic is strictly rounded fp32 in the synth's operation order with the tracers' polynomial log / exp, so the
 * samples are bit-reproducible (they differ from the synth's libm results in the last bits, DESIGN.md §6).  The context
 * is left as gvpm_upload_vpm_samples of the same arrays leaves it; *n_samples (may be NULL) = the number drawn.  The
 * gathers and gvpm_dump_neighbours_vpm refuse the drawn samples once another ray set has been committed.  Fails with
 * GVPM_ERR_INVALID without a committed ray set or a medium, for nb_camera_samples <= 0, epsilon not > 0, a scalar
 * radius that is not finite and > 0 (without a per-ray array), n_rays * nb_camera_samples > 0xfffffff0, or a per-ray
 * radius of a drawing ray that is negative or not finite. */
int gvpm_generate_vpm_samples(gvpm_ctx *ctx, int nb_camera_samples, int stratified, uint64_t seed, float epsilon,
                              float radius, const float *radius_per_ray_dev, size_t *n_samples);

/* ---- hand-off: computeGradient (gvpm.cpp:1205-1306) on the 27-float planes -------------
 * acc: device or host? -> host [h*w*27] APA-averaged accumulators in pixel order;
 * writes throughput, gx, gy [h*w*3] (interleaved RGB, row-major; poisson hand-off layout
 * gvpm.cpp:560-578).  use_abs as the reference's useAbs flag. */
int gvpm_compute_gradient(gvpm_ctx *ctx, const float *acc, int w, int h, int use_abs,
                          float *throughput, float *gx, float *gy);
/* Same gradients; the throughput plane is the reusePrimal estimate (GPMConfig::reusePrimal, gvpm.cpp:503-532): the
 * shifted flux the four neighbouring pixels send to a pixel plus its own four weighted fluxes, over 4.  inv_emitted =
 * 1 for the APA estimators (BRE, beams, planes), 1 / m_totalEmittedVolume for G-VPM (:527-531). */
int gvpm_compute_gradient_reuse_primal(gvpm_ctx *ctx, const float *acc, int w, int h, int use_abs, float inv_emitted,
                                       float *throughput, float *gx, float *gy);

/* ---- next step of the hand-off: screened-Poisson reconstruction (gvpm.cpp:610-690) -----------------------------
 * Replaces poisson::Solver (src/integrators/poisson_solver/Solver.cpp: importImagesMTS + setupBackend +
 * solveIndirect + exportImagesMTS) on the three planes gvpm_compute_gradient returns: iteratively reweighted least
 * squares around conjugate gradients on P' W^2 P, P = [alpha I; Dx; Dy].  gvpm_poisson_preset fills the parameters of
 * Solver::Params::setConfigPreset ("L1D", "L1Q", "L1L", "L2D", "L2Q"; the integrator uses L1D and L2D with
 * alpha = reconstructAlpha).  throughput, dx, dy, direct, reconstruction: host [h*w*3], interleaved RGB, row-major;
 * throughput and direct may be NULL (then alpha = 0, x starts at 0 / nothing is added: Solver.cpp:323,338-343,559-563).
 * The preconditioned branch (cg_precond, which no preset enables) returns GVPM_ERR_UNSUPPORTED. */
typedef struct gvpm_poisson_params {
  float alpha;            /* weight of the throughput image against the gradients */
  int32_t irls_iter_max;  /* 1 = plain L2 */
  float irls_reg_init, irls_reg_iter;
  int32_t cg_iter_max, cg_iter_check, cg_precond;
  float cg_tolerance;
} gvpm_poisson_params;
int gvpm_poisson_preset(const char *preset, gvpm_poisson_params *p);
int gvpm_poisson_solve(gvpm_ctx *ctx, int w, int h, const float *throughput, const float *dx, const float *dy,
                       const float *direct, const gvpm_poisson_params *params, float *reconstruction);
/* gvpm_compute_gradient + gvpm_poisson_solve in one call: the accumulators go up once, throughput / gx / gy stay on
 * the device between the two steps (each may be NULL when the caller does not want the plane back). */
int gvpm_reconstruct(gvpm_ctx *ctx, const float *acc, int w, int h, int use_abs, const float *direct,
                     const gvpm_poisson_params *params, float *throughput, float *gx, float *gy, float *reconstruction);
/* device time of the last gvpm_poisson_solve / gvpm_reconstruct, copies included (CUDA events, ms) */
float gvpm_last_poisson_ms(const gvpm_ctx *ctx);

/* ---- per-pixel accumulators on the device: the fold of every iteration of a progressive render -------------------
 * GatherPoint's volume accumulators (gvpm_struct.h:421-455; sppm: GatherPoint::fluxVol) kept in the context's device
 * memory across iterations, updated as GPMIntegrator (gvpm.cpp:1054-1069, G-VPM :1176-1181) and SPPMIntegrator
 * (sppm.cpp:866-871) update them, and handed to the gradient and the Poisson solve without a host round trip.  The
 * results are the host mirror's (VolumeGatherB200 / SPPMVolumeGatherB200 foldIteration) bit for bit, given the same
 * per-ray gather output.  Per iteration:
 *     gather (any of gvpm_gather_bre / _device / _host, gvpm_gather_sppm_bre, gvpm_gather_vpm / _device,
 *             gvpm_gather_beams / _device, gvpm_gather_planes / _device, gvpm_gather_sppm_beams);
 *     gvpm_accum_add;              (once per ray set: an iteration may come in several ray batches)
 *     gvpm_accum_fold(it, n_paths);
 * and after the last one gvpm_reconstruct_accum (or gvpm_accum_read for the image itself).
 *
 * gvpm_accum_reset: w x h pixels (w * h < 2^30) of `channels` floats - 27 for gvpm, 3 for sppm's fluxVol - zeroed,
 *   with one have_smoke byte per pixel and the emitted-path total (grow-only allocations, like every context buffer).
 *   apa = 1: the APA running mean (BRE, beams, planes, sppm); apa = 0: the plain sum of G-VPM, divided by the total
 *   number of emitted paths when read normalised.
 * gvpm_accum_add: the per-ray results the last gather left in the context's output, for the current ray set, added to
 *   their pixels (px, py of the rays): into the iteration's sum (apa = 1) or straight into the accumulators (apa = 0).
 *   Only the first `channels` floats of each ray's row are read.  Rays outside the film are skipped; every ray inside
 *   it sets its pixel's have_smoke byte.  The rays of one pixel are added in ray order, and batches in call order add
 *   up to the same bits as one batch holding their concatenation.  Rays of gvpm_generate_rays (one per pixel) are
 *   scattered directly; other ray sets are first sorted by pixel.  Fails with GVPM_ERR_INVALID when no gather has run
 *   on the current ray set (gvpm_ray_staging, gvpm_upload_rays and gvpm_generate_rays start a new one), when the last
 *   gather's output has already been added, when the last gather wrote to caller memory (gvpm_gather_bre_into), or when
 *   it wrote fewer floats per ray than there are channels (gvpm_gather_sppm_beams writes 3).  It first completes any
 *   asynchronous gather still in flight (gvpm_gather_bre_device: waits for it, and re-runs it when its pair list
 *   overflowed, as gvpm_sync does), so it never adds an incomplete result; this costs one wait per add while such a
 *   gather is queued.  The work itself is queued on the context's stream.
 * gvpm_accum_fold: the end of iteration `it` (1, 2, ...) whose light paths numbered n_paths.  apa = 1: for EVERY
 *   pixel, reached or not, acc = (acc * (float)(it - 1) + sum * (1.0f / (float)n_paths)) * (1.0f / (float)it), then
 *   the iteration's sum is cleared.  apa = 0: n_paths is added to the emitted total.  it >= 1, n_paths >= 1.
 * gvpm_accum_read: host copies [h*w*channels] floats, [h*w] bytes and the emitted total; each pointer may be NULL.
 *   normalized = 1 with apa = 0 multiplies by 1.0f / (float)total (the G-VPM image; nothing when total is 0).
 * gvpm_accum_device: the device arrays themselves, read-only (valid until the next gvpm_accum_reset).  A sharded
 *   render whose ranks own disjoint pixels (column bands) sums the ranks' arrays to the single-GPU result exactly.
 * gvpm_compute_gradient_accum / gvpm_reconstruct_accum: gvpm_compute_gradient (reuse_primal = 0) or
 *   gvpm_compute_gradient_reuse_primal (reuse_primal = 1, inv_emitted > 0), and gvpm_reconstruct, applied to the
 *   accumulators as they are stored (27 channels only).
 * Every call but gvpm_accum_reset fails with GVPM_ERR_INVALID before the first gvpm_accum_reset. */
int gvpm_accum_reset(gvpm_ctx *ctx, int w, int h, int channels, int apa);
int gvpm_accum_add(gvpm_ctx *ctx);
int gvpm_accum_fold(gvpm_ctx *ctx, int it, uint64_t n_paths);
int gvpm_accum_read(gvpm_ctx *ctx, int normalized, float *acc, uint8_t *have_smoke, uint64_t *total_emitted);
int gvpm_accum_device(gvpm_ctx *ctx, const float **acc, const uint8_t **have_smoke);
int gvpm_compute_gradient_accum(gvpm_ctx *ctx, int use_abs, int reuse_primal, float inv_emitted, float *throughput,
                                float *gx, float *gy);
int gvpm_reconstruct_accum(gvpm_ctx *ctx, int use_abs, const float *direct, const gvpm_poisson_params *params,
                           float *throughput, float *gx, float *gy, float *reconstruction);


/* ---- next rows (SURVEY.md 8 f-1, f-2): the two host stages on either side of the gather, on the device -------------
 * Scene class covered (the synthetic scenes of SURVEY.md 8d): an axis-aligned box filled with the homogeneous
 * medium set by gvpm_set_medium, diffuse walls with one albedo per face, the face z = lo[2] OPEN (index-matched
 * boundary towards the sensor: light paths leave through it, camera rays enter through it), up to 4 two-sided
 * diffuse rectangles parallel to the xz plane inside the box, and a rectangular diffuse area light on the plane
 * y = light_y pointing down (-y).  gvpm_box_scene_default() is the Cornell box of the bench / test workloads.
 * Triangle meshes inside the medium's box have entry points of their own (gvpm_mesh_scene below); glossy BSDFs and
 * other emitters stay with the host renderer and the upload entry points above. */
typedef struct gvpm_box_scene {
  float lo[3], hi[3];           /* the medium's box */
  float face_albedo[5][3];      /* x = lo, x = hi, y = lo, y = hi, z = hi (z = lo is open) */
  int32_t n_rects;              /* <= 4 */
  struct { float y, x0, x1, z0, z1, albedo[3]; } rect[4];
  float light_y, light_x0, light_x1, light_z0, light_z1, light_power;
} gvpm_box_scene;
int gvpm_box_scene_default(gvpm_box_scene *s);

/* f-2: camera-ray medium segments + their four offset segments (what gvpm_upload_rays takes) generated on the device
 * for a pinhole sensor at `pos` looking down +z: replaces, for this scene class, the camera sub-path tracing of
 * GatherPointMap::generate (gvpm/gvpm_gatherpoint.h:259-486), the offset paths of ShiftGatherPoint::generate
 * (gvpm/shift/shift_cameraPath.h:146-413; offsets at +-1 pixel, shift_utilities.h:255-261) and sensorMIS
 * (gvpm_struct.h:608-631, = 1 for a pinhole).  One jittered sample per pixel from the counter-based RNG
 * PCG32(seed, pixel index); rays are emitted block by block (block x block pixels like m_gatherBlocks,
 * gvpm.cpp:271-290; block < 0: Z-order inside a block), rows [y0, y1) of the image.  tan_half_fov_x is the half width
 * of the image plane at distance 1.  The rays are committed (as after gvpm_upload_rays); n_rays = w * (y1 - y0). */
typedef struct gvpm_pinhole_camera {
  float pos[3];
  float tan_half_fov_x;
  int32_t film_w, film_h;
  int32_t inside_medium;        /* 1: the sensor sits in the medium (segments start at pos, edge 1); 0: in front of the
                                   open face (segments start on it, edge 2) */
} gvpm_pinhole_camera;
int gvpm_generate_rays(gvpm_ctx *ctx, const gvpm_box_scene *scene, const gvpm_pinhole_camera *cam, uint64_t seed,
                       int block, int y0, int y1, float epsilon);

/* f-1: the iteration's volume photons traced on the device: replaces, for this scene class, the light-path random walk
 * of GradientPhotonProcess (gvpm/gvpm_proc.cpp:125-210,336-350) and GPhotonMap::tryAppend (gvpm_accel.h:119-199).
 * Light path k draws from PCG32(seed, k); free paths are exponential, scattering follows the phase function of
 * gvpm_set_medium, walls and rectangles reflect diffusely, russian roulette from depth rr_depth with
 * q = min(max throughput, 0.95); every medium vertex with index >= max(2, min_depth + 1) is stored until n photons
 * exist (paths are taken in index order, so the set does not depend on the launch geometry).  log / exp / sin / cos
 * are evaluated by fixed polynomial routines in strictly rounded fp32 (no libm), so the records are bit-reproducible
 * and an independent CPU restatement produces the same bits.  The photons land in the selected staging buffer exactly
 * as gvpm_upload_photons leaves them (call gvpm_build_points / _for_rays next).  n_paths: light paths traced up to and
 * including the one that completed the set (nbPathVolume, the gather's normalisation). */
int gvpm_trace_photons(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth, int rr_depth,
                       int min_depth, uint64_t *n_paths);
/* Same photons, written straight into the 128-byte records the gather reads (no staging buffer, no packing pass in the
 * build): the layout a renderer that lives on the device would produce.  gvpm_build_points / gvpm_build_points_for_rays
 * and the BRE / VPM gathers work on them as on uploaded photons, with identical results; the staging-based entry points
 * (gvpm_photon_staging, peer exchange) do not see them. */
int gvpm_trace_photons_direct(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth,
                              int rr_depth, int min_depth, uint64_t *n_paths);
/* f-1, beams: the iteration's photon beams traced on the device by the same light-path walk as gvpm_trace_photons
 * (same random numbers, arithmetic and termination), storing instead every edge vertex(i) -> vertex(i+1) that does not
 * escape, for i >= max(1, min_depth) - LTBeamMap::tryAppendLT (gvpm/gvpm_beams.h:54-84) with the fields of
 * gvpm_beam_soa; path_id counts the paths that store at least one beam.  Paths are taken in index order until n beams
 * exist.  The context is left exactly as gvpm_upload_beams of the same arrays leaves it (records packed, sub-beam
 * size = the in-order fp32 mean length / 10 summed on the device, gvpm_beam_subbeam_count known): call
 * gvpm_build_beams next.  n_paths = nbPathBeams (light paths up to and including the one that completed the set).
 * max_depth <= 255; n <= 0x0ffffff0. */
int gvpm_trace_beams(gvpm_ctx *ctx, const gvpm_box_scene *scene, size_t n, uint64_t seed, int max_depth, int rr_depth,
                     int min_depth, uint64_t *n_paths);
/* G-Planes 0D inputs made on the device: one photon plane per beam of the current beam set (uploaded or traced),
 * as LTPhotonPlane::transformBeam (gvpm/gvpm_plane.h:53-73) extends it - origin, w0, length0 = the beam's
 * setEndPoint, length1 = a free-flight distance + Epsilon, w1 = a phase-function direction (isotropic or HG in the
 * coherent frame of the beam; directions parallel to the beam are drawn again), flux and edge_id = depth copied.
 * Beam i draws from PCG32(seed ^ 0xA0761D6478BD642F, i) instead of the integrator's single sequential sampler
 * (DESIGN.md §6); log / sin / cos are the polynomial routines of the tracers, so the planes are bit-reproducible.
 * The context is left as gvpm_upload_planes of the same arrays leaves it: call gvpm_build_planes next.  Fails when
 * there is no beam set, no medium, or the medium's sampling_weight is not 1. */
int gvpm_planes_from_beams(gvpm_ctx *ctx, uint64_t seed);

/* ---- rows f-1 / f-2 on triangle-mesh scenes ---------------------------------------------------------------------------
 * Scene class: the homogeneous medium of gvpm_set_medium fills the axis-aligned box lo / hi, whose boundary is
 * index-matched everywhere (a ray that reaches it before any triangle leaves the scene: the light path ends there, a
 * camera segment ends there).  Inside the box: n_tri triangles (tri = 9 floats each, p0 p1 p2), each with one diffuse
 * albedo, two-sided; the shading normal is normalize(cross(p1 - p0, p2 - p0)) turned to face the incoming ray.  Every
 * vertex must lie in the box, up to 1e-6 of the box extent on each axis.  The triangles flagged emissive (emissive[i] !=
 * 0) are also one diffuse area light of total power light_power, emitting on the side of their winding normal only;
 * they are surfaces too, with their own albedo (0 absorbs).
 * Emitter sampling (a restatement, not Mitsuba's shape-sampling sequence): the areas of the emissive triangles are
 * summed in fp32 in triangle index order on the host; a light path draws u0 and picks the first emissive triangle whose
 * running sum exceeds u0 * total (the last emissive triangle of non-zero area when none does), then u1, u2 for the
 * point p0 + (e1 * (1 - sqrt(u1)) + e2 * (u2 * sqrt(u1))), then the cosine direction about the winding normal as the
 * box tracer draws it.  u0 is the only draw the box walk does not make; every later draw is the box walk's.
 * Intersection: the nearest triangle with a strictly rounded Moller-Trumbore parameter t > 1e-6 (Triangle::rayIntersect,
 * include/mitsuba/core/triangle.h:109-145), ties to the smaller triangle index, skipping the triangle the ray starts
 * on, searched up to the exit of the box grown by 2e-6 of its extent (strictly rounded slab tests): a triangle wins over
 * the box exit when t <= t_exit, and so does a wall on a face of the box that rounding puts just beyond it.  The walk
 * goes down a BVH built on the device once per scene; its answer is that of the brute-force loop over all triangles.
 * This scene does not change the occluders: pass the same triangles to gvpm_set_occluders for the shadow rays. */
typedef struct gvpm_mesh_scene {
  float lo[3], hi[3];           /* the medium's box */
  size_t n_tri;                 /* <= GVPM_MAX_OCCLUDERS (2^24) */
  const float *tri;             /* [n_tri*9] */
  const float *albedo;          /* [n_tri*3] */
  const uint8_t *emissive;      /* [n_tri] */
  float light_power;
} gvpm_mesh_scene;
/* Copies the arrays to the device and builds the scene's BVH there; the mesh entries below then use it until the next
 * call.  Fails with GVPM_ERR_INVALID (and the reason in gvpm_last_error) on a null array, an empty or non-finite box,
 * more than 2^24 triangles, a non-finite coordinate, albedo or power, a vertex outside the box, or no emissive
 * triangle of positive area; the context then has no mesh scene. */
int gvpm_set_trace_mesh(gvpm_ctx *ctx, const gvpm_mesh_scene *scene);
/* gvpm_trace_photons / gvpm_trace_photons_direct / gvpm_trace_beams on the mesh scene: the same walk, random numbers
 * (plus the emitter pick), records, batching and limits, and the context is left as they leave it.  Fail with
 * GVPM_ERR_INVALID when there is no mesh scene or no medium. */
int gvpm_trace_photons_mesh(gvpm_ctx *ctx, size_t n, uint64_t seed, int max_depth, int rr_depth, int min_depth,
                            uint64_t *n_paths);
int gvpm_trace_photons_direct_mesh(gvpm_ctx *ctx, size_t n, uint64_t seed, int max_depth, int rr_depth, int min_depth,
                                   uint64_t *n_paths);
int gvpm_trace_beams_mesh(gvpm_ctx *ctx, size_t n, uint64_t seed, int max_depth, int rr_depth, int min_depth,
                          uint64_t *n_paths);
/* A pinhole with a look-at frame: f = normalize(forward), r = normalize(cross(up, f)), u = cross(f, r); the ray of
 * film point (sx, sy) has direction normalize((r * x + u * y) + f) with x = ((sx / film_w - 0.5) * 2) * tan_half_fov_x,
 * y = ((sy / film_h - 0.5) * 2) * tan_half_fov_x * film_h / film_w (forward = +z, up = +y is gvpm_pinhole_camera's
 * frame).  A camera strictly inside the box starts its segments at pos (edge 1); one outside starts them where the ray
 * enters the box (edge 2): the entry face is the slab test's, the entry point is snapped onto that face's plane and
 * must lie inside the face, and no triangle may be hit before the face moved inwards by that 2e-6 margin. */
typedef struct gvpm_lookat_camera {
  float pos[3], forward[3], up[3];
  float tan_half_fov_x;
  int32_t film_w, film_h;
} gvpm_lookat_camera;
/* gvpm_generate_rays on the mesh scene: the same pixels, PCG32 draws, segments (ending at the nearest triangle or at
 * the box exit), offsets, edge_id, eye_contrib and off_sensor = 1.  Fails with GVPM_ERR_INVALID without a mesh scene,
 * on a bad block, film or row range, or a camera whose forward is zero, parallel to up, or whose field of view is not
 * positive and finite. */
int gvpm_generate_rays_mesh(gvpm_ctx *ctx, const gvpm_lookat_camera *cam, uint64_t seed, int block, int y0, int y1,
                            float epsilon);

/* parity aid: copy `bytes` bytes at `dev` (a pointer handed out by this library, e.g. gvpm_photon_staging /
 * gvpm_ray_staging) to host memory, after the work queued on the context's stream */
int gvpm_read_device(gvpm_ctx *ctx, const void *dev, void *host, size_t bytes);
/* measurement aid (the roofline's L2 denominator, BASELINE.json "% of HBM/L2 peak"): `reps` passes of 128-bit loads
 * over a `bytes`-byte device buffer by a machine-filling grid, timed with CUDA events on the context's stream;
 * gb_per_s = bytes * reps / time.  A buffer well below the 126 MB L2 gives the L2 read bandwidth, one far above it the
 * HBM read bandwidth. */
int gvpm_measure_read_bandwidth(gvpm_ctx *ctx, size_t bytes, int reps, double *gb_per_s);
/* parity aid: the selected photon staging buffer (which = 0), the ray staging buffer (1), the beam staging buffer (2),
 * the plane staging buffer (3) or the G-VPM sample staging buffer (4) as they are, without the side effects of gvpm_photon_staging / gvpm_ray_staging
 * (which invalidate the build / the committed rays).  Each holds its SoA's arrays back to back, every array starting
 * on a 256-byte boundary; count = the number of elements of the current set. */
int gvpm_staging_peek(gvpm_ctx *ctx, int which, void **dev, size_t *count);

/* ---- timing of the last build / gather on the context's stream (CUDA events, ms) ----- */
int gvpm_last_timings(gvpm_ctx *ctx, float *build_ms, float *gather_ms);
/* split of the last gather: traversal kernel, shading kernel (of the last ray range), and the number of
 * contributing (ray, photon) pairs the traversal handed to the shading kernel */
int gvpm_last_gather_detail(gvpm_ctx *ctx, float *traverse_ms, float *shade_ms, uint64_t *pairs);
/* number of kernel launches issued by this context since creation */
uint64_t gvpm_launch_count(const gvpm_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* GVPM_B200_H */
