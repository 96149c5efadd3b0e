// pack_prims.cu — device-side flattening of the raw beam / plane / distance-sample SoA arrays into the records the
// gathers read.  Round 1 did this in host loops inside gvpm_upload_*, which is fine for test sizes and hopeless at
// BASELINE sizes (cfg3: 500 k beams -> 5 M sub-beams, cfg2: 10.5 M samples per iteration).  The arithmetic that
// decides anything downstream (beam direction / length, sub-beam cuts) is the reference's, in its operation order,
// with explicitly rounded intrinsics (no FMA contraction), so the records are bit-identical to the host loops
// they replace:
//   PhotonBeam::setEndPoint                         photonmapper/beams_struct.h:73-81
//   SubBeamBVH constructor (sub-beam cuts)          photonmapper/beams_accel.h:98-124
//   PhotonPlane edges / getCenter                   photonmapper/plane_struct.h:45-74,107-108
#include "gvpm_device.cuh"
#include "warp_ops.cuh"

namespace gvpm {

// beam record (8 float4, DESIGN.md §3) + its length in a separate plane for the sub-beam split
__global__ void __launch_bounds__(256) k_pack_beams(const BeamStaging S, uint32_t n, float4 *__restrict__ rec,
                                                     float *__restrict__ len_out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t i3 = 3 * (size_t)i;
  const float o0 = S.origin[i3], o1 = S.origin[i3 + 1], o2 = S.origin[i3 + 2];
  const float e0 = S.end[i3], e1 = S.end[i3 + 1], e2 = S.end[i3 + 2];
  // dir = p2 - p1; length = |dir|; dir /= length (multiplication by the reciprocal, vector.h:535-542)
  float d0 = __fsub_rn(e0, o0), d1 = __fsub_rn(e1, o1), d2 = __fsub_rn(e2, o2);
  const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2)));
  const float rcp = __fdiv_rn(1.0f, len);
  d0 = __fmul_rn(d0, rcp); d1 = __fmul_rn(d1, rcp); d2 = __fmul_rn(d2, rcp);
  const uint32_t meta = pack_meta(S.parent_type[i], S.depth[i], S.path_id[i]) | ((S.end_on_surface[i] ? 1u : 0u) << 11);
  float4 *r = rec + (size_t)i * 8;
  r[0] = make_float4(o0, o1, o2, len);
  r[1] = make_float4(d0, d1, d2, __uint_as_float(meta));
  r[2] = make_float4(S.flux[i3], S.flux[i3 + 1], S.flux[i3 + 2], S.parent_pdf[i]);
  r[3] = make_float4(S.prefix_flux[i3], S.prefix_flux[i3 + 1], S.prefix_flux[i3 + 2], S.rr_weight[i]);
  r[4] = make_float4(S.parent_n[i3], S.parent_n[i3 + 1], S.parent_n[i3 + 2], e0);
  r[5] = make_float4(S.parent_albedo[i3], S.parent_albedo[i3 + 1], S.parent_albedo[i3 + 2], e1);
  r[6] = make_float4(S.pred_pos[i3], S.pred_pos[i3 + 1], S.pred_pos[i3 + 2], e2);
  r[7] = make_float4(S.end_n[i3], S.end_n[i3 + 1], S.end_n[i3 + 2], 0.f);
  len_out[i] = len;
}

// `Float avgSize = 0; for (b : beams) avgSize += b.getLength();` is a SEQUENTIAL fp32 sum (beams_accel.h:98-102): its
// rounding depends on the order, and the sub-beam size derived from it decides how every beam is cut.  One warp
// streams the lengths through shared memory and lane 0 adds them in index order (a ~4-cycle dependent chain per beam).
// gvpm_upload_beams has the host do this sum while the DMA runs; this kernel serves the beams gvpm_trace_beams makes
// on the device (capi_prims.cu commit_beams).  out[0] = subbeamSize = avg / 10.
__global__ void __launch_bounds__(32) k_beam_subsize_seq(const float *__restrict__ len, uint32_t n, float *__restrict__ out) {
  __shared__ float buf[2][32 * 8];
  const int lane = threadIdx.x;
  float sum = 0.f;
  for (uint32_t base = 0; base < n; base += 256) {
    float *b = buf[(base >> 8) & 1];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const uint32_t i = base + 32u * k + lane;
      b[32 * k + lane] = i < n ? __ldg(len + i) : 0.f;
    }
    __syncwarp();
    if (lane == 0) {
      const uint32_t m = min(256u, n - base);
      for (uint32_t k = 0; k < m; ++k) sum = __fadd_rn(sum, b[k]);
    }
    __syncwarp();
  }
  if (lane == 0) {
    float avg = n ? __fdiv_rn(sum, (float)n) : 0.f;
    out[0] = __fdiv_rn(avg, 10.f);
  }
}

__device__ __forceinline__ int beam_nsub(float len, float subbeamSize) {
  int nSub = subbeamSize > 0.f ? (int)ceilf(__fdiv_rn(len, subbeamSize)) : 1;
  return nSub < 1 ? 1 : nSub;
}

// per-beam sub-beam count -> exclusive offsets: block totals (k_sub_count), one-block scan of them (k_scan_exclusive), and
// the emit pass re-scans inside each block
__global__ void __launch_bounds__(256) k_sub_count(const float *__restrict__ len, uint32_t n, const float *__restrict__ subsize,
                                                    uint32_t *__restrict__ block_tot) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t t = block_total<8>(i < n ? (uint32_t)beam_nsub(len[i], subsize[0]) : 0u);
  if (threadIdx.x == 0) block_tot[blockIdx.x] = t;
}
// sub-beam records in beam order: pos = midpoint (Hilbert key input), raw = (t1, t2, beam index, flags)
//   flags: bit 0 first, bit 1 last sub-beam of its beam, bits 2.. ordinal (the naive sppm technique's RNG dimension)
__global__ void __launch_bounds__(256) k_sub_emit(const float4 *__restrict__ rec, const float *__restrict__ len, uint32_t n,
                                                   const float *__restrict__ subsize, const uint32_t *__restrict__ block_off,
                                                   uint32_t cap, float *__restrict__ sub_pos, float4 *__restrict__ sub_raw) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const float L = i < n ? len[i] : 0.f;
  const int nSub = i < n ? beam_nsub(L, subsize[0]) : 0;
  const uint32_t off = block_off[blockIdx.x] + block_exclusive<8>((uint32_t)nSub);
  if (i >= n) return;
  const float4 b0 = rec[(size_t)i * 8], b1 = rec[(size_t)i * 8 + 1];
  const float lengthSub = __fdiv_rn(L, (float)nSub);
  for (int k = 0; k < nSub; ++k) {
    const uint32_t s = off + (uint32_t)k;
    if (s >= cap) break;
    const float t1 = __fmul_rn(lengthSub, (float)k), t2 = __fmul_rn(lengthSub, (float)(k + 1)),
                tm = __fmul_rn(lengthSub, __fadd_rn((float)k, 0.5f));
    sub_pos[3 * (size_t)s] = __fadd_rn(b0.x, __fmul_rn(b1.x, tm));
    sub_pos[3 * (size_t)s + 1] = __fadd_rn(b0.y, __fmul_rn(b1.y, tm));
    sub_pos[3 * (size_t)s + 2] = __fadd_rn(b0.z, __fmul_rn(b1.z, tm));
    const uint32_t fl = (k == 0 ? 1u : 0u) | (k == nSub - 1 ? 2u : 0u) | ((uint32_t)k << 2);
    sub_raw[s] = make_float4(t1, t2, __uint_as_float(i), __uint_as_float(fl));
  }
}

// plane record (6 float4) + centre; flag[0] |= 1 when an edge length is zero or not finite (PhotonPlane ctor asserts)
__global__ void __launch_bounds__(256) k_pack_planes(const PlaneStaging S, uint32_t n, float4 *__restrict__ rec,
                                                      float *__restrict__ centre, uint32_t *__restrict__ flag) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t i3 = 3 * (size_t)i;
  const float l0 = S.length0[i], l1 = S.length1[i];
  if (!(l0 != 0.f && isfinite(l0) && l1 != 0.f && isfinite(l1))) atomicOr(flag, 1u);
  const float o[3] = {S.origin[i3], S.origin[i3 + 1], S.origin[i3 + 2]};
  const float w0[3] = {S.w0[i3], S.w0[i3 + 1], S.w0[i3 + 2]}, w1[3] = {S.w1[i3], S.w1[i3 + 1], S.w1[i3 + 2]};
  // e0 = _w0 * _length0, e1 = _w1 * _length1 exactly as intersectPlane0D forms them (plane_struct.h:107-108)
  float e0[3], e1[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) { e0[a] = __fmul_rn(w0[a], l0); e1[a] = __fmul_rn(w1[a], l1); }
  float4 *r = rec + (size_t)i * GVPM_PLANE_PLANES;
  r[0] = make_float4(o[0], o[1], o[2], l0);
  r[1] = make_float4(e0[0], e0[1], e0[2], l1);
  r[2] = make_float4(e1[0], e1[1], e1[2], __uint_as_float((uint32_t)S.edge_id[i]));
  r[3] = make_float4(S.flux[i3], S.flux[i3 + 1], S.flux[i3 + 2], 0.f);
  r[4] = make_float4(w0[0], w0[1], w0[2], 0.f);
  r[5] = make_float4(w1[0], w1[1], w1[2], 0.f);
#pragma unroll
  for (int a = 0; a < 3; ++a)  // getCenter: ori + 0.5 e0 + 0.5 e1
    centre[i3 + a] = __fadd_rn(__fadd_rn(o[a], __fmul_rn(0.5f, e0[a])), __fmul_rn(0.5f, e1[a]));
}

// distance samples: 2 float4 per sample of the staging buffer holding n samples (n_dev: a count known on the device
// only, n is then the grid's bound); stats[0] = max radius (float bits; radii are positive), stats[1] |= 1 when a sample
// refers to a ray that is not uploaded (the index is clamped so that the gather stays in bounds; the error is reported
// by the caller), |= 2 when a radius is negative or not finite
__global__ void __launch_bounds__(256) k_pack_samples(const void *staging, uint32_t n, const uint32_t *n_dev,
                                                       uint32_t n_rays, float4 *__restrict__ packed,
                                                       uint32_t *__restrict__ stats) {
  if (n_dev) n = *n_dev;
  const SampleStaging S = sample_staging_at(staging, n);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  float rad = 0.f;
  bool bad = false, badRad = false;
  if (i < n) {
    uint32_t rb = S.ray[i];
    if (rb >= n_rays) { bad = true; rb = n_rays ? n_rays - 1 : 0u; }
    rad = S.radius[i];
    badRad = !(rad >= 0.f && rad < INFINITY);
    packed[2 * (size_t)i] = make_float4(S.t[i], S.pdf_success[i], S.pdf_sel[i], rad);
    packed[2 * (size_t)i + 1] = make_float4(S.transmittance[3 * (size_t)i], S.transmittance[3 * (size_t)i + 1],
                                            S.transmittance[3 * (size_t)i + 2], __uint_as_float(rb));
  }
  rad = fmaxf(rad, 0.f);
  rad = warp_max(rad);
  const uint32_t anyBad = __ballot_sync(0xffffffffu, bad), anyBadRad = __ballot_sync(0xffffffffu, badRad);
  if ((threadIdx.x & 31) == 0) {
    atomicMax(stats, __float_as_uint(rad));
    if (anyBad || anyBadRad) atomicOr(stats + 1, (anyBad ? 1u : 0u) | (anyBadRad ? 2u : 0u));
  }
}

// ---- measurement aid: read bandwidth of a buffer that fits in L2 (the roofline's L2 denominator) --------------------------
// every CTA streams the whole buffer `reps` times with 128-bit loads, 4 in flight per thread; the xor of everything read
// goes to `sink` so that nothing is optimised away
__global__ void __launch_bounds__(256) k_l2_read(const uint4 *__restrict__ p, uint32_t n16, int reps, unsigned *__restrict__ sink) {
  uint4 acc = make_uint4(0u, 0u, 0u, 0u);
  const uint32_t stride = gridDim.x * blockDim.x;
  for (int r = 0; r < reps; ++r) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n16; i += 4 * stride) {
      const uint4 a = __ldcg(p + i), b = __ldcg(p + i + stride), c = __ldcg(p + i + 2 * stride), d = __ldcg(p + i + 3 * stride);
      acc.x ^= a.x ^ b.x ^ c.x ^ d.x; acc.y ^= a.y ^ b.y ^ c.y ^ d.y;
      acc.z ^= a.z ^ b.z ^ c.z ^ d.z; acc.w ^= a.w ^ b.w ^ c.w ^ d.w;
    }
    for (; i < n16; i += stride) { const uint4 a = __ldcg(p + i); acc.x ^= a.x; acc.y ^= a.y; acc.z ^= a.z; acc.w ^= a.w; }
  }
  if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x9e3779b9u) atomicAdd(sink, 1u);
}
void launch_l2_read(const void *p, size_t bytes, int reps, unsigned *sink, int sm_count, cudaStream_t st) {
  k_l2_read<<<sm_count * 8, 256, 0, st>>>((const uint4 *)p, (uint32_t)(bytes / 16), reps, sink);
}

// ---- launchers ------------------------------------------------------------------------------------------------------
void launch_pack_beams(const BeamStaging &S, uint32_t n, float4 *rec, float *len, cudaStream_t st) {
  if (n) k_pack_beams<<<(n + 255) / 256, 256, 0, st>>>(S, n, rec, len);
}
void launch_beam_subsize_seq(const float *len, uint32_t n, float *subsize, cudaStream_t st) {
  k_beam_subsize_seq<<<1, 32, 0, st>>>(len, n, subsize);
}
// block_tot: [(n + 255) / 256] words; total: 1 word
void launch_sub_count(const float *len, uint32_t n, const float *subsize, uint32_t *block_tot, uint32_t *total, cudaStream_t st) {
  const uint32_t nb = (n + 255) / 256;
  if (n) k_sub_count<<<nb, 256, 0, st>>>(len, n, subsize, block_tot);
  k_scan_exclusive<uint32_t, 8><<<1, 1024, 0, st>>>(block_tot, n ? nb : 0u, total, 0);   // 8 per thread: tens of thousands
}
void launch_sub_emit(const float4 *rec, const float *len, uint32_t n, const float *subsize, const uint32_t *block_off,
                     uint32_t cap, float *sub_pos, float4 *sub_raw, cudaStream_t st) {
  if (n) k_sub_emit<<<(n + 255) / 256, 256, 0, st>>>(rec, len, n, subsize, block_off, cap, sub_pos, sub_raw);
}
void launch_pack_planes(const PlaneStaging &S, uint32_t n, float4 *rec, float *centre, uint32_t *flag, cudaStream_t st) {
  if (n) k_pack_planes<<<(n + 255) / 256, 256, 0, st>>>(S, n, rec, centre, flag);
}
void launch_pack_samples(const void *staging, uint32_t n, const uint32_t *n_dev, uint32_t n_rays, float4 *packed,
                         uint32_t *stats, cudaStream_t st) {
  if (n) k_pack_samples<<<(n + 255) / 256, 256, 0, st>>>(staging, n, n_dev, n_rays, packed, stats);
}

}  // namespace gvpm
