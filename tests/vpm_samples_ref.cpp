// vpm_samples_ref.cpp — TEST INFRASTRUCTURE.  CPU restatement of gvpm_generate_vpm_samples (include/gvpm_b200.h), the
// checker the device-drawn G-VPM camera distance samples are compared with BIT FOR BIT (tests/test_gpu_vpm_samples.py).
// It reuses, unchanged, the PCG32 stream and the polynomial log / exp of the photon tracer's restatement
// (oracle/gvpm_oracle_trace.cpp, included below), and follows gvpm_synth_vpm_samples' operation order;
// tests/test_oracle_vpm_samples.py pins it to that host generator.  Compiled with -ffp-contract=off: every operation is
// rounded on its own.
#include "../oracle/gvpm_oracle_trace.cpp"

extern "C" {

// the G-VPM camera distance samples of gvpm_generate_vpm_samples: gvpm_synth_vpm_samples' draws in its operation order,
// with the polynomial log / exp and radius = radius_per_ray[r] (NULL: `radius`); `out` holds n_rays * nb entries.
// Returns the number of samples stored.
long long vpm_samples_ref(const gvpm_ray_soa *rays, size_t n_rays, int nb, int stratified, uint64_t seed,
                                const gvpm_medium *med, float epsilon, float radius, const float *radius_per_ray,
                                gvpm_vpm_sample_soa *out) {
  if (!rays || !med || !out || nb <= 0) return -1;
  const float sigT[3] = {med->sigma_s[0] + med->sigma_a[0], med->sigma_s[1] + med->sigma_a[1],
                         med->sigma_s[2] + med->sigma_a[2]};
  const float density = sigT[1], normalization = 1.f / (float)nb;
  size_t n = 0;
  for (size_t r = 0; r < n_rays; ++r) {
    const float len = rays->edge_len[r];
    if (!(len > 4.f * epsilon)) continue;
    const float mint = epsilon, maxt = len;
    const float maxDist = std::max((maxt - mint) - epsilon, 0.0f);
    const float norm = 1.f - pmExp(-density * maxDist);
    const float distSurf = maxt - mint;
    float coef[3];
    for (int c = 0; c < 3; ++c) coef[c] = sigT[c] / (1.f - pmExp(-sigT[c] * distSurf));
    const float *o = rays->o + 3 * r, *d = rays->d + 3 * r;
    Rng rng(seed ^ 0xD1B54A32D192ED03ULL, r);
    for (int i = 0; i < nb; ++i) {
      float rand = rng.uniform();
      if (stratified) rand = (float)i * normalization + rand * normalization;
      const float dist = -pmLog(1.f - rand * norm) / density;
      if (!(dist < distSurf)) continue;
      const float t = dist + mint;
      if (o[0] + d[0] * t == o[0] && o[1] + d[1] * t == o[1] && o[2] + d[2] * t == o[2]) continue;
      float tr[3], pdf = 0.f;
      for (int c = 0; c < 3; ++c) tr[c] = pmExp(-sigT[c] * dist);
      for (int c = 0; c < 3; ++c) pdf = pdf + coef[c] * tr[c];
      pdf = pdf / 3.f;
      if (std::max(tr[0], std::max(tr[1], tr[2])) < 1e-20f) tr[0] = tr[1] = tr[2] = 0.f;
      const_cast<uint32_t *>(out->ray)[n] = (uint32_t)r;
      const_cast<float *>(out->t)[n] = t;
      put(out->transmittance, n, V{tr[0], tr[1], tr[2]});
      const_cast<float *>(out->pdf_success)[n] = pdf;
      const_cast<float *>(out->pdf_sel)[n] = 1.0f;
      const_cast<float *>(out->radius)[n] = radius_per_ray ? radius_per_ray[r] : radius;
      ++n;
    }
  }
  return (long long)n;
}

}  // extern "C"
