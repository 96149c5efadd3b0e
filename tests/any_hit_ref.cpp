// any_hit_ref.cpp — TEST INFRASTRUCTURE.  The oracle's Occluders<float>::anyHit (oracle/gvpm_oracle.hpp, unchanged: the
// restatement of Triangle::rayIntersect over a flat list) for each of m rays over a whole triangle list, split over
// `threads` std::threads: the reference answer the device's list and BVH any-hit paths are compared with
// (tests/test_gpu_occluder_bvh.py).  Compiled with the oracle's flags (no FMA contraction).
#include <algorithm>
#include <thread>
#include <vector>

#include "../oracle/gvpm_oracle.hpp"

using namespace gvpm_oracle;

extern "C" {

void any_hit_ref(const float *tri, size_t n_tri, const float *ro, const float *rd, const float *mint, const float *maxt,
                 size_t m, int threads, uint8_t *hit) {
  Occluders<float> occ;
  occ.set(tri, n_tri);
  if (threads < 1) threads = 1;
  const size_t chunk = (m + (size_t)threads - 1) / (size_t)threads;
  auto worker = [&](size_t b, size_t e) {
    for (size_t i = b; i < e; ++i)
      hit[i] = occ.anyHit(V3<float>(ro + 3 * i), V3<float>(rd + 3 * i), mint[i], maxt[i]) ? 1 : 0;
  };
  std::vector<std::thread> pool;
  for (size_t b = 0; b < m; b += chunk) pool.emplace_back(worker, b, std::min(m, b + chunk));
  for (auto &t : pool) t.join();
}

}  // extern "C"
