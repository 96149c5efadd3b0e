// Checks gvpm::quotient_negative(a, b) (gvpm_device.cuh) against the sign of the correctly rounded quotient a / b, over
// the edge values of the side tests (+-0, +-inf, NaN, subnormals, |b| near 1) crossed with each other, plus random pairs.
// `host`: the host's IEEE division; `device`: __fdiv_rn in a kernel.  Prints the mismatches and their count.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../gvpm_b200/csrc/gvpm_device.cuh"

static float bits(uint32_t u) { float f; std::memcpy(&f, &u, 4); return f; }

__global__ void k_check(const float *a, const float *b, int n, unsigned char *want, unsigned char *got) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  want[i] = __fdiv_rn(a[i], b[i]) < 0.f;
  got[i] = gvpm::quotient_negative(a[i], b[i]);
}

int main(int argc, char **argv) {
  const bool device = argc > 1 && std::strcmp(argv[1], "device") == 0;
  std::vector<float> as = {0.f, 1.f, 0.5f, 1e-30f, 3.4e38f, bits(1u), bits(0x007fffffu), bits(0x00800000u), INFINITY,
                           NAN, 0.7071068f};
  std::vector<float> bs = {0.f, 1.f, bits(0x3f800001u), bits(0x3f800003u), bits(0x3fffffffu), 0.5f, 1e-30f, bits(1u),
                           bits(0x007fffffu), INFINITY, NAN, 0.3f};
  const size_t na = as.size(), nb = bs.size();
  for (size_t i = 0; i < na; ++i) as.push_back(-as[i]);
  for (size_t i = 0; i < nb; ++i) bs.push_back(-bs[i]);
  std::vector<float> A, B;
  for (float a : as)
    for (float b : bs) { A.push_back(a); B.push_back(b); }
  uint32_t s = 12345u;
  auto next = [&s]() { s = s * 1664525u + 1013904223u; return s; };
  for (int i = 0; i < 200000; ++i) {
    A.push_back(bits(next()));                                                       // any bit pattern
    const float b = bits((next() & 0x807fffffu) | ((next() % 128u) << 23));          // |b| < 2 (exponents 0 .. 127)
    B.push_back(b);
  }
  const int n = (int)A.size();
  std::vector<unsigned char> want(n), got(n);
  if (device) {
    float *dA, *dB;
    unsigned char *dW, *dG;
    cudaMalloc(&dA, n * 4); cudaMalloc(&dB, n * 4); cudaMalloc(&dW, n); cudaMalloc(&dG, n);
    cudaMemcpy(dA, A.data(), n * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dB, B.data(), n * 4, cudaMemcpyHostToDevice);
    k_check<<<(n + 255) / 256, 256>>>(dA, dB, n, dW, dG);
    cudaMemcpy(want.data(), dW, n, cudaMemcpyDeviceToHost);
    cudaMemcpy(got.data(), dG, n, cudaMemcpyDeviceToHost);
    const cudaError_t e = cudaGetLastError();
    cudaFree(dA); cudaFree(dB); cudaFree(dW); cudaFree(dG);
    if (e != cudaSuccess) { std::printf("cuda error: %s\n", cudaGetErrorString(e)); return 2; }
  } else {
    for (int i = 0; i < n; ++i) {
      volatile float q = A[i] / B[i];
      want[i] = q < 0.f;
      got[i] = gvpm::quotient_negative(A[i], B[i]);
    }
  }
  int bad = 0;
  for (int i = 0; i < n; ++i)
    if (want[i] != got[i] && bad++ < 20) std::printf("mismatch a=%a b=%a quotient<0: %d\n", A[i], B[i], want[i]);
  std::printf("%d pairs, %d mismatches\n", n, bad);
  return bad ? 1 : 0;
}
