// Device functions shared by the geometry translation units (metric_inputs.cu, associate.cu), defined once so that every
// kernel applies the same candidate rule and draws from the same generator.
#pragma once
#include <cstdint>

namespace mpl {

// The view takes part iff conf > min_conf and the pixel lies strictly inside the w x h image (build_inputs_kernel's tests).
__device__ __forceinline__ bool tri_candidate(float conf, double u, double w, float min_conf, const double (&wh)[2]) {
  return conf > min_conf && 0.0 < u && u < wh[0] - 1.0 && 0.0 < w && w < wh[1] - 1.0;
}

// numpy's Philox4x64-10 block function, bit for bit (openmpl_b200/synth.py draws the same uniforms on the host).
__device__ __forceinline__ void philox4x64_10(uint64_t n, uint64_t key0, uint64_t key1, uint64_t (&out)[4]) {
  uint64_t c0 = n, c1 = 0, c2 = 0, c3 = 0, k0 = key0, k1 = key1;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k0 += 0x9E3779B97F4A7C15ull; k1 += 0xBB67AE8584CAA73Bull; }
    const uint64_t hi0 = __umul64hi(0xD2E7470EE14C6C93ull, c0), lo0 = 0xD2E7470EE14C6C93ull * c0;
    const uint64_t hi1 = __umul64hi(0xCA5A826395121157ull, c2), lo1 = 0xCA5A826395121157ull * c2;
    const uint64_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

}  // namespace mpl
