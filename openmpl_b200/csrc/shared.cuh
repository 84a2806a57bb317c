// Device functions shared by the geometry translation units (metric_inputs.cu, associate.cu, track.cu), defined once so that every
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

// Sum over the 32 lanes of a full warp, in a fixed butterfly order.
__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct UniformCursor {  // sequential reader of one item's uniform stream under key (key, key1) with a one-block cache
  uint64_t v[4];
  int64_t blk;
  uint64_t base, key, key1;
  __device__ UniformCursor(uint64_t base_, uint64_t key_, uint64_t key1_ = 0ull) : blk(-1), base(base_), key(key_), key1(key1_) {}
  __device__ double get(int i) {
    const int64_t b = i >> 2;
    if (b != blk) { philox4x64_10(base + (uint64_t)b + 1ull, key, key1, v); blk = b; }  // numpy increments the counter before generating
    const int k = i & 3;
    const uint64_t raw = k == 0 ? v[0] : (k == 1 ? v[1] : (k == 2 ? v[2] : v[3]));
    return (double)(raw >> 11) * (1.0 / 9007199254740992.0);
  }
};

// The synthetic camera model of mpl_synth_project and mpl_synth_motion: x_cam = R (X - t), u = f x_cam / z + c, no clipping;
// o = (u, v, conf) in fp32, conf 0 behind the camera.  c is one [18] calibration row.
__device__ __forceinline__ void project_pixel(const double* c, const double (&X)[3], double conf, float* o) {
  double xc[3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
    xc[r] = c[3 * r] * (X[0] - c[9]) + c[3 * r + 1] * (X[1] - c[10]) + c[3 * r + 2] * (X[2] - c[11]);
  const double u = xc[0] / xc[2] * c[12] + c[14], w = xc[1] / xc[2] * c[13] + c[15];
  if (!(xc[2] > 0.0)) conf = 0.0;  // behind the camera: never a detection
  o[0] = (float)u; o[1] = (float)w; o[2] = (float)conf;
}

}  // namespace mpl
