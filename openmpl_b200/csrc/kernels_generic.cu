// Shape-generic CUDA kernels of the MPL lifter forward: every constructor flag of the reference is served by these
// (fp32 CUDA-core arithmetic).  The hot configurations additionally have tensor-core kernels (gemm_tcgen05.cu,
// spt_fused.cu) that replace the Linear / attention launches.
#include <algorithm>
#include <type_traits>

#include <cuda_fp16.h>

#include "kernels.cuh"

namespace mpl {

__device__ __forceinline__ float ldf(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldf(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void stf(float* p, float v) { *p = v; }
__device__ __forceinline__ void stf(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// split-plane operand format of the fp32-grade tensor-core mode: x ~ hi + lo with hi = bf16(x), lo = bf16(x - hi)
// (16 significand bits; the planes are `plane` elements apart)
__device__ __forceinline__ void store_split4(__nv_bfloat16* hi, int64_t plane, float a, float b, float c, float d) {
  const __nv_bfloat162 h0 = __floats2bfloat162_rn(a, b), h1 = __floats2bfloat162_rn(c, d);
  const uint32_t u0 = *reinterpret_cast<const uint32_t*>(&h0), u1 = *reinterpret_cast<const uint32_t*>(&h1);
  const __nv_bfloat162 l0 = __floats2bfloat162_rn(a - __uint_as_float(u0 << 16), b - __uint_as_float(u0 & 0xffff0000u));
  const __nv_bfloat162 l1 = __floats2bfloat162_rn(c - __uint_as_float(u1 << 16), d - __uint_as_float(u1 & 0xffff0000u));
  *reinterpret_cast<uint2*>(hi) = make_uint2(u0, u1);
  *reinterpret_cast<uint2*>(hi + plane) = make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
}
__device__ __forceinline__ void store_split1(__nv_bfloat16* hi, int64_t plane, float a) {
  const __nv_bfloat16 h = __float2bfloat16_rn(a);
  *hi = h;
  hi[plane] = __float2bfloat16_rn(a - __bfloat162float(h));
}

// ---------------------------------------------------------------------------------------------------------------------
// K1 joint embedding.  One thread per output element of x [V, B, J, d]; the 12-byte pose record is a warp broadcast.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embed_kernel(const EmbedArgs a) {
  const int64_t total = (int64_t)a.V * a.B * a.J * a.d;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = (int)(idx % a.d);
  int64_t row = idx / a.d;
  const int j = (int)(row % a.J);
  row /= a.J;
  const int64_t b = row % a.B;
  const int v = (int)(row / a.B);
  const float* p = a.poses[v] + b * a.pose_stride + j * 3;
  const float px = __ldg(p), py = __ldg(p + 1), pc = __ldg(p + 2);
  const float* W = a.We[v] + c * a.in_ch;
  float val = __ldg(a.be[v] + c);
  val = fmaf(__ldg(W), px, val);
  val = fmaf(__ldg(W + 1), py, val);
  if (a.in_ch == 3) val = fmaf(__ldg(W + 2), pc, val);
  if (a.add_conf || a.mult_conf) {
    const float ce = fmaf(__ldg(a.Wc[v] + c), pc, __ldg(a.bc[v] + c));
    if (a.add_conf) val += ce;
    if (a.mult_conf) val *= ce;
  }
  val += __ldg(a.Ps[v] + j * a.d + c);
  if (a.spatial_pos_mode == 1) {
    val += __ldg(a.pos3d + j * a.pos3d_ld + c);
  } else if (a.spatial_pos_mode == 2) {
    const float* r = a.rays[v] + b * a.pose_stride + j * 3;
    const float* ce = a.centers[v] + b * a.center_stride;
    const float dx = __ldg(r) - __ldg(ce), dy = __ldg(r + 1) - __ldg(ce + 1), dz = __ldg(r + 2) - __ldg(ce + 2);
    const float inv = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);  // F.normalize eps
    float pe = __ldg(a.bl + c);
    pe = fmaf(__ldg(a.Wl + c * 3), dx * inv, pe);
    pe = fmaf(__ldg(a.Wl + c * 3 + 1), dy * inv, pe);
    pe = fmaf(__ldg(a.Wl + c * 3 + 2), dz * inv, pe);
    val += pe;
  }
  a.x[idx] = val;
  if (a.conf != nullptr && c == 0) a.conf[(v * a.B + b) * a.J + j] = pc;
}

int launch_embed(const EmbedArgs& a, cudaStream_t s) {
  const int64_t total = (int64_t)a.V * a.B * a.J * a.d;
  if (total == 0) return MPL_OK;
  const int vec = try_launch_embed_vec(a, s);
  if (vec != 1) return vec;
  embed_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(a);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// FPT token build: one thread per element of tok [B, V, tok_w].
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ray_dir(const TokenArgs& a, int v, int64_t b, int j, float& dx, float& dy, float& dz) {
  const float* r = a.rays[v] + b * a.pose_stride + j * 3;
  const float* ce = a.centers[v] + b * a.center_stride;
  dx = __ldg(r) - __ldg(ce);
  dy = __ldg(r + 1) - __ldg(ce + 1);
  dz = __ldg(r + 2) - __ldg(ce + 2);
}

__global__ void __launch_bounds__(256) token_build_kernel(const TokenArgs a) {
  const int64_t total = a.B * a.V * (int64_t)a.tok_w;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int e = (int)(idx % a.tok_w);
  const int64_t bv = idx / a.tok_w;
  const int v = (int)(bv % a.V);
  const int64_t b = bv / a.V;
  const int d = a.d, J = a.J;
  int j, c;             // joint, channel inside the (possibly 2d-wide) joint slot
  bool is_ray = false;  // this element is a ray-embedding channel
  bool add_pos = true;
  int pos_c;  // channel inside the positional table row
  if (a.ray_layout == 1) {  // [J, 2d]: [x | ray]
    j = e / (2 * d);
    c = e % (2 * d);
    pos_c = c;
    if (c >= d) { is_ray = true; c -= d; }
  } else if (a.ray_layout == 2) {  // [2J, d]: J pose tokens then J ray tokens
    const int t = e / d;
    c = e % d;
    pos_c = c;
    if (t >= J) { is_ray = true; j = t - J; add_pos = false; } else { j = t; }
  } else {
    j = e / d;
    c = e % d;
    pos_c = c;
  }
  float val;
  float dx = 0.f, dy = 0.f, dz = 0.f;
  const bool need_dir = is_ray || (add_pos && a.pos_table == nullptr);
  if (need_dir) ray_dir(a, v, b, j, dx, dy, dz);
  if (is_ray) {
    val = __ldg(a.br + c);
    val = fmaf(__ldg(a.Wr + c * 3), dx, val);
    val = fmaf(__ldg(a.Wr + c * 3 + 1), dy, val);
    val = fmaf(__ldg(a.Wr + c * 3 + 2), dz, val);
  } else {
    val = a.xn[(((int64_t)v * a.B + b) * J + j) * d + c];
    if (a.Wcf != nullptr) {
      const float pc = __ldg(a.poses[v] + b * a.pose_stride + j * 3 + 2);
      val += fmaf(__ldg(a.Wcf + c), pc, __ldg(a.bcf + c));
    }
  }
  if (add_pos) {
    if (a.pos_table != nullptr) {
      val += __ldg(a.pos_table + j * a.pos_w + pos_c);
    } else {
      const float inv = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);
      float pe = __ldg(a.bl + pos_c);
      pe = fmaf(__ldg(a.Wl + pos_c * 3), dx * inv, pe);
      pe = fmaf(__ldg(a.Wl + pos_c * 3 + 1), dy * inv, pe);
      pe = fmaf(__ldg(a.Wl + pos_c * 3 + 2), dz * inv, pe);
      val += pe;
    }
  }
  a.tok[idx] = val;
}

int launch_token_build(const TokenArgs& a, cudaStream_t s) {
  const int64_t total = a.B * a.V * (int64_t)a.tok_w;
  if (total == 0) return MPL_OK;
  const int vec = try_launch_token_build_vec(a, s);
  if (vec != 1) return vec;
  token_build_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(a);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// LayerNorm: one warp per row, two passes over the row (second one hits L1), biased variance like nn.LayerNorm.
// MODE 0: fp32 out, 1: bf16 out, 2: split bf16 planes out (hi at y, lo at y + plane).
// ---------------------------------------------------------------------------------------------------------------------
template <int MODE, typename TO>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, int64_t ldx, int seg_len, int seg_stride,
                                                        const float* __restrict__ w, const float* __restrict__ b, float eps,
                                                        TO* __restrict__ y, int64_t ldy, int64_t rows, int C, int64_t plane) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* xr = x + row * ldx;
  const bool plain = (seg_len == seg_stride);
  float s = 0.f;
  for (int e = lane; e < C; e += 32) {
    const int col = plain ? e : (e / seg_len) * seg_stride + (e % seg_len);
    s += xr[col];
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
  for (int e = lane; e < C; e += 32) {
    const int col = plain ? e : (e / seg_len) * seg_stride + (e % seg_len);
    const float t = xr[col] - mean;
    q = fmaf(t, t, q);
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
  TO* yr = y + row * ldy;
  for (int e = lane; e < C; e += 32) {
    const int col = plain ? e : (e / seg_len) * seg_stride + (e % seg_len);
    const float o = (xr[col] - mean) * rstd * __ldg(w + e) + __ldg(b + e);
    if constexpr (MODE == 2) store_split1(yr + e, plane, o);
    else stf(yr + e, o);
  }
}

// Vectorised LayerNorm for the FPT widths (C % 128 == 0 is not required; C % 4 == 0 and C <= 32*4*MAXV4): the row
// lives in registers, one pass over HBM.  Used for the bf16 / tf32 operand-producing LayerNorms.
template <int MODE, typename TO, int MAXV4>
__global__ void __launch_bounds__(256) layernorm_vec_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ w,
                                                            const float* __restrict__ b, float eps, TO* __restrict__ y,
                                                            int64_t ldy, int64_t rows, int C, int64_t plane) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float4* xr = reinterpret_cast<const float4*>(x + row * ldx);
  const int n4 = C >> 2;
  float4 v[MAXV4];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV4; ++i) {
    const int e4 = lane + i * 32;
    if (e4 < n4) {
      v[i] = xr[e4];
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV4; ++i) {
    const int e4 = lane + i * 32;
    if (e4 < n4) {
      const float t0 = v[i].x - mean, t1 = v[i].y - mean, t2 = v[i].z - mean, t3 = v[i].w - mean;
      q += t0 * t0 + t1 * t1 + t2 * t2 + t3 * t3;
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
  const float4* w4 = reinterpret_cast<const float4*>(w);
  const float4* b4 = reinterpret_cast<const float4*>(b);
#pragma unroll
  for (int i = 0; i < MAXV4; ++i) {
    const int e4 = lane + i * 32;
    if (e4 < n4) {
      const float4 g = __ldg(w4 + e4), bb = __ldg(b4 + e4);
      float o0 = (v[i].x - mean) * rstd * g.x + bb.x;
      float o1 = (v[i].y - mean) * rstd * g.y + bb.y;
      float o2 = (v[i].z - mean) * rstd * g.z + bb.z;
      float o3 = (v[i].w - mean) * rstd * g.w + bb.w;
      if constexpr (MODE == 1) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o0, o1), hi = __floats2bfloat162_rn(o2, o3);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        reinterpret_cast<uint2*>(y + row * ldy)[e4] = pk;
      } else if constexpr (MODE == 2) {
        store_split4(y + row * ldy + 4 * e4, plane, o0, o1, o2, o3);
      } else {
        reinterpret_cast<float4*>(y + row * ldy)[e4] = make_float4(o0, o1, o2, o3);
      }
    }
  }
}

template <int MODE, typename TO>
static int launch_ln_any(const float* x, int64_t ldx, int seg_len, int seg_stride, const float* w, const float* b, float eps,
                         TO* y, int64_t ldy, int64_t rows, int C, cudaStream_t s, int64_t plane = 0) {
  if (rows == 0) return MPL_OK;
  const unsigned grid = (unsigned)ceil_div(rows, 8);
  const bool vec_ok = (seg_len == seg_stride) && (C % 4 == 0) && (ldx % 4 == 0) && (ldy % 4 == 0) && (plane % 4 == 0) &&
                      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(w) |
                        reinterpret_cast<uintptr_t>(b)) % 16 == 0);
  if (vec_ok && C <= 32 * 4 * 5) {
    layernorm_vec_kernel<MODE, TO, 5><<<grid, 256, 0, s>>>(x, ldx, w, b, eps, y, ldy, rows, C, plane);
  } else if (vec_ok && C <= 32 * 4 * 9) {
    layernorm_vec_kernel<MODE, TO, 9><<<grid, 256, 0, s>>>(x, ldx, w, b, eps, y, ldy, rows, C, plane);
  } else if (vec_ok && C <= 32 * 4 * 17) {
    layernorm_vec_kernel<MODE, TO, 17><<<grid, 256, 0, s>>>(x, ldx, w, b, eps, y, ldy, rows, C, plane);
  } else {
    layernorm_kernel<MODE, TO><<<grid, 256, 0, s>>>(x, ldx, seg_len, seg_stride, w, b, eps, y, ldy, rows, C, plane);
  }
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

int launch_layernorm(const float* x, int64_t ldx, int seg_len, int seg_stride, const float* w, const float* b, float eps,
                     float* y, int64_t ldy, int64_t rows, int C, cudaStream_t s) {
  return launch_ln_any<0, float>(x, ldx, seg_len, seg_stride, w, b, eps, y, ldy, rows, C, s);
}
int launch_layernorm_bf16(const float* x, int64_t ldx, const float* w, const float* b, float eps, __nv_bfloat16* y,
                          int64_t ldy, int64_t rows, int C, cudaStream_t s) {
  return launch_ln_any<1, __nv_bfloat16>(x, ldx, C, C, w, b, eps, y, ldy, rows, C, s);
}
int launch_layernorm_split(const float* x, int64_t ldx, const float* w, const float* b, float eps, __nv_bfloat16* y,
                           int64_t ldy, int64_t plane, int64_t rows, int C, cudaStream_t s) {
  return launch_ln_any<2, __nv_bfloat16>(x, ldx, C, C, w, b, eps, y, ldy, rows, C, s, plane);
}

// ---------------------------------------------------------------------------------------------------------------------
// Entry of the LayerNorm-fused FPT (bf16 mode): the residual rows as two bf16 planes (hi, lo) + their (sum, sum of squares)
// in statistics slot 0 (the other slots zeroed) -- what the residual-emit GEMM epilogue produces for every later block.
// ---------------------------------------------------------------------------------------------------------------------
template <int MAXV4>
__global__ void __launch_bounds__(256) ln_prep_kernel(const float* __restrict__ x, int64_t ldx, __nv_bfloat16* __restrict__ xb,
                                                      __nv_bfloat16* __restrict__ xl, int64_t ldb, float2* __restrict__ stats,
                                                      int slots, int64_t rows, int C) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float4* xr = reinterpret_cast<const float4*>(x + row * ldx);
  const int n4 = C >> 2;
  float s = 0.f, q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV4; ++i) {
    const int e4 = lane + i * 32;
    if (e4 < n4) {
      const float4 v = xr[e4];
      s += (v.x + v.y) + (v.z + v.w);
      q = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, q))));
      store_split4(xb + row * ldb + 4 * e4, xl - xb, v.x, v.y, v.z, v.w);
    }
  }
  s = warp_sum(s);
  q = warp_sum(q);
  const int64_t ld = (int64_t)((rows + 255) / 256 * 256);  // slot-major planes of `rows` rounded up to 256 (see gemm_tcgen05.cu)
  for (int i = lane; i < slots; i += 32) stats[i * ld + row] = (i == 0) ? make_float2(s, q) : make_float2(0.f, 0.f);
}

int launch_ln_prep(const float* x, int64_t ldx, __nv_bfloat16* xb, __nv_bfloat16* xl, int64_t ldb, void* stats, int slots,
                   int64_t rows, int C, cudaStream_t s) {
  if (rows == 0) return MPL_OK;
  if (C % 4 != 0 || ldx % 4 != 0 || ldb % 4 != 0 || C > 32 * 4 * 17) {
    set_error("launch_ln_prep: width %d is not supported", C);
    return MPL_ERR_UNSUPPORTED;
  }
  const unsigned grid = (unsigned)ceil_div(rows, 8);
  float2* st = reinterpret_cast<float2*>(stats);
  if (C <= 32 * 4 * 5) ln_prep_kernel<5><<<grid, 256, 0, s>>>(x, ldx, xb, xl, ldb, st, slots, rows, C);
  else if (C <= 32 * 4 * 9) ln_prep_kernel<9><<<grid, 256, 0, s>>>(x, ldx, xb, xl, ldb, st, slots, rows, C);
  else ln_prep_kernel<17><<<grid, 256, 0, s>>>(x, ldx, xb, xl, ldb, st, slots, rows, C);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// Pack-time fold of a LayerNorm into the Linear that consumes it: W' = bf16(W diag(gamma)), colsum[n] = sum_k W'[n,k]
// (of the ROUNDED values: it must cancel exactly what the tensor core multiplies), bias'[n] = b[n] + sum_k W[n,k] beta[k].
__global__ void __launch_bounds__(256) ln_fold_kernel(const float* __restrict__ W, const float* __restrict__ b,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      __nv_bfloat16* __restrict__ Wf, float* __restrict__ colsum,
                                                      float* __restrict__ bias_f, int N, int K, const int* __restrict__ kperm) {
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= N) return;
  const int lane = threadIdx.x & 31;
  float cs = 0.f, bb = 0.f;
  for (int k = lane; k < K; k += 32) {
    const int ks = kperm ? kperm[k] : k;  // source channel of packed input channel k
    const float w = W[(int64_t)n * K + ks];
    const __nv_bfloat16 r = __float2bfloat16_rn(w * gamma[ks]);
    Wf[(int64_t)n * K + k] = r;
    cs += __bfloat162float(r);
    bb = fmaf(w, beta[ks], bb);
  }
  cs = warp_sum(cs);
  bb = warp_sum(bb);
  if (lane == 0) {
    colsum[n] = cs;
    bias_f[n] = (b != nullptr ? b[n] : 0.f) + bb;
  }
}

int launch_ln_fold(const float* W, const float* b, const float* gamma, const float* beta, __nv_bfloat16* Wf, float* colsum,
                   float* bias_f, int N, int K, cudaStream_t s, const int* kperm) {
  if (N == 0) return MPL_OK;
  ln_fold_kernel<<<(unsigned)ceil_div(N, 8), 256, 0, s>>>(W, b, gamma, beta, Wf, colsum, bias_f, N, K, kperm);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// fp32 Linear on CUDA cores: 64x64 output tile, K step 16, 256 threads x (4x4) accumulators.  Any M, N, K, strides.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int LBM = 64, LBN = 64, LBK = 16;

__global__ void __launch_bounds__(256) linear_f32_kernel(const float* __restrict__ X, int64_t lda, const float* __restrict__ W,
                                                         const float* __restrict__ bias, const float* R, int64_t ldr,
                                                         float* Y, int64_t ldc, int64_t M, int N, int K, int act) {
  __shared__ float As[LBK][LBM + 4];
  __shared__ float Bs[LBK][LBN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t m0 = (int64_t)blockIdx.x * LBM;
  const int n0 = blockIdx.y * LBN;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int lr = tid >> 2;         // 0..63 : row of the tile this thread loads
  const int lk = (tid & 3) * 4;    // 0,4,8,12 : first k of its 4 consecutive elements
  for (int k0 = 0; k0 < K; k0 += LBK) {
    {
      const int64_t m = m0 + lr;
      const float* src = X + m * lda + k0 + lk;
#pragma unroll
      for (int i = 0; i < 4; ++i) As[lk + i][lr] = (m < M && k0 + lk + i < K) ? src[i] : 0.f;
      const int n = n0 + lr;
      const float* wsrc = W + (int64_t)n * K + k0 + lk;
#pragma unroll
      for (int i = 0; i < 4; ++i) Bs[lk + i][lr] = (n < N && k0 + lk + i < K) ? __ldg(wsrc + i) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < LBK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a4[4] = {av.x, av.y, av.z, av.w};
      const float b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j];
      if (bias != nullptr) v += __ldg(bias + n);
      v = apply_act(v, act);
      if (R != nullptr) v += R[m * ldr + n];
      Y[m * ldc + n] = v;
    }
  }
}

int launch_linear_f32(const float* X, int64_t lda, const float* W, const float* bias, const float* R, int64_t ldr, float* Y,
                      int64_t ldc, int64_t M, int N, int K, int act, cudaStream_t s) {
  if (M == 0 || N == 0) return MPL_OK;
  dim3 grid((unsigned)ceil_div(M, LBM), (unsigned)ceil_div(N, LBN));
  linear_f32_kernel<<<grid, 256, 0, s>>>(X, lda, W, bias, R, ldr, Y, ldc, M, N, K, act);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Generic attention core.  One warp per (set, head, query row); probabilities staged in shared memory.
// Narrow heads (hd <= 16: the 17-token spatial sets and the V*J keypoint-token sets): lanes sweep the keys.
// Wide heads (view tokens, hd = D/H): lanes sweep the head channels, scores by warp reduction.
// ---------------------------------------------------------------------------------------------------------------------
template <typename TI, typename TO>
__global__ void __launch_bounds__(128) attention_kernel(const TI* __restrict__ qkv, TO* __restrict__ out, int64_t sets, int N,
                                                        int H, int hd, float scale, const float* __restrict__ conf) {
  extern __shared__ float psm[];  // [4 warps][N]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t task = (int64_t)blockIdx.x * 4 + warp;
  const int64_t total = sets * H * N;
  if (task >= total) return;
  const int i = (int)(task % N);
  const int h = (int)((task / N) % H);
  const int64_t set = task / ((int64_t)N * H);
  const int C = H * hd;
  const int64_t ld = 3 * (int64_t)C;
  const TI* base = qkv + set * N * ld;
  const TI* q = base + (int64_t)i * ld + h * hd;
  const TI* kb = base + C + h * hd;
  const TI* vb = base + 2 * C + h * hd;
  float* p = psm + warp * N;
  float mx = -INFINITY;
  if (hd <= 16) {
    float qr[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) qr[t] = (t < hd) ? ldf(q + t) : 0.f;
    for (int j = lane; j < N; j += 32) {
      const TI* kj = kb + (int64_t)j * ld;
      float sc = 0.f;
#pragma unroll
      for (int t = 0; t < 16; ++t)
        if (t < hd) sc = fmaf(qr[t], ldf(kj + t), sc);
      sc *= scale;
      p[j] = sc;
      mx = fmaxf(mx, sc);
    }
  } else {
    for (int j = 0; j < N; ++j) {
      const TI* kj = kb + (int64_t)j * ld;
      float part = 0.f;
      for (int t = lane; t < hd; t += 32) part = fmaf(ldf(q + t), ldf(kj + t), part);
      part = warp_sum(part) * scale;
      if (lane == 0) p[j] = part;
      mx = fmaxf(mx, part);
    }
  }
  mx = warp_max(mx);
  __syncwarp();
  float sum = 0.f;
  for (int j = lane; j < N; j += 32) {
    const float e = expf(p[j] - mx);
    p[j] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  float norm = 1.0f / sum;
  if (conf != nullptr) norm *= __ldg(conf + set * N + i);  // post-softmax query-row scaling, multiview_mpl.py:61-62
  __syncwarp();
  TO* o = out + (set * N + i) * (int64_t)C + h * hd;
  for (int t = lane; t < hd; t += 32) {
    float acc = 0.f;
    for (int j = 0; j < N; ++j) acc = fmaf(p[j], ldf(vb + (int64_t)j * ld + t), acc);
    acc *= norm;
    stf(o + t, acc);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Narrow heads (hd <= 8; the 17-token spatial sets and the V*J keypoint-token sets): a CTA stages the q|k|v rows of G
// whole sets in shared memory with coalesced 16-byte loads, then one thread per (set, head, query) runs the exact
// two-pass softmax (max, then exp / sum) over the N keys reading k_j / v_j as broadcast shared-memory vectors.
// ---------------------------------------------------------------------------------------------------------------------
template <typename TI, typename TO, int HD>
__global__ void __launch_bounds__(256) attention_narrow_kernel(const TI* __restrict__ qkv, TO* __restrict__ out, int64_t sets,
                                                               int N, int H, int G, float scale, const float* __restrict__ conf) {
  extern __shared__ float sm[];  // [G][N][3C]
  const int C = H * HD;
  const int ld = 3 * C;
  const int64_t set0 = (int64_t)blockIdx.x * G;
  const int g_here = (int)min((int64_t)G, sets - set0);
  const int64_t n_el = (int64_t)g_here * N * ld;
  const TI* src = qkv + set0 * N * ld;
  for (int64_t i = threadIdx.x; i < n_el; i += blockDim.x) sm[i] = ldf(src + i);
  __syncthreads();
  const int items = g_here * H * N;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int i = it % N;
    const int h = (it / N) % H;
    const int g = it / (N * H);
    const float* base = sm + (size_t)g * N * ld;
    const float* q = base + i * ld + h * HD;
    const float* kb = base + C + h * HD;
    const float* vb = base + 2 * C + h * HD;
    float qr[HD];
#pragma unroll
    for (int t = 0; t < HD; ++t) qr[t] = q[t] * scale;
    float mx = -INFINITY;
    for (int j = 0; j < N; ++j) {
      const float* kj = kb + j * ld;
      float sc = 0.f;
#pragma unroll
      for (int t = 0; t < HD; ++t) sc = fmaf(qr[t], kj[t], sc);
      mx = fmaxf(mx, sc);
    }
    float sum = 0.f, acc[HD];
#pragma unroll
    for (int t = 0; t < HD; ++t) acc[t] = 0.f;
    for (int j = 0; j < N; ++j) {
      const float* kj = kb + j * ld;
      const float* vj = vb + j * ld;
      float sc = 0.f;
#pragma unroll
      for (int t = 0; t < HD; ++t) sc = fmaf(qr[t], kj[t], sc);
      const float e = expf(sc - mx);
      sum += e;
#pragma unroll
      for (int t = 0; t < HD; ++t) acc[t] = fmaf(e, vj[t], acc[t]);
    }
    float norm = 1.0f / sum;
    if (conf != nullptr) norm *= __ldg(conf + (set0 + g) * N + i);  // post-softmax query-row scaling, multiview_mpl.py:61-62
    TO* o = out + ((set0 + g) * N + i) * (int64_t)C + h * HD;
#pragma unroll
    for (int t = 0; t < HD; ++t) {
      stf(o + t, acc[t] * norm);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Keypoint-token attention of the FPT in bf16 mode where the fused FPT kernel does not apply (FPT_blocks_view_keypoint_tokens
// with J != 17 or an MLP hidden width != 64: N = V * J <= 272 tokens of width 32, 8 heads of 4; N need not be a multiple of
// the 17-key chunk below): a CTA keeps G whole token sets in shared memory as fp16 with the channels of each head PAIR interleaved
// (word = (head 2p, head 2p+1) at one head-dim, q pre-scaled by scale * log2 e), exactly the staging format of the SPT
// kernel, so the softmax of two heads runs in packed half2 arithmetic straight from 16-byte shared-memory loads.  One
// thread per (token row, head pair), two passes over the keys (max; then exp2 / sum / PV with the scores recomputed --
// N is too long for registers).  Partial sums are kept in fp16 for 17 keys at a time and flushed into fp32.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ __half2 as_h2(uint32_t u) { return *reinterpret_cast<__half2*>(&u); }

__global__ void __launch_bounds__(256) attention_kp_h4_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out,
                                                             int64_t sets, int N, int G, float scale_log2e) {
  constexpr int QP = 104, QPW = QP / 2, RP4 = QPW / 4;  // fp16 row pitch 208 B (see spt_fused.cu)
  extern __shared__ __align__(16) uint32_t kp_sm[];       // [G * N][QPW]
  const int64_t set0 = (int64_t)blockIdx.x * G;
  const int g_here = (int)min((int64_t)G, sets - set0);
  const int rows = g_here * N;
  // stage: 12 groups of 8 channels per row, bf16 -> fp16, interleave the two heads of a group
  for (int it = threadIdx.x; it < rows * 12; it += blockDim.x) {
    const int r = it / 12, grp = it - r * 12;
    const uint4 u = *reinterpret_cast<const uint4*>(qkv + ((set0 * N + r) * 96 + grp * 8));
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    float f[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) { f[2 * i] = __uint_as_float(w[i] << 16); f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
    const float sc = grp < 4 ? scale_log2e : 1.0f;
    uint4 o;
    uint32_t* op = &o.x;
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(op[d]) : "f"(f[4 + d] * sc), "f"(f[d] * sc));
    }
    *reinterpret_cast<uint4*>(kp_sm + r * QPW + grp * 4) = o;
  }
  __syncthreads();
  for (int it = threadIdx.x; it < rows * 4; it += blockDim.x) {
    const int r = it >> 2, p = it & 3;
    const int s0 = (r / N) * N;  // first row of the row's set
    const uint4* setp = reinterpret_cast<const uint4*>(kp_sm + s0 * QPW);
    const uint4 q = reinterpret_cast<const uint4*>(kp_sm + r * QPW)[p];
    __half2 mx = __float2half2_rn(-60000.f);
    for (int j = 0; j < N; ++j) {
      const uint4 k = setp[j * RP4 + 4 + p];
      __half2 s = __hmul2(as_h2(q.x), as_h2(k.x));
      s = __hfma2(as_h2(q.y), as_h2(k.y), s);
      s = __hfma2(as_h2(q.z), as_h2(k.z), s);
      s = __hfma2(as_h2(q.w), as_h2(k.w), s);
      mx = __hmax2(mx, s);
    }
    float sum0 = 0.f, sum1 = 0.f, o0[4] = {0.f, 0.f, 0.f, 0.f}, o1[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j0 = 0; j0 < N; j0 += 17) {
      const __half2 z = __float2half2_rn(0.f);
      __half2 hs = z, a0 = z, a1 = z, a2 = z, a3 = z;
#pragma unroll
      for (int jj = 0; jj < 17; ++jj) {
        const int j = j0 + jj;
        if (j < N) {
          const uint4 k = setp[j * RP4 + 4 + p];
          const uint4 v = setp[j * RP4 + 8 + p];
          __half2 s = __hmul2(as_h2(q.x), as_h2(k.x));
          s = __hfma2(as_h2(q.y), as_h2(k.y), s);
          s = __hfma2(as_h2(q.z), as_h2(k.z), s);
          s = __hfma2(as_h2(q.w), as_h2(k.w), s);
          const __half2 d = __hsub2(s, mx);
          uint32_t eu;
          asm("ex2.approx.f16x2 %0, %1;" : "=r"(eu) : "r"(*reinterpret_cast<const uint32_t*>(&d)));
          const __half2 e = as_h2(eu);
          hs = __hadd2(hs, e);
          a0 = __hfma2(e, as_h2(v.x), a0);
          a1 = __hfma2(e, as_h2(v.y), a1);
          a2 = __hfma2(e, as_h2(v.z), a2);
          a3 = __hfma2(e, as_h2(v.w), a3);
        }
      }
      const float2 fs = __half22float2(hs), f0 = __half22float2(a0), f1 = __half22float2(a1), f2 = __half22float2(a2),
                   f3 = __half22float2(a3);
      sum0 += fs.x; sum1 += fs.y;
      o0[0] += f0.x; o1[0] += f0.y; o0[1] += f1.x; o1[1] += f1.y; o0[2] += f2.x; o1[2] += f2.y; o0[3] += f3.x; o1[3] += f3.y;
    }
    const float i0 = 1.0f / sum0, i1 = 1.0f / sum1;
    __nv_bfloat162 b[4] = {__floats2bfloat162_rn(o0[0] * i0, o0[1] * i0), __floats2bfloat162_rn(o0[2] * i0, o0[3] * i0),
                           __floats2bfloat162_rn(o1[0] * i1, o1[1] * i1), __floats2bfloat162_rn(o1[2] * i1, o1[3] * i1)};
    uint4 ou;
    ou.x = *reinterpret_cast<uint32_t*>(&b[0]); ou.y = *reinterpret_cast<uint32_t*>(&b[1]);
    ou.z = *reinterpret_cast<uint32_t*>(&b[2]); ou.w = *reinterpret_cast<uint32_t*>(&b[3]);
    *reinterpret_cast<uint4*>(out + (set0 * N + r) * 32 + p * 8) = ou;  // channels 8p .. 8p+7 = heads 2p, 2p+1
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// K4 view-token attention of the FPT (N = V tokens of width D, hd = D / H = 136 | 68): HBM-bound, 3 D in / D out per
// row.  One CTA per pose, one thread per CE-element chunk of the row (D / CE threads): each thread loads its chunk of
// q, k, v for all V views with 16- or 8-byte loads, forms partial V x V scores over its chunk, the chunks of a head are
// summed through shared memory, softmax on V values, then the thread writes its chunk of all V output rows.
// ---------------------------------------------------------------------------------------------------------------------
template <typename T, int CE> struct ChunkIO;
template <> struct ChunkIO<__nv_bfloat16, 8> {
  using Pack = uint4;
  static __device__ __forceinline__ void unpack(const uint4& u, float (&f)[8]) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { f[2 * i] = __uint_as_float(w[i] << 16); f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
  }
  static __device__ __forceinline__ void unpack2(const uint4& u, float2 (&f)[4]) {  // element pairs for f32x2 arithmetic
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = make_float2(__uint_as_float(w[i] << 16), __uint_as_float(w[i] & 0xffff0000u));
  }
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&f)[8]) {
    unpack(*reinterpret_cast<const uint4*>(p), f);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = u;
  }
};
template <> struct ChunkIO<__nv_bfloat16, 4> {
  using Pack = uint2;
  static __device__ __forceinline__ void unpack(const uint2& u, float (&f)[4]) {
    f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xffff0000u);
    f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xffff0000u);
  }
  static __device__ __forceinline__ void unpack2(const uint2& u, float2 (&f)[2]) {
    f[0] = make_float2(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u));
    f[1] = make_float2(__uint_as_float(u.y << 16), __uint_as_float(u.y & 0xffff0000u));
  }
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&f)[4]) {
    unpack(*reinterpret_cast<const uint2*>(p), f);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[4]) {
    uint2 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 2; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    *reinterpret_cast<uint2*>(p) = u;
  }
};
template <> struct ChunkIO<float, 4> {
  using Pack = float4;
  static __device__ __forceinline__ void unpack(const float4& u, float (&f)[4]) { f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w; }
  static __device__ __forceinline__ void unpack2(const float4& u, float2 (&f)[2]) { f[0] = make_float2(u.x, u.y); f[1] = make_float2(u.z, u.w); }
  static __device__ __forceinline__ void load(const float* p, float (&f)[4]) { unpack(*reinterpret_cast<const float4*>(p), f); }
  static __device__ __forceinline__ void store(float* p, const float (&f)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
  }
};

// DT / CPH: row width and chunks per head compiled in for the shipped widths (1088 / 544, 17), 0 = the runtime arguments
// SPLIT_OUT (fp32 q|k|v in, the fp32-grade tensor-core mode): `out` is the hi plane of a split bf16 pair, lo `plane` elements on
template <typename T, int V, int CE, bool SPLIT_OUT, int DT, int CPH>
__global__ void __launch_bounds__(288) attention_views_kernel(const T* __restrict__ qkv, T* __restrict__ out, int64_t poses,
                                                              int D_arg, int hd, float scale, int64_t plane) {
  const int D = DT ? DT : D_arg;
  extern __shared__ float sm[];       // partial [nchunks][V*V] then probs [H][V*V]
  const int nchunks = D / CE;         // == blockDim.x
  const int cph = CPH ? CPH : hd / CE;  // chunks per head
  const int H = D / hd;
  const int c = threadIdx.x;
  float* part = sm;
  float* prob = sm + (size_t)nchunks * V * V;
  // The q / k / v chunks of the pose stay PACKED in registers (one 16- or 8-byte word per view and operand) and are
  // widened at the point of use: the kernel is HBM-bound and register-limited, and the packed form doubles the number
  // of poses in flight per SM.
  using Pack = typename ChunkIO<T, CE>::Pack;
  for (int64_t pose = blockIdx.x; pose < poses; pose += gridDim.x) {
    const T* row0 = qkv + pose * V * 3 * (int64_t)D;
    Pack q[V], k[V], vv[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      q[v] = *reinterpret_cast<const Pack*>(row0 + (int64_t)v * 3 * D + c * CE);
      k[v] = *reinterpret_cast<const Pack*>(row0 + (int64_t)v * 3 * D + D + c * CE);
      vv[v] = *reinterpret_cast<const Pack*>(row0 + (int64_t)v * 3 * D + 2 * D + c * CE);
    }
    // the dot products and the probability-weighted sums below run on packed f32x2 FMAs (element pairs of the chunk)
    {
      float2 k2[V][CE / 2];  // the keys are widened once, the queries one at a time
#pragma unroll
      for (int j = 0; j < V; ++j) ChunkIO<T, CE>::unpack2(k[j], k2[j]);
#pragma unroll
      for (int i = 0; i < V; ++i) {
        float2 qi[CE / 2];
        ChunkIO<T, CE>::unpack2(q[i], qi);
#pragma unroll
        for (int j = 0; j < V; ++j) {
          float2 a = make_float2(0.f, 0.f);
#pragma unroll
          for (int e = 0; e < CE / 2; ++e) a = __ffma2_rn(qi[e], k2[j][e], a);
          part[c * (V * V) + i * V + j] = a.x + a.y;
        }
      }
    }
    __syncthreads();
    if ((V & (V - 1)) == 0 && blockDim.x % V == 0) {
      // one thread per (head, query, key): sum the head's chunk partials (17 conflict-free loads instead of a 68-long
      // chain on one warp), softmax across the V lanes of the row with shuffles
      const unsigned mask = __activemask();
      const int total = H * V * V;
      for (int base = 0; base < total; base += blockDim.x) {
        const int idx = base + threadIdx.x;
        const bool live = idx < total;
        const int h = (live ? idx : 0) / (V * V), ij = (live ? idx : 0) % (V * V);
        float a = 0.f;
        const float* pp = part + h * cph * (V * V) + ij;
        if (CPH) {
#pragma unroll
          for (int cc = 0; cc < CPH; ++cc) a += pp[cc * (V * V)];
        } else {
          for (int cc = 0; cc < cph; ++cc) a += pp[cc * (V * V)];
        }
        a *= scale;
        float mx = a;
#pragma unroll
        for (int o = V / 2; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(mask, mx, o));
        const float e = expf(a - mx);
        float sum = e;
#pragma unroll
        for (int o = V / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(mask, sum, o);
        if (live) prob[idx] = e / sum;
      }
    } else {
      // V = 3, 5, 6, 7 (CMU Panoptic: 5 views): the same one-thread-per-(head, query, key) spread, the row's V scores
      // exchanged through shared memory instead of shuffles (a separate compile-time path: the V = 4 kernel is untouched)
      const int total = H * V * V;
      for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        const int h = idx / (V * V), ij = idx % (V * V);
        float a = 0.f;
        const float* pp = part + h * cph * (V * V) + ij;
        if (CPH) {
#pragma unroll
          for (int cc = 0; cc < CPH; ++cc) a += pp[cc * (V * V)];
        } else {
          for (int cc = 0; cc < cph; ++cc) a += pp[cc * (V * V)];
        }
        prob[idx] = a * scale;
      }
      __syncthreads();
      float pr[V];  // this thread's probabilities: the launcher guarantees blockDim >= H * V, i.e. at most V rounds
      int n_mine = 0;
      for (int idx = threadIdx.x; idx < total; idx += blockDim.x, ++n_mine) {
        const float* row = prob + (idx / V) * V;
        float mx = row[0];
#pragma unroll
        for (int j = 1; j < V; ++j) mx = fmaxf(mx, row[j]);
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < V; ++j) sum += expf(row[j] - mx);
        if (n_mine < (int)(sizeof(pr) / sizeof(float))) pr[n_mine] = expf(prob[idx] - mx) / sum;
      }
      __syncthreads();  // every score has been read
      n_mine = 0;
      for (int idx = threadIdx.x; idx < total; idx += blockDim.x, ++n_mine)
        if (n_mine < (int)(sizeof(pr) / sizeof(float))) prob[idx] = pr[n_mine];
    }
    __syncthreads();
    const int h = c / cph;
    float2 o2[V][CE / 2];
#pragma unroll
    for (int i = 0; i < V; ++i)
#pragma unroll
      for (int e = 0; e < CE / 2; ++e) o2[i][e] = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float2 vj[CE / 2];
      ChunkIO<T, CE>::unpack2(vv[j], vj);
#pragma unroll
      for (int i = 0; i < V; ++i) {
        const float pj = prob[h * (V * V) + i * V + j];
        const float2 pj2 = make_float2(pj, pj);
#pragma unroll
        for (int e = 0; e < CE / 2; ++e) o2[i][e] = __ffma2_rn(pj2, vj[e], o2[i][e]);
      }
    }
#pragma unroll
    for (int i = 0; i < V; ++i) {
      if constexpr (SPLIT_OUT) {
        static_assert(!SPLIT_OUT || CE == 4, "split output works on 4-element chunks");
        store_split4(reinterpret_cast<__nv_bfloat16*>(out) + (pose * V + i) * (int64_t)D + c * CE, plane, o2[i][0].x, o2[i][0].y,
                     o2[i][1].x, o2[i][1].y);
      } else {
        float o[CE];
#pragma unroll
        for (int e = 0; e < CE / 2; ++e) {
          o[2 * e] = o2[i][e].x;
          o[2 * e + 1] = o2[i][e].y;
        }
        ChunkIO<T, CE>::store(out + (pose * V + i) * (int64_t)D + c * CE, o);
      }
    }
    __syncthreads();  // prob / part are reused by the next pose
  }
}

template <typename T, int CE, bool SPLIT_OUT>
static int launch_attention_views(const T* qkv, T* out, int64_t poses, int V, int D, int hd, float scale, cudaStream_t s,
                                  int64_t plane = 0) {
  const int threads = D / CE;
  const int H = D / hd;
  const size_t smem = ((size_t)threads + H) * V * V * sizeof(float);
  const unsigned grid = (unsigned)std::min<int64_t>(poses, (int64_t)kNumSMs * 32);
#define MPL_AV(VV)                                                                                                      \
  case VV: {                                                                                                            \
    auto kern = (D == 136 * CE && hd == 17 * CE) ? attention_views_kernel<T, VV, CE, SPLIT_OUT, 136 * CE, 17>                   \
                                                 : attention_views_kernel<T, VV, CE, SPLIT_OUT, 0, 0>;                           \
    if (smem > 48 * 1024) MPL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<grid, threads, smem, s>>>(qkv, out, poses, D, hd, scale, plane);                                                  \
  } break;
  switch (V) {
    MPL_AV(2) MPL_AV(3) MPL_AV(4) MPL_AV(5) MPL_AV(6) MPL_AV(7) MPL_AV(8)
    default: return MPL_ERR_UNSUPPORTED;
  }
#undef MPL_AV
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

template <typename TI, typename TO>
static int launch_attention_any(const TI* qkv, TO* out, int64_t sets, int N, int H, int hd, float scale, const float* conf,
                                cudaStream_t s) {
  const int64_t total = sets * H * N;
  if (total == 0) return MPL_OK;
  const int C = H * hd;
  // (1) view tokens with wide heads: the HBM-bound K4 kernel (same element type in and out, no confidence scaling)
  if constexpr (std::is_same<TI, TO>::value) {
    if (conf == nullptr && N >= 2 && N <= 8 && hd >= 16) {
      constexpr bool is_bf16 = std::is_same<TI, __nv_bfloat16>::value;
      const bool aligned = (reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out)) % 16 == 0;
      if constexpr (is_bf16) {
        if (aligned && hd % 8 == 0 && N <= 4 && C / 8 <= 288 && C / 8 >= H * N)
          return launch_attention_views<TI, 8, false>(qkv, out, sets, N, C, hd, scale, s);
        if (aligned && hd % 4 == 0 && C / 4 <= 288 && C / 4 >= H * N)
          return launch_attention_views<TI, 4, false>(qkv, out, sets, N, C, hd, scale, s);
      } else {
        if (aligned && hd % 4 == 0 && C / 4 <= 288 && C / 4 >= H * N)
          return launch_attention_views<TI, 4, false>(qkv, out, sets, N, C, hd, scale, s);
      }
    }
  }
  // (2a) bf16 keypoint tokens, 8 heads of 4: fp16 head-pair staging + packed half2 softmax
  if constexpr (std::is_same<TI, __nv_bfloat16>::value && std::is_same<TO, __nv_bfloat16>::value) {
    if (conf == nullptr && hd == 4 && H == 8 && N <= 272 &&
        (reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out)) % 16 == 0) {
      const size_t per_set = (size_t)N * 208;
      const int G = (int)std::max<size_t>(1, std::min<size_t>(56 * 1024 / per_set, 8));
      const size_t smem = per_set * G;
      static bool attr_set[64] = {};
      int dev = 0;
      MPL_CUDA(cudaGetDevice(&dev));
      if (dev < 0 || dev >= 64 || !attr_set[dev]) {
        MPL_CUDA(cudaFuncSetAttribute(attention_kp_h4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 57 * 1024));
        if (dev >= 0 && dev < 64) attr_set[dev] = true;
      }
      attention_kp_h4_kernel<<<(unsigned)ceil_div(sets, G), 256, smem, s>>>(qkv, out, sets, N, G, scale * 1.4426950408889634f);
      MPL_LAUNCH_CHECK();
      return MPL_OK;
    }
  }
  // (2) narrow heads: whole sets staged in shared memory
  if (hd == 4 || hd == 8 || hd == 2) {
    const size_t per_set = (size_t)N * 3 * C * sizeof(float);
    if (per_set <= 96 * 1024) {
      int G = (int)std::max<size_t>(1, std::min<size_t>(48 * 1024 / per_set, 16));
      const size_t smem = per_set * G;
      const unsigned grid = (unsigned)ceil_div(sets, G);
#define MPL_AN(HD)                                                                                                   \
  {                                                                                                                  \
    auto kern = attention_narrow_kernel<TI, TO, HD>;                                                       \
    if (smem > 48 * 1024) MPL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)); \
    kern<<<grid, 256, smem, s>>>(qkv, out, sets, N, H, G, scale, conf);                                              \
  }
      if (hd == 4) MPL_AN(4) else if (hd == 8) MPL_AN(8) else MPL_AN(2)
#undef MPL_AN
      MPL_LAUNCH_CHECK();
      return MPL_OK;
    }
  }
  // (3) anything else: one warp per (set, head, query)
  const size_t smem = 4 * (size_t)N * sizeof(float);
  attention_kernel<TI, TO><<<(unsigned)ceil_div(total, 4), 128, smem, s>>>(qkv, out, sets, N, H, hd, scale, conf);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

int launch_attention_f32(const float* qkv, float* out, int64_t sets, int N, int H, int hd, float scale, const float* conf,
                         cudaStream_t s) {
  return launch_attention_any<float, float>(qkv, out, sets, N, H, hd, scale, conf, s);
}
int launch_attention_bf16(const __nv_bfloat16* qkv, __nv_bfloat16* out, int64_t sets, int N, int H, int hd, float scale,
                          cudaStream_t s) {
  return launch_attention_any<__nv_bfloat16, __nv_bfloat16>(qkv, out, sets, N, H, hd, scale, nullptr, s);
}
// fp32 q|k|v in, split bf16 planes out (A operand of the split-mode proj GEMM).  View tokens with wide heads write the
// planes directly; every other shape runs the fp32 kernel into `scratch` ([sets * N, C] fp32) and splits it afterwards.
int launch_attention_split(const float* qkv, __nv_bfloat16* out, int64_t plane, float* scratch, int64_t sets, int N, int H,
                           int hd, float scale, cudaStream_t s) {
  if (sets == 0) return MPL_OK;
  const int C = H * hd;
  const bool aligned = (reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out)) % 16 == 0 && plane % 4 == 0;
  if (N >= 2 && N <= 8 && hd >= 16 && aligned && hd % 4 == 0 && C / 4 <= 288 && C / 4 >= H * N)
    return launch_attention_views<float, 4, true>(qkv, reinterpret_cast<float*>(out), sets, N, C, hd, scale, s, plane);
  MPL_TRY((launch_attention_any<float, float>(qkv, scratch, sets, N, H, hd, scale, nullptr, s)));
  return launch_to_split(scratch, out, sets * N * (int64_t)C, plane, s);
}

// ---------------------------------------------------------------------------------------------------------------------
// Conv1d(V -> 1, k = 1) over the view axis.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) view_mean_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                        const float* __restrict__ bias, float* __restrict__ y, int64_t B, int V,
                                                        int E) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * E) return;
  const int e = (int)(idx % E);
  const int64_t b = idx / E;
  float acc = __ldg(bias);
  for (int v = 0; v < V; ++v) acc = fmaf(__ldg(w + v), x[(b * V + v) * E + e], acc);
  y[idx] = acc;
}

int launch_view_mean(const float* x, const float* w, const float* bias, float* y, int64_t B, int V, int E, cudaStream_t s) {
  if (B * E == 0) return MPL_OK;
  view_mean_kernel<<<(unsigned)ceil_div(B * E, 256), 256, 0, s>>>(x, w, bias, y, B, V, E);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// K5 fused default head.  One CTA (128 threads) per pose: the V rows of E channels are normalised (View_norm),
// combined with the Conv1d weights, normalised again (eps 1e-5) in shared memory, then each warp computes output
// channels of the E -> 3J Linear by warp-reduced dot products.  Reads V*E floats, writes 3J floats per pose.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_sum_128(float v, float* red) {
  v = warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  return red[0] + red[1] + red[2] + red[3];
}

__global__ void __launch_bounds__(128) head_fused_kernel(const HeadArgs a) {
  extern __shared__ float sm[];  // pooled [E]
  __shared__ float red[4];
  float* pooled = sm;
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x;
  const int E = a.E;
  for (int e = tid; e < E; e += 128) pooled[e] = __ldg(a.wm_b);
  for (int v = 0; v < a.V; ++v) {
    const float* row = a.tok + (b * a.V + v) * (int64_t)a.tok_w;
    float s = 0.f;
    for (int e = tid; e < E; e += 128) s += row[(e / a.seg_len) * a.seg_stride + (e % a.seg_len)];
    const float mean = block_sum_128(s, red) / (float)E;
    float q = 0.f;
    for (int e = tid; e < E; e += 128) {
      const float t = row[(e / a.seg_len) * a.seg_stride + (e % a.seg_len)] - mean;
      q = fmaf(t, t, q);
    }
    const float rstd = rsqrtf(block_sum_128(q, red) / (float)E + 1e-6f);
    const float wv = __ldg(a.wm_w + v);
    for (int e = tid; e < E; e += 128) {
      const float xv = row[(e / a.seg_len) * a.seg_stride + (e % a.seg_len)];
      pooled[e] += wv * ((xv - mean) * rstd * __ldg(a.vn_w + e) + __ldg(a.vn_b + e));
    }
  }
  __syncthreads();
  float s = 0.f;
  for (int e = tid; e < E; e += 128) s += pooled[e];
  const float mean = block_sum_128(s, red) / (float)E;
  float q = 0.f;
  for (int e = tid; e < E; e += 128) {
    const float t = pooled[e] - mean;
    q = fmaf(t, t, q);
  }
  const float rstd = rsqrtf(block_sum_128(q, red) / (float)E + 1e-5f);  // head LayerNorm: default eps (multiview_mpl.py:284)
  __syncthreads();
  for (int e = tid; e < E; e += 128) pooled[e] = (pooled[e] - mean) * rstd * __ldg(a.hn_w + e) + __ldg(a.hn_b + e);
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  for (int o = warp; o < a.out_dim; o += 4) {
    const float* wr = a.hw + (int64_t)o * E;
    float acc = 0.f;
    for (int e = lane; e < E; e += 32) acc = fmaf(pooled[e], __ldg(wr + e), acc);
    acc = warp_sum(acc);
    if (lane == 0) a.out[b * a.out_dim + o] = acc + __ldg(a.hb + o);
  }
}

int launch_head_fused(const HeadArgs& a, cudaStream_t s) {
  if (a.B == 0) return MPL_OK;
  const int vec = try_launch_head_warp(a, s);
  if (vec != 1) return vec;
  head_fused_kernel<<<(unsigned)a.B, 128, (size_t)a.E * sizeof(float), s>>>(a);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// pack helpers
// ---------------------------------------------------------------------------------------------------------------------
__global__ void fold_bn_kernel(const float* W, const float* b, const float* g, const float* beta, const float* mean,
                               const float* var, float eps, float* Wf, float* bf, int N, int K) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * K) return;
  const int n = (int)(idx / K);
  const float sc = g[n] / sqrtf(var[n] + eps);
  Wf[idx] = W[idx] * sc;
  if (idx % K == 0) bf[n] = (b[n] - mean[n]) * sc + beta[n];
}
int launch_fold_bn(const float* W, const float* b, const float* g, const float* beta, const float* mean, const float* var,
                   float eps, float* Wf, float* bf, int N, int K, cudaStream_t s) {
  fold_bn_kernel<<<(unsigned)ceil_div((int64_t)N * K, 256), 256, 0, s>>>(W, b, g, beta, mean, var, eps, Wf, bf, N, K);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

__global__ void to_bf16_kernel(const float* src, __nv_bfloat16* dst, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __float2bfloat16_rn(src[i]);
}
int launch_to_bf16(const float* src, __nv_bfloat16* dst, int64_t n, cudaStream_t s) {
  if (n == 0) return MPL_OK;
  to_bf16_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(src, dst, n);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}
__global__ void to_f16_kernel(const float* src, __half* dst, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __float2half_rn(src[i]);
}
int launch_to_f16(const float* src, void* dst, int64_t n, cudaStream_t s) {
  if (n == 0) return MPL_OK;
  to_f16_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(src, reinterpret_cast<__half*>(dst), n);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}
template <typename T>
__global__ void to_half_rows_kernel(const float* __restrict__ src, T* __restrict__ dst, int N, int K, const int* __restrict__ perm) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)N * K) return;
  const int n = (int)(i / K), k = (int)(i - (int64_t)n * K);
  const float v = src[(int64_t)perm[n] * K + k];
  if constexpr (sizeof(T) == 2 && std::is_same<T, __half>::value) dst[i] = __float2half_rn(v);
  else dst[i] = __float2bfloat16_rn(v);
}
int launch_to_half_rows(const float* src, void* dst, int N, int K, const int* perm, int fp16, cudaStream_t s) {
  const int64_t n = (int64_t)N * K;
  if (n == 0) return MPL_OK;
  if (fp16) to_half_rows_kernel<__half><<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(src, reinterpret_cast<__half*>(dst), N, K, perm);
  else to_half_rows_kernel<__nv_bfloat16><<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), N, K, perm);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}
__global__ void gather_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, int n, const int* __restrict__ perm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[perm[i]];
}
int launch_gather_f32(const float* src, float* dst, int n, const int* perm, cudaStream_t s) {
  if (n == 0) return MPL_OK;
  gather_f32_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(src, dst, n, perm);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}
__global__ void join_planes_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo,
                                   float* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(hi[i]) + __bfloat162float(lo[i]);
}
int launch_join_planes(const __nv_bfloat16* hi, const __nv_bfloat16* lo, float* out, int64_t n, cudaStream_t s) {
  if (n == 0) return MPL_OK;
  join_planes_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(hi, lo, out, n);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}
__global__ void to_split_kernel(const float* src, __nv_bfloat16* dst, int64_t n, int64_t plane) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) store_split1(dst + i, plane, src[i]);
}
int launch_to_split(const float* src, __nv_bfloat16* dst, int64_t n, int64_t plane, cudaStream_t s) {
  if (n == 0) return MPL_OK;
  to_split_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(src, dst, n, plane);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

}  // namespace mpl
