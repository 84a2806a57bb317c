// K6: MPJPE accumulators (evaluate.py:91-125 + function_mpl.py:674-687), P-MPJPE accumulators (pose_utils.py:61-143)
// and the batched input builder
// (joints_dataset_mpl.py:615-648,701-715,762-772,817-820,872-904).  Both are HBM-bound streaming kernels.  Also the linear
// multi-view triangulation of the same raw detections (multiviews/triangulate.py:59-115), the lifter's baseline, its
// outlier-robust counterpart (pair RANSAC + weighted refit), the synthetic projector, a detector-error model for its
// pixels and a generator of random camera setups (the last three have no reference counterpart).  Every kernel that reads
// calibrations is instantiated twice: one [V, 18] block for the batch (kPerPose = false) or one per pose (true).
#include "kernels.cuh"
#include "shared.cuh"
#include "so3.cuh"

namespace mpl {

// acc layout (doubles), L = MPL_METRIC_ACC_LEN(J) = 11 J + 1:
//   [0,J)      sum_b sqrt(nansum_k d^2)  absolute
//   [J,2J)     same, root-relative (a masked root coordinate blanks that coordinate of the whole pose, as the double
//              root-centring of evaluate() + calc_mpjpe(mode='relative') does with NaNs)
//   [2J,5J)    sum_b |d| per joint-dim over unmasked entries, absolute
//   [5J,8J)    same, root-relative
//   [8J,11J)   unmasked count per joint-dim
//   [11J]      pose count
// room: the un-scaling validate() applies to predictions and targets of room-normalised datasets before storing them
// (function_mpl.py:476-488): v * scale + centre per coordinate, in fp32 like the numpy arrays it works on (identity when unused)
struct RoomAffine {
  float scale[3], offset[3];
  int live;
};

// kGrouped (mpl_mpjpe_accumulate_grouped): acc is [G][L] and pose b adds into block group[b] (nothing when it is outside
// [0, G)).  Every lane of a warp works on the same pose, so the group is warp-uniform: the register partials are kept while
// consecutive poses of the warp share a group and flushed into that group's block when it changes.  They go to a shared
// copy of the G L block sums when ssum != 0 (flushed to acc at the end like the ungrouped kernel's), else straight to acc.
template <bool kGrouped>
__global__ void __launch_bounds__(256) mpjpe_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                    const float* __restrict__ conf, int64_t B, int J, float unit,
                                                    const RoomAffine room, double* __restrict__ acc,
                                                    const int32_t* __restrict__ group, int G, int ssum) {
  extern __shared__ double sacc[];  // 11 J + 1; kGrouped: G (11 J + 1) when ssum, else unused
  const int L = 11 * J + 1;
  const int nsh = kGrouped ? (ssum ? G * L : 0) : L;
  double* const dst = kGrouped && !ssum ? acc : sacc;
  for (int i = threadIdx.x; i < nsh; i += blockDim.x) sacc[i] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const int64_t warp_global = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  const int64_t warp_stride = (int64_t)gridDim.x * warps_per_block;
  for (int j0 = 0; j0 < J; j0 += 32) {
    const int j = j0 + lane;
    const bool live = j < J;
    double a_abs = 0, a_rel = 0, d_abs[3] = {0, 0, 0}, d_rel[3] = {0, 0, 0}, cnt[3] = {0, 0, 0}, poses = 0;
    int cur = -1;                                          // kGrouped: group of the partials
    auto flush = [&](double* blk) {
      atomicAdd(&blk[j], a_abs);
      atomicAdd(&blk[J + j], a_rel);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        atomicAdd(&blk[2 * J + j * 3 + k], d_abs[k]);
        atomicAdd(&blk[5 * J + j * 3 + k], d_rel[k]);
        atomicAdd(&blk[8 * J + j * 3 + k], cnt[k]);
      }
    };
    for (int64_t b = warp_global; b < B; b += warp_stride) {
      if (!live) continue;
      if (kGrouped) {
        const int g = group == nullptr ? 0 : group[b];
        if (g != cur) {
          if (cur >= 0) {
            flush(dst + (size_t)cur * L);
            if (j == 0) atomicAdd(&dst[(size_t)cur * L + L - 1], poses);
            a_abs = a_rel = poses = 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k) d_abs[k] = d_rel[k] = cnt[k] = 0.0;
          }
          cur = g >= 0 && g < G ? g : -1;
        }
        if (cur < 0) continue;
        poses += 1.0;
      }
      const float* p = pred + (b * J + j) * 3;
      const float* g = gt + (b * J + j) * 3;
      const float* p0 = pred + b * J * 3;
      const float* g0 = gt + b * J * 3;
      double sa = 0.0, sr = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const bool ok = conf == nullptr || conf[(b * J + j) * 3 + k] > 0.f;
        const bool root_ok = conf == nullptr || conf[b * J * 3 + k] > 0.f;
        float pf = p[k], gf = g[k], p0f = p0[k], g0f = g0[k];
        if (room.live) {
          pf = __fadd_rn(__fmul_rn(pf, room.scale[k]), room.offset[k]);
          gf = __fadd_rn(__fmul_rn(gf, room.scale[k]), room.offset[k]);
          p0f = __fadd_rn(__fmul_rn(p0f, room.scale[k]), room.offset[k]);
          g0f = __fadd_rn(__fmul_rn(g0f, room.scale[k]), room.offset[k]);
        }
        const double pk = (double)pf * unit, gk = (double)gf * unit;
        const double da = pk - gk;
        const double dr = (pk - (double)p0f * unit) - (gk - (double)g0f * unit);
        if (ok) {
          sa = fma(da, da, sa);
          d_abs[k] += fabs(da);
          d_rel[k] += fabs(dr);
          cnt[k] += 1.0;
          if (root_ok) sr = fma(dr, dr, sr);
        }
      }
      a_abs += sqrt(sa);
      a_rel += sqrt(sr);
    }
    if (kGrouped) {
      if (cur >= 0) {
        flush(dst + (size_t)cur * L);
        if (j == 0) atomicAdd(&dst[(size_t)cur * L + L - 1], poses);
      }
    } else if (live) {
      flush(sacc);
    }
  }
  __syncthreads();
  if (kGrouped) {
    for (int i = threadIdx.x; i < nsh; i += blockDim.x)
      if (sacc[i] != 0.0) atomicAdd(&acc[i], sacc[i]);
  } else {
    for (int i = threadIdx.x; i < L - 1; i += blockDim.x)
      if (sacc[i] != 0.0) atomicAdd(&acc[i], sacc[i]);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&acc[L - 1], (double)B);
  }
}

int launch_mpjpe_accumulate(const float* pred, const float* gt, const float* conf3d, const int32_t* group, int G, int64_t B,
                            int J, float unit_scale, const float* room_affine, double* acc, cudaStream_t s) {
  if (B == 0) return MPL_OK;
  RoomAffine room{};
  if (room_affine != nullptr) {
    for (int k = 0; k < 3; ++k) { room.scale[k] = room_affine[k]; room.offset[k] = room_affine[3 + k]; }
    room.live = 1;
  }
  const int64_t want = ceil_div(B, 8 * 16);  // 8 warps per block, ~16 poses per warp
  const unsigned grid = (unsigned)(want < 1 ? 1 : (want > 8 * kNumSMs ? 8 * kNumSMs : want));
  if (G == 0) {
    mpjpe_kernel<false><<<grid, 256, (size_t)(11 * J + 1) * sizeof(double), s>>>(pred, gt, conf3d, B, J, unit_scale, room,
                                                                                 acc, nullptr, 0, 0);
  } else {
    // the G blocks go to shared memory when they fit what a block may opt into, else the flushes are global atomics
    const size_t bytes = (size_t)G * (11 * J + 1) * sizeof(double);
    int dev = 0, optin = 48 * 1024;
    MPL_CUDA(cudaGetDevice(&dev));
    MPL_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const bool ssum = bytes <= (size_t)optin;
    if (ssum && bytes > 48 * 1024)
      MPL_CUDA(cudaFuncSetAttribute(mpjpe_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    mpjpe_kernel<true><<<grid, 256, ssum ? bytes : 0, s>>>(pred, gt, conf3d, B, J, unit_scale, room, acc, group, G, (int)ssum);
  }
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- P-MPJPE: Procrustes-aligned error (pose_utils.py:61-143) -----------------------------------------------------
// One thread per pose, fp64 throughout; a tile of poses is staged through shared memory with coalesced loads (a pose
// is 3 J consecutive floats, so per-thread global reads would be strided).  Per pose, with A = gt, B = pred (x unit):
// centre both, normalise by their Frobenius norms, M = A0^T B0 (3x3) = U S V^T, R = V U^T, optional reflection rule
// on the smallest singular value, then Z = a_norm * tr(S) * B0 R + mean(A) (scaling) or b_norm * B0 R + mean(A).
// acc layout (doubles), L = MPL_PMETRIC_ACC_LEN(J) = J + 3:
//   [0,J) sum_b ||Z_j - A_j||;  [J] sum_b d (normalised residual);  [J+1] sum_b scale;  [J+2] pose count

// One-sided Jacobi on the columns of G (3x3): on return G = U diag(sigma) with orthogonal columns and the rotations
// accumulated in V, i.e. M = U diag(sigma) V^T.  Unordered sigma >= 0.
__device__ __forceinline__ void svd3_one_sided(double (&G)[3][3], double (&V)[3][3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) V[i][k] = i == k ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 12; ++sweep) {              // converges in <= 4 sweeps in practice
    bool rotated = false;
#pragma unroll
    for (int pq = 0; pq < 3; ++pq) {
      const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
      double alpha = 0, beta = 0, gamma = 0;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        alpha = fma(G[i][p], G[i][p], alpha);
        beta = fma(G[i][q], G[i][q], beta);
        gamma = fma(G[i][p], G[i][q], gamma);
      }
      if (gamma * gamma <= 1e-30 * alpha * beta) continue;   // columns orthogonal to 1e-15 relative
      rotated = true;
      const double zeta = (beta - alpha) / (2.0 * gamma);
      const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
      const double c = rsqrt(1.0 + t * t), sn = c * t;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const double gp = G[i][p], gq = G[i][q];
        G[i][p] = c * gp - sn * gq;
        G[i][q] = sn * gp + c * gq;
        const double vp = V[i][p], vq = V[i][q];
        V[i][p] = c * vp - sn * vq;
        V[i][q] = sn * vp + c * vq;
      }
    }
    if (!rotated) break;
  }
}

// Procrustes of one pose over the joints j with use(j), n of them: on return Z_j = zs * (B_j - bm) R + am, with d and scale.
// kMasked (mpl_pmpjpe_accumulate_masked) returns false for a skipped pose: n < 3, or a centred sum of squares not > 0.  With
// every joint used its arithmetic is the unmasked one in the same order (n = J).  kMasked also finds imin / imax and
// completes U without run-time indices into sig / U, which would put them in a stack frame; the unmasked kernel keeps its
// original form, the same arithmetic.
template <bool kMasked, typename Use>
__device__ __forceinline__ bool procrustes_pose(const float* p, const float* g, int J, int n, double u, int scaling,
                                                int reflection, Use use, double (&am)[3], double (&bm)[3], double (&R)[3][3],
                                                double& zs, double& d, double& scale) {
  if constexpr (kMasked) if (n < 3) return false;
  for (int j = 0; j < J; ++j) {
    if (!use(j)) continue;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      am[k] += (double)g[j * 3 + k] * u;
      bm[k] += (double)p[j * 3 + k] * u;
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    am[k] /= (double)n;
    bm[k] /= (double)n;
  }
  double ssx = 0, ssy = 0, G[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}}, V[3][3];
  for (int j = 0; j < J; ++j) {
    if (!use(j)) continue;
    double a0[3], c0[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      a0[k] = (double)g[j * 3 + k] * u - am[k];
      c0[k] = (double)p[j * 3 + k] * u - bm[k];
      ssx = fma(a0[k], a0[k], ssx);
      ssy = fma(c0[k], c0[k], ssy);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int k = 0; k < 3; ++k) G[i][k] = fma(a0[i], c0[k], G[i][k]);
  }
  if constexpr (kMasked) if (!(ssx > 0.0 && ssy > 0.0)) return false;
  const double a_norm = sqrt(ssx), b_norm = sqrt(ssy), inv = 1.0 / (a_norm * b_norm);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) G[i][k] *= inv;
  svd3_one_sided(G, V);
  double sig[3], U[3][3];
  int imin = 0, imax = 0;
  double smax = 0.0;
  if constexpr (kMasked) {
    double smin = 0.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      sig[c] = sqrt(G[0][c] * G[0][c] + G[1][c] * G[1][c] + G[2][c] * G[2][c]);
      if (c == 0) smin = smax = sig[0];
      if (sig[c] < smin) { imin = c; smin = sig[c]; }
      if (sig[c] > smax) { imax = c; smax = sig[c]; }
    }
  } else {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      sig[c] = sqrt(G[0][c] * G[0][c] + G[1][c] * G[1][c] + G[2][c] * G[2][c]);
      if (sig[c] < sig[imin]) imin = c;
      if (sig[c] > sig[imax]) imax = c;
    }
  }
  // left vectors; a vanishing singular value (planar / collinear prediction) gets the completion of the others
  const double tiny = 1e-14 * (kMasked ? smax : sig[imax]);
  int n_ok = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const bool ok = sig[c] > tiny;
    n_ok += ok;
#pragma unroll
    for (int i = 0; i < 3; ++i) U[i][c] = ok ? G[i][c] / sig[c] : 0.0;
  }
  if (n_ok == 2) {
    if constexpr (kMasked) {
#pragma unroll
      for (int c = 0; c < 3; ++c)
        if (c == imin) {
          const int a = (c + 1) % 3, b = (c + 2) % 3;
          U[0][c] = U[1][a] * U[2][b] - U[2][a] * U[1][b];
          U[1][c] = U[2][a] * U[0][b] - U[0][a] * U[2][b];
          U[2][c] = U[0][a] * U[1][b] - U[1][a] * U[0][b];
        }
    } else {
      const int c = imin, a = (c + 1) % 3, b = (c + 2) % 3;
      U[0][c] = U[1][a] * U[2][b] - U[2][a] * U[1][b];
      U[1][c] = U[2][a] * U[0][b] - U[0][a] * U[2][b];
      U[2][c] = U[0][a] * U[1][b] - U[1][a] * U[0][b];
    }
  }
  if (reflection >= 0) {                                  // :112-120, det(R) = det(V) det(U)
    double detR;
    {
      double Rt[3][3];
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) Rt[a][b] = V[a][0] * U[b][0] + V[a][1] * U[b][1] + V[a][2] * U[b][2];
      detR = Rt[0][0] * (Rt[1][1] * Rt[2][2] - Rt[1][2] * Rt[2][1]) - Rt[0][1] * (Rt[1][0] * Rt[2][2] - Rt[1][2] * Rt[2][0]) +
             Rt[0][2] * (Rt[1][0] * Rt[2][1] - Rt[1][1] * Rt[2][0]);
    }
    if ((reflection != 0) != (detR < 0.0)) {
#pragma unroll
      for (int c = 0; c < 3; ++c)
        if (c == imin) {
          V[0][c] = -V[0][c];
          V[1][c] = -V[1][c];
          V[2][c] = -V[2][c];
          sig[c] = -sig[c];
        }
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) R[a][b] = V[a][0] * U[b][0] + V[a][1] * U[b][1] + V[a][2] * U[b][2];
  const double s_trace = sig[0] + sig[1] + sig[2];
  if (scaling) {
    scale = s_trace * a_norm / b_norm;
    d = 1.0 - s_trace * s_trace;
    zs = scale;                                           // a_norm * s_trace * (B0 / b_norm)
  } else {
    scale = 1.0;
    d = 1.0 + ssy / ssx - 2.0 * s_trace * b_norm / a_norm;
    zs = 1.0;                                             // b_norm * (B0 / b_norm)
  }
  return true;
}

// x summed over the lanes of `peers` (the lanes holding the same group), valid in the lowest lane of the set.  A log-step
// tree over each set's members; every lane of the warp must call it.
__device__ __forceinline__ double reduce_peers(unsigned peers, double x) {
  const int lane = threadIdx.x & 31;
  unsigned rel = __popc(peers & ((1u << lane) - 1u));    // my rank within the set
  unsigned above = peers & (0xfffffffeu << lane);
  while (__any_sync(0xffffffffu, above != 0u)) {
    const int next = __ffs(above);
    const double t = __shfl_sync(0xffffffffu, x, next > 0 ? next - 1 : lane);
    if (next > 0) x += t;
    above &= __ballot_sync(0xffffffffu, (rel & 1u) == 0u);
    rel >>= 1;
  }
  return x;
}

// kMasked (mpl_pmpjpe_accumulate_masked): the mask tile [tile][J] is staged with the poses, joint j of a pose is used iff its
// mask is > 0 (or mask is null) and its six coordinates are finite, and pose b adds into block group[b] of the
// MPL_PMETRIC_MASKED_ACC_LEN(J) layout.  Lanes of a warp may hold different groups: each set of lanes with the same group
// (__match_any_sync) is reduced and its lowest lane adds into acc.  The unmasked kernel keeps one shared block sum.
template <bool kMasked>
__global__ void __launch_bounds__(64) pmpjpe_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                    int64_t B, int J, float unit, int scaling, int reflection,
                                                    double* __restrict__ acc, const float* __restrict__ mask,
                                                    const int32_t* __restrict__ group, int G) {
  extern __shared__ __align__(16) unsigned char psm[];
  const int tile = blockDim.x, row = 3 * J;
  double* sacc = reinterpret_cast<double*>(psm);                       // J + 3 (unmasked only)
  float* sp = reinterpret_cast<float*>(sacc + (kMasked ? 0 : (J + 3 + 1) / 2 * 2));   // [tile][3 J]
  float* sg = sp + (size_t)tile * row;
  float* sm = sg + (size_t)tile * row;                                 // kMasked: [tile][J]
  if (!kMasked)
    for (int i = threadIdx.x; i < J + 3; i += blockDim.x) sacc[i] = 0.0;
  const int64_t n_tiles = (B + tile - 1) / tile;
  for (int64_t tl = blockIdx.x; tl < n_tiles; tl += gridDim.x) {
    const int64_t b0 = tl * tile;
    const int n = (int)(B - b0 < tile ? B - b0 : tile);
    __syncthreads();
    for (int i = threadIdx.x; i < n * row; i += blockDim.x) {
      sp[i] = pred[b0 * row + i];
      sg[i] = gt[b0 * row + i];
    }
    if (kMasked && mask != nullptr)
      for (int i = threadIdx.x; i < n * J; i += blockDim.x) sm[i] = mask[b0 * J + i];
    __syncthreads();
    const bool live = (int)threadIdx.x < n;
    const float* p = sp + (size_t)threadIdx.x * row;
    const float* g = sg + (size_t)threadIdx.x * row;
    const float* m = sm + (size_t)threadIdx.x * J;
    const double u = (double)unit;
    auto use = [&](int j) {
      if (!kMasked) return true;
      return (mask == nullptr || m[j] > 0.f) && isfinite(p[j * 3]) && isfinite(p[j * 3 + 1]) && isfinite(p[j * 3 + 2]) &&
             isfinite(g[j * 3]) && isfinite(g[j * 3 + 1]) && isfinite(g[j * 3 + 2]);
    };
    // kMasked: gid = the pose's block, or -1 when it adds nothing (a dead lane, or a group outside [0, G))
    int gid = 0, nu = J;
    if (kMasked) {
      gid = live ? (group == nullptr ? 0 : group[b0 + threadIdx.x]) : -1;
      if (gid >= G) gid = -1;
      nu = 0;
      if (gid >= 0)
        for (int j = 0; j < J; ++j) nu += use(j);
    }
    double am[3] = {0, 0, 0}, bm[3] = {0, 0, 0}, R[3][3], zs = 0.0, d = 0.0, scale = 0.0;
    bool aligned = false;
    if (kMasked ? gid >= 0 : live)
      aligned = procrustes_pose<kMasked>(p, g, J, nu, u, scaling, reflection, use, am, bm, R, zs, d, scale);
    const int lane = threadIdx.x & 31;
    const unsigned peers = kMasked ? __match_any_sync(0xffffffffu, gid) : 0xffffffffu;
    const bool leader = kMasked ? gid >= 0 && lane == __ffs(peers) - 1 : lane == 0;
    double* blk = kMasked ? acc + (size_t)(gid < 0 ? 0 : gid) * (2 * J + 4) : sacc;
    for (int j = 0; j < J; ++j) {
      double e = 0.0;
      const bool on = kMasked ? aligned && use(j) : live;
      if (on) {
        double c0[3], acc2 = 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) c0[k] = (double)p[j * 3 + k] * u - bm[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double z = zs * (c0[0] * R[0][k] + c0[1] * R[1][k] + c0[2] * R[2][k]) + am[k];
          const double df = z - (double)g[j * 3 + k] * u;
          acc2 = fma(df, df, acc2);
        }
        e = sqrt(acc2);
      }
      if (kMasked) {
        e = reduce_peers(peers, e);
        const int cnt = __popc(__ballot_sync(0xffffffffu, on) & peers);
        if (leader && cnt > 0) {
          atomicAdd(&blk[j], e);
          atomicAdd(&blk[J + j], (double)cnt);
        }
      } else {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
        if (lane == 0) atomicAdd(&sacc[j], e);
      }
    }
    if (kMasked) {
      const double sd = reduce_peers(peers, aligned ? d : 0.0), ssc = reduce_peers(peers, aligned ? scale : 0.0);
      const int na = __popc(__ballot_sync(0xffffffffu, aligned) & peers);
      const int ns = __popc(__ballot_sync(0xffffffffu, gid >= 0 && !aligned) & peers);
      if (leader) {
        if (na > 0) {
          atomicAdd(&blk[2 * J], sd);
          atomicAdd(&blk[2 * J + 1], ssc);
          atomicAdd(&blk[2 * J + 2], (double)na);
        }
        if (ns > 0) atomicAdd(&blk[2 * J + 3], (double)ns);
      }
    } else {
      double sd = live ? d : 0.0, ssc = live ? scale : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sd += __shfl_xor_sync(0xffffffffu, sd, o);
        ssc += __shfl_xor_sync(0xffffffffu, ssc, o);
      }
      if (lane == 0) {
        atomicAdd(&sacc[J], sd);
        atomicAdd(&sacc[J + 1], ssc);
      }
    }
  }
  if (!kMasked) {
    __syncthreads();
    for (int i = threadIdx.x; i < J + 2; i += blockDim.x) atomicAdd(&acc[i], sacc[i]);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&acc[J + 2], (double)B);
  }
}

// mask == nullptr and G == 0: mpl_pmpjpe_accumulate; G >= 1: mpl_pmpjpe_accumulate_masked (mask may still be null)
int launch_pmpjpe_accumulate(const float* pred, const float* gt, const float* mask, const int32_t* group, int G, int64_t B,
                             int J, float unit_scale, int scaling, int reflection, double* acc, cudaStream_t s) {
  if (B == 0) return MPL_OK;
  const bool masked = G > 0;
  int tile = 64;
  auto smem = [&](int t) {
    return masked ? (size_t)t * 7 * J * sizeof(float)
                  : (size_t)((J + 3 + 1) / 2 * 2) * sizeof(double) + (size_t)2 * t * 3 * J * sizeof(float);
  };
  if (smem(tile) > 48 * 1024) tile = 32;
  if (smem(tile) > 48 * 1024) {
    set_error("%s: num_joints too large for the shared-memory pose tile",
              masked ? "mpl_pmpjpe_accumulate_masked" : "mpl_pmpjpe_accumulate");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  const int64_t n_tiles = ceil_div(B, (int64_t)tile);
  const unsigned grid = (unsigned)(n_tiles > 16 * kNumSMs ? 16 * kNumSMs : n_tiles);
  if (masked)
    pmpjpe_kernel<true><<<grid, tile, smem(tile), s>>>(pred, gt, B, J, unit_scale, scaling, reflection, acc, mask, group, G);
  else
    pmpjpe_kernel<false><<<grid, tile, smem(tile), s>>>(pred, gt, B, J, unit_scale, scaling, reflection, acc, nullptr,
                                                        nullptr, 0);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// One thread per (pose, view, joint).  Double arithmetic in the order numpy applies it (the dataset code works in
// float64 and casts to float32 at the end), so results are bit-identical to the reference's per-sample path.
// kPerPose: pose b reads its calibration at calib + b * cstride; otherwise every pose reads calib [V, 18].
template <bool kPerPose>
__global__ void __launch_bounds__(256) build_inputs_kernel(const float* __restrict__ pix, const double* __restrict__ calib,
                                                           int64_t cstride, int64_t B, int V, int J, float* __restrict__ poses,
                                                           float* __restrict__ rays, float* __restrict__ centers) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = B * V * J;
  if (idx >= total) return;
  const int j = (int)(idx % J);
  const int v = (int)((idx / J) % V);
  const double* c = (kPerPose ? calib + idx / ((int64_t)V * J) * cstride : calib) + v * 18;
  const double w = c[16], h = c[17];
  double u = pix[idx * 3], vv = pix[idx * 3 + 1], conf = pix[idx * 3 + 2];
  // clip + confidence zeroing (joints_dataset_mpl.py:709-715)
  if (!(0.0 < u)) conf = 0.0;
  if (!(u < w - 1.0)) conf = 0.0;
  if (!(0.0 < vv)) conf = 0.0;
  if (!(vv < h - 1.0)) conf = 0.0;
  u = fmin(fmax(u, 0.0), w - 1.0);
  vv = fmin(fmax(vv, 0.0), h - 1.0);
  // screen normalisation (:817-820) of the joint and of the intrinsics (:615-623)
  const double x = (u / w) * 2.0 - 1.0, y = (vv / w) * 2.0 - h / w;
  const double cx = ((double)c[14] / w) * 2.0 - 1.0, cy = ((double)c[15] / w) * 2.0 - h / w;
  const double fx = (double)c[12] / w * 2.0, fy = (double)c[13] / w * 2.0;
  poses[idx * 3] = (float)x;
  poses[idx * 3 + 1] = (float)y;
  poses[idx * 3 + 2] = (float)conf;
  // rays = R^T [ (x - cx) / fx, (y - cy) / fy, 1 ] + t   (:872-898, USE_T)
  const double dx = (x - cx) / fx, dy = (y - cy) / fy, dz = 1.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double r = (double)c[0 + k] * dx + (double)c[3 + k] * dy + (double)c[6 + k] * dz + (double)c[9 + k];
    rays[idx * 3 + k] = (float)r;
  }
  if (j == 0) {
    const int64_t bv = idx / J;
#pragma unroll
    for (int k = 0; k < 3; ++k) centers[bv * 3 + k] = (float)c[9 + k];
  }
}

// ---- linear multi-view triangulation (MPL/lib/multiviews/triangulate.py:59-115, pymvg find3d) -----------------------
// One thread per (pose, joint), fp64 throughout.  View v takes part iff conf > min_conf and the pixel lies strictly inside
// the image, the comparisons build_inputs_kernel makes.  Each used view adds the two pixel-space rows u P3 - P1 and
// v P3 - P2 of the DLT system A X~ = 0 (Hartley & Zisserman section 12.2) into the 4x4 Gram matrix A^T A, so A is never
// stored; the right singular vector of A's smallest singular value is the eigenvector of A^T A's smallest eigenvalue,
// found with cyclic Jacobi.  Fewer than two used views leave the point undetermined: NaN.
// A block stages the pixels of its kTriTile (pose, joint) items for every view through shared memory: for a fixed view the
// items of one pose are consecutive floats, so the copy is coalesced where per-thread reads would be 12-byte strided.
constexpr int kTriTile = 128;

// Cyclic Jacobi on the symmetric 4x4 S (upper triangle used): on return diag(S) holds the eigenvalues and the columns of
// V the eigenvectors.  A pair is skipped once |S_pq| <= 1e-15 sqrt|S_pp S_qq|, the rule of svd3_one_sided.
__device__ __forceinline__ void eig4_jacobi(double (&S)[4][4], double (&V)[4][4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int k = 0; k < 4; ++k) V[i][k] = i == k ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 12; ++sweep) {              // <= 7 sweeps on the synthetic rigs with 2 px noise
    bool rotated = false;
#pragma unroll
    for (int pq = 0; pq < 6; ++pq) {
      const int p = pq < 3 ? 0 : (pq < 5 ? 1 : 2);
      const int q = pq < 3 ? pq + 1 : (pq < 5 ? pq - 1 : 3);
      const double g = S[p][q];
      if (g * g <= 1e-30 * fabs(S[p][p] * S[q][q])) continue;
      rotated = true;
      const double zeta = (S[q][q] - S[p][p]) / (2.0 * g);
      const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
      const double c = rsqrt(1.0 + t * t), sn = c * t;
      S[p][p] -= t * g;
      S[q][q] += t * g;
      S[p][q] = 0.0;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        if (r == p || r == q) continue;
        double& srp = r < p ? S[r][p] : S[p][r];
        double& srq = r < q ? S[r][q] : S[q][r];
        const double a = srp, b = srq;
        srp = c * a - sn * b;
        srq = sn * a + c * b;
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const double a = V[r][p], b = V[r][q];
        V[r][p] = c * a - sn * b;
        V[r][q] = sn * a + c * b;
      }
    }
    if (!rotated) break;
  }
}

// P = K [R | -R t] (row-major 3x4) and (w, h) of one [18] calibration row.
__device__ __forceinline__ void tri_camera(const double* __restrict__ c, double (&P)[12], double (&wh)[2]) {
  const double fx = c[12], fy = c[13], cx = c[14], cy = c[15];
  double Rt[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) Rt[r] = c[3 * r] * c[9] + c[3 * r + 1] * c[10] + c[3 * r + 2] * c[11];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    P[k] = fx * c[k] + cx * c[6 + k];
    P[4 + k] = fy * c[3 + k] + cy * c[6 + k];
    P[8 + k] = c[6 + k];
  }
  P[3] = -(fx * Rt[0] + cx * Rt[2]);
  P[7] = -(fy * Rt[1] + cy * Rt[2]);
  P[11] = -Rt[2];
  wh[0] = c[16];
  wh[1] = c[17];
}

// Per-pose calibrations (kPerPose): a tile of T consecutive items spans at most (J + T - 2) / J + 1 poses, and each needs
// its own V projection matrices, so they go to a dynamic shared-memory table [poses][V] of P (12 doubles), then one of
// (w, h), next to the static pixel tile.  The launch picks the largest T <= kTriTile whose table fits the 48 KB a block
// gets without opting in (tri_pose_tile): T = kTriTile for J = 17 and every V <= 16, T = 12 for J = 1 and V = 16.
constexpr int kTriStaticSmem = kMaxViews * (12 + 2) * 8 + kMaxViews * 3 * kTriTile * 4;   // sP, sWH, sx
__host__ __device__ __forceinline__ int tri_tile_poses(int T, int J) { return (J + T - 2) / J + 1; }

// Stages a block's tile of T (pose, joint) items: P_v = K_v [R_v | -R_v t_v] (row-major 3x4) and (w, h) per view, and per
// view the (u, v, conf) of the tile's items.  T = kTriTile with one calibration [V, 18] for the whole batch; with per-pose
// calibrations T = blockDim.x and pose b's are at calib + b * cstride.  Sets i0 to the tile's first item (item i = (pose i / J,
// joint i % J)), P / WH to the V cameras of this thread's pose, and returns the number of items in the tile.  Every thread
// of the block must call it (it ends with a barrier).
template <bool kPerPose>
__device__ __forceinline__ int tri_stage_tile(const float* __restrict__ pix, const double* __restrict__ calib, int64_t cstride,
                                              int64_t B, int V, int J, double (&sP)[kMaxViews][12],
                                              double (&sWH)[kMaxViews][2], float (&sx)[kMaxViews][3 * kTriTile], int64_t& i0,
                                              const double (*&P)[12], const double (*&WH)[2]) {
  const int tid = threadIdx.x;
  if (!kPerPose && tid < V) tri_camera(calib + tid * 18, sP[tid], sWH[tid]);
  const int T = kPerPose ? (int)blockDim.x : kTriTile;
  i0 = (int64_t)blockIdx.x * T;
  const int n = (int)(B * J - i0 < T ? B * J - i0 : T);
  const int row = 3 * n;
  // float f of the tile in view v is coordinate f % 3 of item i0 + f / 3 = (pose b0 + jj / J, joint jj % J), jj = j0 + f / 3
  const int64_t b0 = i0 / J;
  const int j0 = (int)(i0 - b0 * J);
  if (kPerPose) {
    extern __shared__ double tri_cams[];
    double(*tP)[12] = reinterpret_cast<double(*)[12]>(tri_cams);
    double(*tWH)[2] = reinterpret_cast<double(*)[2]>(tri_cams + 12 * tri_tile_poses(T, J) * V);
    const int np = (j0 + n - 1) / J + 1;
    for (int e = tid; e < np * V; e += T) {
      const int p = e / V;
      tri_camera(calib + (b0 + p) * cstride + (e - p * V) * 18, tP[e], tWH[e]);
    }
    P = tP + (j0 + tid) / J * V;
    WH = tWH + (j0 + tid) / J * V;
  } else {
    P = sP;
    WH = sWH;
  }
  for (int e = tid; e < V * row; e += T) {
    const int v = e / row, f = e - v * row;
    const int jj = j0 + f / 3, db = jj / J;
    sx[v][f] = pix[(((b0 + db) * V + v) * J + (jj - db * J)) * 3 + f % 3];
  }
  __syncthreads();
  return n;
}

// Items per block and dynamic shared memory of the per-pose triangulation kernels.
static int tri_pose_tile(int V, int J, size_t& smem) {
  auto bytes = [&](int t) { return (size_t)tri_tile_poses(t, J) * V * (12 + 2) * sizeof(double); };
  int T = kTriTile;
  while (T > 1 && bytes(T) > (size_t)(48 * 1024 - kTriStaticSmem)) T -= T > 32 ? 32 : 1;
  smem = bytes(T);
  return T;
}

// Adds the DLT rows s (u P3 - P1) and s (w P3 - P2) of one view into the Gram matrix G (upper triangle).  s = 1 is an
// exact multiply, so the unweighted sum has the same bits with or without it.
__device__ __forceinline__ void gram_add_view(double (&G)[4][4], const double (&P)[12], double u, double w, double s) {
  double a[4], b[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    a[k] = s * fma(u, P[8 + k], -P[k]);
    b[k] = s * fma(w, P[8 + k], -P[4 + k]);
  }
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int k = r; k < 4; ++k) G[r][k] = fma(a[r], a[k], fma(b[r], b[k], G[r][k]));
}

// x = eigenvector of G's smallest eigenvalue (G is overwritten), i.e. the homogeneous DLT solution.  Compile-time indices
// only, so G and the eigenvectors stay in registers.
__device__ __forceinline__ void gram_null_vector(double (&G)[4][4], double (&x)[4]) {
  double E[4][4];
  eig4_jacobi(G, E);
  double lmin = G[0][0];
#pragma unroll
  for (int k = 0; k < 4; ++k) x[k] = E[k][0];
#pragma unroll
  for (int m = 1; m < 4; ++m)
    if (G[m][m] < lmin) {
      lmin = G[m][m];
#pragma unroll
      for (int k = 0; k < 4; ++k) x[k] = E[k][m];
    }
}

template <bool kPerPose>
__global__ void __launch_bounds__(kTriTile) triangulate_kernel(const float* __restrict__ pix, const double* __restrict__ calib,
                                                               int64_t cstride, int64_t B, int V, int J, float min_conf,
                                                               float* __restrict__ points, int32_t* __restrict__ views_used) {
  __shared__ double sP[kMaxViews][12];
  __shared__ double sWH[kMaxViews][2];
  __shared__ float sx[kMaxViews][3 * kTriTile];
  const int tid = threadIdx.x;
  int64_t i0;
  const double(*P)[12];
  const double(*WH)[2];
  const int n = tri_stage_tile<kPerPose>(pix, calib, cstride, B, V, J, sP, sWH, sx, i0, P, WH);
  if (tid >= n) return;
  // Gram matrix A^T A, upper triangle
  double G[4][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
  int used = 0;
  for (int v = 0; v < V; ++v) {
    const double u = sx[v][3 * tid], w = sx[v][3 * tid + 1];
    if (!tri_candidate(sx[v][3 * tid + 2], u, w, min_conf, WH[v])) continue;
    ++used;
    gram_add_view(G, P[v], u, w, 1.0);
  }
  const int64_t i = i0 + tid;
  float out[3] = {__int_as_float(0x7fc00000), __int_as_float(0x7fc00000), __int_as_float(0x7fc00000)};
  if (used >= 2) {
    double x[4];
    gram_null_vector(G, x);
#pragma unroll
    for (int k = 0; k < 3; ++k) out[k] = (float)(x[k] / x[3]);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) points[i * 3 + k] = out[k];
  views_used[i] = used;
}

int launch_triangulate(const float* pix, const double* calib, int64_t calib_stride, int64_t B, int V, int J, float min_conf,
                       float* points, int32_t* views_used, cudaStream_t s) {
  const int64_t items = B * J;
  if (items == 0) return MPL_OK;
  if (calib_stride == 0) {
    triangulate_kernel<false><<<(unsigned)ceil_div(items, kTriTile), kTriTile, 0, s>>>(pix, calib, 0, B, V, J, min_conf,
                                                                                      points, views_used);
  } else {
    size_t smem;
    const int T = tri_pose_tile(V, J, smem);
    triangulate_kernel<true><<<(unsigned)ceil_div(items, (int64_t)T), T, smem, s>>>(pix, calib, calib_stride, B, V, J,
                                                                                   min_conf, points, views_used);
  }
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- robust multi-view triangulation: exhaustive-pair RANSAC with the MSAC cost, then a confidence-weighted DLT refit --
// Same items, staging and candidate views as triangulate_kernel.  Every candidate pair (a < b, lexicographic) gives one
// hypothesis, the unweighted two-view DLT; its MSAC cost is sum_c min(e_c^2, tau^2) over all candidates c, e_c the pixel
// reprojection error (infinite where the hypothesis lies behind camera c or at infinity).  The cheapest hypothesis wins
// (an exact tie keeps the earlier pair); its inliers are the candidates with e_c < tau, and with at least two of them the
// point is the DLT over the inliers with each view's rows scaled by its confidence.  All pairs are searched -- at most 120
// for V = 16 -- so the result is deterministic and independent of how the batch is split.  Per-view errors are recomputed
// for the inlier mask rather than kept in a dynamically indexed array, which would live in local memory.

// Squared reprojection error (pixels^2) of the homogeneous point x through P at pixel (u, w); +inf where the depth
// (P3 . x) / x_4 is not > 0 or not finite.
__device__ __forceinline__ double reproj_err2(const double (&P)[12], const double (&x)[4], double u, double w) {
  const double z = P[8] * x[0] + P[9] * x[1] + P[10] * x[2] + P[11] * x[3];
  const double depth = z / x[3];
  if (!(depth > 0.0) || isinf(depth)) return __longlong_as_double(0x7ff0000000000000ll);
  const double du = (P[0] * x[0] + P[1] * x[1] + P[2] * x[2] + P[3] * x[3]) / z - u;
  const double dv = (P[4] * x[0] + P[5] * x[1] + P[6] * x[2] + P[7] * x[3]) / z - w;
  return du * du + dv * dv;
}

template <bool kPerPose>
__global__ void __launch_bounds__(kTriTile) triangulate_robust_kernel(const float* __restrict__ pix,
                                                                      const double* __restrict__ calib, int64_t cstride, int64_t B,
                                                                      int V, int J, float min_conf, float inlier_px,
                                                                      float* __restrict__ points,
                                                                      int32_t* __restrict__ inliers) {
  __shared__ double sP[kMaxViews][12];
  __shared__ double sWH[kMaxViews][2];
  __shared__ float sx[kMaxViews][3 * kTriTile];
  const int tid = threadIdx.x;
  int64_t i0;
  const double(*P)[12];
  const double(*WH)[2];
  const int n = tri_stage_tile<kPerPose>(pix, calib, cstride, B, V, J, sP, sWH, sx, i0, P, WH);
  if (tid >= n) return;
  unsigned cand = 0;                                       // bit v: view v is a candidate
  for (int v = 0; v < V; ++v)
    if (tri_candidate(sx[v][3 * tid + 2], sx[v][3 * tid], sx[v][3 * tid + 1], min_conf, WH[v])) cand |= 1u << v;
  const double tau2 = (double)inlier_px * (double)inlier_px;
  unsigned inl = 0;
  float out[3] = {__int_as_float(0x7fc00000), __int_as_float(0x7fc00000), __int_as_float(0x7fc00000)};
  if (__popc(cand) >= 2) {
    double best = __longlong_as_double(0x7ff0000000000000ll), xb[4] = {0.0, 0.0, 0.0, 0.0};
    for (unsigned ma = cand; ma; ma &= ma - 1) {
      const int a = __ffs(ma) - 1;
      for (unsigned mb = ma & (ma - 1); mb; mb &= mb - 1) {
        const int b = __ffs(mb) - 1;
        double G[4][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
        gram_add_view(G, P[a], sx[a][3 * tid], sx[a][3 * tid + 1], 1.0);
        gram_add_view(G, P[b], sx[b][3 * tid], sx[b][3 * tid + 1], 1.0);
        double x[4];
        gram_null_vector(G, x);
        double cost = 0.0;                                 // MSAC; fmin maps an infinite (or NaN) error to tau^2
        for (unsigned mc = cand; mc; mc &= mc - 1) {
          const int c = __ffs(mc) - 1;
          cost += fmin(reproj_err2(P[c], x, sx[c][3 * tid], sx[c][3 * tid + 1]), tau2);
        }
        if (cost < best) {
          best = cost;
#pragma unroll
          for (int k = 0; k < 4; ++k) xb[k] = x[k];
        }
      }
    }
    for (unsigned mc = cand; mc; mc &= mc - 1) {
      const int c = __ffs(mc) - 1;
      if (reproj_err2(P[c], xb, sx[c][3 * tid], sx[c][3 * tid + 1]) < tau2) inl |= 1u << c;
    }
    if (__popc(inl) >= 2) {
      // refit in triangulate_kernel's view order, rows scaled by conf (the ML weighting when the pixel noise is sigma / conf)
      double G[4][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
      for (int v = 0; v < V; ++v)
        if ((inl >> v) & 1u) gram_add_view(G, P[v], sx[v][3 * tid], sx[v][3 * tid + 1], (double)sx[v][3 * tid + 2]);
      double x[4];
      gram_null_vector(G, x);
#pragma unroll
      for (int k = 0; k < 3; ++k) out[k] = (float)(x[k] / x[3]);
    } else {
      inl = 0;
    }
  }
  const int64_t i = i0 + tid;
#pragma unroll
  for (int k = 0; k < 3; ++k) points[i * 3 + k] = out[k];
  inliers[i] = (int32_t)inl;
}

int launch_triangulate_robust(const float* pix, const double* calib, int64_t calib_stride, int64_t B, int V, int J,
                              float min_conf, float inlier_px, float* points, int32_t* inliers, cudaStream_t s) {
  const int64_t items = B * J;
  if (items == 0) return MPL_OK;
  if (calib_stride == 0) {
    triangulate_robust_kernel<false><<<(unsigned)ceil_div(items, kTriTile), kTriTile, 0, s>>>(
        pix, calib, 0, B, V, J, min_conf, inlier_px, points, inliers);
  } else {
    size_t smem;
    const int T = tri_pose_tile(V, J, smem);
    triangulate_robust_kernel<true><<<(unsigned)ceil_div(items, (int64_t)T), T, smem, s>>>(
        pix, calib, calib_stride, B, V, J, min_conf, inlier_px, points, inliers);
  }
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- Levenberg-Marquardt refinement of given points on the confidence-weighted reprojection error ------------------
// Same items, staging and candidate views as triangulate_kernel; the views used are the candidates in the item's
// view_mask.  C(X) = sum_v w_v |pi(P_v [X; 1]) - x_v|^2 with w_v = conf_v^2, the maximum-likelihood cost when the pixel
// noise has std sigma / conf (Hartley & Zisserman section 12.3).  The 3 x 3 normal equations A = sum w D^T D,
// g = sum w D^T r are rebuilt after each accepted step only, (A + mu I) delta = -g is solved by Cholesky, and the step is
// kept iff it lowers C.  The used views are walked with __ffs on a bitmask so that P is indexed by a run-time view in shared
// memory, never in a local array; the thread's pixels stay in the staged tile.

// C(X) over the views of `used`; +inf as soon as a view sees X at a depth that is not > 0 or not finite.
__device__ __forceinline__ double refine_cost(const double (*P)[12], const float (&sx)[kMaxViews][3 * kTriTile], int tid,
                                              unsigned used, const double (&X)[3]) {
  double cost = 0.0;
  for (unsigned m = used; m; m &= m - 1) {
    const int v = __ffs(m) - 1;
    const double* p = P[v];
    const double z = fma(p[8], X[0], fma(p[9], X[1], fma(p[10], X[2], p[11])));
    if (!(z > 0.0) || isinf(z)) return __longlong_as_double(0x7ff0000000000000ll);
    const double iz = 1.0 / z;
    const double du = fma(p[0], X[0], fma(p[1], X[1], fma(p[2], X[2], p[3]))) * iz - (double)sx[v][3 * tid];
    const double dv = fma(p[4], X[0], fma(p[5], X[1], fma(p[6], X[2], p[7]))) * iz - (double)sx[v][3 * tid + 1];
    const double c = (double)sx[v][3 * tid + 2];
    cost = fma(c * c, fma(du, du, dv * dv), cost);
  }
  return cost;
}

template <bool kPerPose>
__global__ void __launch_bounds__(kTriTile) triangulate_refine_kernel(const float* __restrict__ pix,
                                                                      const double* __restrict__ calib, int64_t cstride, int64_t B,
                                                                      int V, int J, float min_conf,
                                                                      const int32_t* __restrict__ view_mask, const float* init,
                                                                      int max_iters, float* points, float* __restrict__ reproj_px) {
  __shared__ double sP[kMaxViews][12];
  __shared__ double sWH[kMaxViews][2];
  __shared__ float sx[kMaxViews][3 * kTriTile];
  const int tid = threadIdx.x;
  int64_t i0;
  const double(*P)[12];
  const double(*WH)[2];
  const int n = tri_stage_tile<kPerPose>(pix, calib, cstride, B, V, J, sP, sWH, sx, i0, P, WH);
  if (tid >= n) return;
  const int64_t i = i0 + tid;
  // init may be points (in-place refinement): every read of init comes before the thread's stores
  float out[3] = {init[i * 3], init[i * 3 + 1], init[i * 3 + 2]};
  unsigned used = 0;
  for (int v = 0; v < V; ++v)
    if (tri_candidate(sx[v][3 * tid + 2], sx[v][3 * tid], sx[v][3 * tid + 1], min_conf, WH[v])) used |= 1u << v;
  if (view_mask != nullptr) used &= (unsigned)view_mask[i];
  double X[3] = {(double)out[0], (double)out[1], (double)out[2]};
  float rp = __int_as_float(0x7fc00000);
  double C = __longlong_as_double(0x7ff0000000000000ll);
  if (isfinite(X[0]) && isfinite(X[1]) && isfinite(X[2]) && __popc(used) >= 2) C = refine_cost(P, sx, tid, used, X);
  if (isfinite(C)) {
    double A[6], g[3], mu = 0.0;                           // A: 00 01 02 11 12 22
    bool relin = true;
    for (int k = 1; k <= max_iters; ++k) {
      if (relin) {
#pragma unroll
        for (int e = 0; e < 6; ++e) A[e] = 0.0;
#pragma unroll
        for (int e = 0; e < 3; ++e) g[e] = 0.0;
        for (unsigned m = used; m; m &= m - 1) {
          const int v = __ffs(m) - 1;
          const double* p = P[v];
          const double iz = 1.0 / fma(p[8], X[0], fma(p[9], X[1], fma(p[10], X[2], p[11])));
          const double qu = fma(p[0], X[0], fma(p[1], X[1], fma(p[2], X[2], p[3]))) * iz;
          const double qv = fma(p[4], X[0], fma(p[5], X[1], fma(p[6], X[2], p[7]))) * iz;
          const double c = (double)sx[v][3 * tid + 2], w = c * c;
          const double ru = qu - (double)sx[v][3 * tid], rv = qv - (double)sx[v][3 * tid + 1];
          double du[3], dv[3];                              // rows of the 2 x 3 Jacobian of pi(P [X; 1])
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            du[a] = fma(-qu, p[8 + a], p[a]) * iz;
            dv[a] = fma(-qv, p[8 + a], p[4 + a]) * iz;
          }
          int e = 0;
#pragma unroll
          for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b, ++e) A[e] = fma(w, fma(du[a], du[b], dv[a] * dv[b]), A[e]);
            g[a] = fma(w, fma(du[a], ru, dv[a] * rv), g[a]);
          }
        }
        if (k == 1) mu = 1e-3 * fmax(A[0], fmax(A[3], A[5]));
        relin = false;
      }
      // Cholesky of A + mu I; a pivot that is not finite and > 0 rejects the step (there is no delta to test)
      const double inf = __longlong_as_double(0x7ff0000000000000ll);
      const double m00 = A[0] + mu;
      if (!(m00 > 0.0 && m00 < inf)) { mu *= 10.0; continue; }
      const double l00 = sqrt(m00), l10 = A[1] / l00, l20 = A[2] / l00;
      const double m11 = A[3] + mu - l10 * l10;
      if (!(m11 > 0.0 && m11 < inf)) { mu *= 10.0; continue; }
      const double l11 = sqrt(m11), l21 = (A[4] - l20 * l10) / l11;
      const double m22 = A[5] + mu - l20 * l20 - l21 * l21;
      if (!(m22 > 0.0 && m22 < inf)) { mu *= 10.0; continue; }
      const double l22 = sqrt(m22);
      const double y0 = -g[0] / l00, y1 = (-g[1] - l10 * y0) / l11, y2 = (-g[2] - l20 * y0 - l21 * y1) / l22;
      const double d2 = y2 / l22, d1 = (y1 - l21 * d2) / l11, d0 = (y0 - l10 * d1 - l20 * d2) / l00;
      const double xnorm = sqrt(X[0] * X[0] + X[1] * X[1] + X[2] * X[2]);
      const double dnorm = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
      const double Xn[3] = {X[0] + d0, X[1] + d1, X[2] + d2};
      const double Cn = refine_cost(P, sx, tid, used, Xn);
      if (Cn < C) {
#pragma unroll
        for (int a = 0; a < 3; ++a) X[a] = Xn[a];
        C = Cn;
        mu *= 0.1;
        relin = true;
      } else {
        mu *= 10.0;
      }
      if (dnorm <= 1e-10 * (xnorm + 1e-10)) break;
    }
    double wsum = 0.0;
    for (unsigned m = used; m; m &= m - 1) {
      const double c = (double)sx[__ffs(m) - 1][3 * tid + 2];
      wsum = fma(c, c, wsum);
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) out[a] = (float)X[a];
    rp = (float)sqrt(C / wsum);
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) points[i * 3 + a] = out[a];
  reproj_px[i] = rp;
}

int launch_triangulate_refine(const float* pix, const double* calib, int64_t calib_stride, int64_t B, int V, int J,
                              float min_conf, const int32_t* view_mask, const float* init, int max_iters, float* points,
                              float* reproj_px, cudaStream_t s) {
  const int64_t items = B * J;
  if (items == 0) return MPL_OK;
  if (calib_stride == 0) {
    triangulate_refine_kernel<false><<<(unsigned)ceil_div(items, kTriTile), kTriTile, 0, s>>>(
        pix, calib, 0, B, V, J, min_conf, view_mask, init, max_iters, points, reproj_px);
  } else {
    size_t smem;
    const int T = tri_pose_tile(V, J, smem);
    triangulate_refine_kernel<true><<<(unsigned)ceil_div(items, (int64_t)T), T, smem, s>>>(
        pix, calib, calib_stride, B, V, J, min_conf, view_mask, init, max_iters, points, reproj_px);
  }
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// N3: MHP-style synthetic projector.  3D poses from a counter-based generator keyed by (seed, GLOBAL pose index) --
// any sharding of the index range over ranks / micro-batches yields the same data -- pushed through V calibrations:
// x_cam = R (X - t), u = f x_cam / z + c (MPL/lib/utils/calib.py:42-77).  Emits raw detector-style pixels (u, v, conf)
// for mpl_build_inputs and the 3D target.  The generator is numpy's Philox4x64-10 stream, bit for bit (openmpl_b200/
// synth.py draws the same uniforms on the host), so the device data can be checked against the host generator.
// philox4x64_10, UniformCursor and project_pixel are in shared.cuh (track.cu's mpl_synth_motion uses them too).
// ---------------------------------------------------------------------------------------------------------------------
template <bool kPerPose>
__global__ void __launch_bounds__(128) synth_project_kernel(uint64_t seed, int64_t start, int64_t B, int V, int J,
                                                            const double* __restrict__ calib, int64_t cstride,
                                                            const double* __restrict__ room, int conf_ones,
                                                            float* __restrict__ pix, float* __restrict__ target) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double* cal = kPerPose ? calib + b * cstride : calib;
  const int n = 3 * (J - 1);
  const int per_pose = 3 + 2 * n + V * J;
  const uint64_t blocks = (uint64_t)((per_pose + 3) / 4);
  const uint64_t base = (uint64_t)(start + b) * blocks;
  UniformCursor ca(base, seed), cb(base, seed);
  double root[3];
  root[0] = room[0] + ca.get(0) * (room[1] - room[0]);
  root[1] = room[2] + ca.get(1) * (room[3] - room[2]);
  root[2] = 0.8 + 0.2 * ca.get(2);
  float* tg = target + b * J * 3;
  float* px = pix + b * V * J * 3;
  UniformCursor cc(base, seed);
  for (int j = 0; j < J; ++j) {
    double X[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      X[k] = root[k];
      if (j > 0) {
        const int i = (j - 1) * 3 + k;
        const double u1 = fmax(ca.get(3 + i), 1e-12), u2 = cb.get(3 + n + i);
        X[k] += 0.25 * (sqrt(-2.0 * log(u1)) * cos(2.0 * 3.14159265358979323846 * u2));  // Box-Muller, fixed draw count
      }
      tg[j * 3 + k] = (float)X[k];
    }
    for (int v = 0; v < V; ++v)
      project_pixel(cal + v * 18, X, conf_ones ? 1.0 : 0.3 + 0.7 * cc.get(3 + 2 * n + v * J + j), px + (v * J + j) * 3);
  }
}

int launch_synth_project(uint64_t seed, int64_t start, int64_t B, int V, int J, const double* calib, int64_t calib_stride,
                         const double* room, int conf_ones, float* pix, float* target, cudaStream_t s) {
  if (B == 0) return MPL_OK;
  const unsigned grid = (unsigned)ceil_div(B, 128);
  if (calib_stride == 0)
    synth_project_kernel<false><<<grid, 128, 0, s>>>(seed, start, B, V, J, calib, 0, room, conf_ones, pix, target);
  else
    synth_project_kernel<true><<<grid, 128, 0, s>>>(seed, start, B, V, J, calib, calib_stride, room, conf_ones, pix, target);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- detector-error model on raw pixels: misses, confident false detections, Gaussian noise of std sigma / conf -----------
// One thread per (pose, view, joint) entry of pix [B, V, J, 3], in place; entries with conf == 0 (behind the camera) stay.
// The six uniforms U0..U5 of an entry come from the Philox4x64-10 stream of synth_project_kernel under key (seed, 1), so
// they are independent of the geometry's key (seed, 0): pose i owns counter blocks [i nb, (i + 1) nb), nb = ceil(6 V J / 4),
// and uniform slot (v J + j) 6 + m is U_m.  openmpl_b200/synth.py (detector_noise) draws the same uniforms on the host.
//   U0 < p_miss                       -> conf = 0, pixel kept
//   U0 < p_miss + p_outlier           -> u = U3 (w - 1), v = U4 (h - 1), conf = 0.3 + 0.7 U5
//   otherwise                         -> (u, v) += sigma / conf * r (cos t, sin t), r = sqrt(-2 ln max(U1, 1e-12)), t = 2 pi U2
// fp64 throughout, rounded once to fp32.  The outlier and threshold arithmetic is written with explicit roundings so it
// matches numpy bit for bit.
// Uniforms U0..U5 of record r of pose (start + b) under Philox key (seed, key1), six per record: pose i owns counter blocks
// [i nb, (i + 1) nb), nb = ceil(6 records / 4), and slot 6 r + m is U_m.
__device__ __forceinline__ void six_uniforms(uint64_t seed, uint64_t key1, int64_t start, int64_t b, int records, int r,
                                             double (&U)[6]) {
  const uint64_t base = (uint64_t)(start + b) * (uint64_t)((6 * records + 3) / 4);
  const int s0 = 6 * r;                                    // slot of U0; s0 % 4 is 0 or 2, so U0..U5 span two blocks
  uint64_t lo[4], hi[4];
  philox4x64_10(base + (uint64_t)(s0 >> 2) + 1ull, seed, key1, lo);  // numpy increments the counter before generating
  philox4x64_10(base + (uint64_t)(s0 >> 2) + 2ull, seed, key1, hi);
  const bool al = (s0 & 3) == 0;
  const uint64_t raw[6] = {al ? lo[0] : lo[2], al ? lo[1] : lo[3], al ? lo[2] : hi[0],
                           al ? lo[3] : hi[1], al ? hi[0] : hi[2], al ? hi[1] : hi[3]};
#pragma unroll
  for (int m = 0; m < 6; ++m) U[m] = (double)(raw[m] >> 11) * (1.0 / 9007199254740992.0);
}

template <bool kPerPose>
__global__ void __launch_bounds__(256) detector_noise_kernel(uint64_t seed, int64_t start, int64_t B, int V, int J,
                                                             const double* __restrict__ calib, int64_t cstride, float sigma_px,
                                                             float p_outlier, float p_miss, float* __restrict__ pix) {
  const int per = V * J;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B * per) return;
  float* p = pix + e * 3;
  const float conf = p[2];
  if (conf == 0.0f) return;
  const int64_t b = e / per;
  const int r = (int)(e - b * per);                        // v J + j
  double U[6];
  six_uniforms(seed, 1ull, start, b, per, r, U);
  const double pm = (double)p_miss;
  if (U[0] < pm) {
    p[2] = 0.0f;
    return;
  }
  if (U[0] < __dadd_rn(pm, (double)p_outlier)) {
    const double* c = (kPerPose ? calib + b * cstride : calib) + (r / J) * 18;
    p[0] = (float)__dmul_rn(U[3], c[16] - 1.0);
    p[1] = (float)__dmul_rn(U[4], c[17] - 1.0);
    p[2] = (float)__dadd_rn(0.3, __dmul_rn(0.7, U[5]));
    return;
  }
  const double s = (double)sigma_px / (double)conf * sqrt(-2.0 * log(fmax(U[1], 1e-12)));
  double sn, cs;
  sincospi(2.0 * U[2], &sn, &cs);                          // = sincos(2 pi U2) without sincos's reduction (a stack frame)
  p[0] = (float)((double)p[0] + s * cs);
  p[1] = (float)((double)p[1] + s * sn);
}

int launch_detector_noise(uint64_t seed, int64_t start, int64_t B, int V, int J, const double* calib, int64_t calib_stride,
                          float sigma_px, float p_outlier, float p_miss, float* pix, cudaStream_t s) {
  const int64_t total = B * V * J;
  if (total == 0) return MPL_OK;
  const unsigned grid = (unsigned)ceil_div(total, 256);
  if (calib_stride == 0)
    detector_noise_kernel<false><<<grid, 256, 0, s>>>(seed, start, B, V, J, calib, 0, sigma_px, p_outlier, p_miss, pix);
  else
    detector_noise_kernel<true><<<grid, 256, 0, s>>>(seed, start, B, V, J, calib, calib_stride, sigma_px, p_outlier, p_miss,
                                                     pix);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- lens distortion: OpenCV's 5-coefficient Brown-Conrady model, k = (k1, k2, p1, p2, k3) -------------------------------
// One thread per (pose, view, joint) entry of pix [B, V, J, 3], fp64.  The model, the validity rule and the Newton
// inversion are stated in include/mpl_b200.h; tests/lens_oracle.py and openmpl_b200/synth.py (distort_pixels) restate them
// in numpy.  kPerPose: pose b reads calib + b * cstride and dist + b * dstride (either stride may be 0); otherwise every
// pose reads the [V, 18] / [V, 5] blocks.  pix_in may equal pix_out: a thread reads its whole entry before it writes.
constexpr int kLensMaxIters = 20;

// D(x, y) and its Jacobian [[a, b], [b, d]] (the two off-diagonal derivatives are the same expression).
__device__ __forceinline__ void lens_map(const double (&k)[5], double x, double y, double& xd, double& yd, double& a,
                                         double& b, double& d) {
  const double r2 = x * x + y * y;
  const double rho = 1.0 + r2 * (k[0] + r2 * (k[1] + r2 * k[4]));
  const double drho = k[0] + r2 * (2.0 * k[1] + r2 * (3.0 * k[4]));     // d rho / d r2
  xd = x * rho + 2.0 * k[2] * x * y + k[3] * (r2 + 2.0 * x * x);
  yd = y * rho + k[2] * (r2 + 2.0 * y * y) + 2.0 * k[3] * x * y;
  a = rho + 2.0 * x * x * drho + 2.0 * k[2] * y + 6.0 * k[3] * x;
  b = 2.0 * x * y * drho + 2.0 * k[2] * x + 2.0 * k[3] * y;
  d = rho + 2.0 * y * y * drho + 6.0 * k[2] * y + 2.0 * k[3] * x;
}

// g(s) = 1 + 3 k1 s + 5 k2 s^2 + 7 k3 s^3 = d (r rho(r)) / dr at r^2 = s.
__device__ __forceinline__ double lens_radial_slope(const double (&k)[5], double s) {
  return 1.0 + s * (3.0 * k[0] + s * (5.0 * k[1] + s * (7.0 * k[4])));
}

// The validity rule of the header at (x, y), given det J there.  False for non-finite input.
__device__ __forceinline__ bool lens_valid(const double (&k)[5], double x, double y, double det) {
  const double r2 = x * x + y * y;
  bool ok = det > 0.0 && lens_radial_slope(k, r2) > 0.0 && r2 < __longlong_as_double(0x7ff0000000000000ll);
  if (k[4] != 0.0) {
    const double disc = 100.0 * k[1] * k[1] - 252.0 * k[0] * k[4];
    if (disc >= 0.0) {
      const double sq = sqrt(disc);
      const double s1 = (-10.0 * k[1] - sq) / (42.0 * k[4]), s2 = (-10.0 * k[1] + sq) / (42.0 * k[4]);
      if (s1 > 0.0 && s1 < r2) ok = ok && lens_radial_slope(k, s1) > 0.0;
      if (s2 > 0.0 && s2 < r2) ok = ok && lens_radial_slope(k, s2) > 0.0;
    }
  } else if (k[1] != 0.0) {
    const double s1 = -3.0 * k[0] / (10.0 * k[1]);
    if (s1 > 0.0 && s1 < r2) ok = ok && lens_radial_slope(k, s1) > 0.0;
  }
  return ok;
}

template <bool kPerPose>
__global__ void __launch_bounds__(256) distort_pixels_kernel(const float* pin, float* pout, const double* __restrict__ calib,
                                                             int64_t cstride, const double* __restrict__ dist, int64_t dstride,
                                                             int64_t B, int V, int J) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B * V * J) return;
  const float u = pin[e * 3], w = pin[e * 3 + 1], conf = pin[e * 3 + 2];
  float ou = u, ow = w, oc = conf;
  if (conf != 0.0f) {
    const int64_t bv = e / J, b = bv / V;
    const int v = (int)(bv - b * V);
    const double* c = (kPerPose ? calib + b * cstride : calib) + v * 18;
    const double* dd = (kPerPose ? dist + b * dstride : dist) + v * 5;
    const double k[5] = {dd[0], dd[1], dd[2], dd[3], dd[4]};
    const double fx = c[12], fy = c[13];
    const double x = ((double)u - c[14]) / fx, y = ((double)w - c[15]) / fy;
    double xd, yd, a, bb, d;
    lens_map(k, x, y, xd, yd, a, bb, d);
    if (k[0] == 0.0 && k[1] == 0.0 && k[2] == 0.0 && k[3] == 0.0 && k[4] == 0.0) {
      // no lens: the entry as it is (the arithmetic below would turn -0 into +0 and zero conf at a non-finite pixel)
    } else if (lens_valid(k, x, y, a * d - bb * bb)) {
      ou = (float)((double)u + fx * (xd - x));
      ow = (float)((double)w + fy * (yd - y));
    } else {
      oc = 0.0f;
    }
  }
  pout[e * 3] = ou;
  pout[e * 3 + 1] = ow;
  pout[e * 3 + 2] = oc;
}

template <bool kPerPose>
__global__ void __launch_bounds__(256) undistort_pixels_kernel(const float* pin, float* pout, const double* __restrict__ calib,
                                                               int64_t cstride, const double* __restrict__ dist,
                                                               int64_t dstride, double margin_x, double margin_y, int64_t B,
                                                               int V, int J) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B * V * J) return;
  const float u = pin[e * 3], w = pin[e * 3 + 1], conf = pin[e * 3 + 2];
  float ou = u, ow = w, oc = conf;
  if (conf != 0.0f) {
    const int64_t bv = e / J, b = bv / V;
    const int v = (int)(bv - b * V);
    const double* c = (kPerPose ? calib + b * cstride : calib) + v * 18;
    if (!(0.0 < (double)u && (double)u < c[16] - 1.0 && 0.0 < (double)w && (double)w < c[17] - 1.0)) {
      oc = 0.0f;                                         // not a candidate of the triangulations on the raw pixels
    } else {
      const double* dd = (kPerPose ? dist + b * dstride : dist) + v * 5;
      const double k[5] = {dd[0], dd[1], dd[2], dd[3], dd[4]};
      const double fx = c[12], fy = c[13];
      const double xd = ((double)u - c[14]) / fx, yd = ((double)w - c[15]) / fy;
      double x = xd, y = yd, px, py, a, bb, d;
      for (int it = 0; it < kLensMaxIters; ++it) {
        lens_map(k, x, y, px, py, a, bb, d);
        const double det = a * d - bb * bb, rx = px - xd, ry = py - yd;
        const double dx = (d * rx - bb * ry) / det, dy = (a * ry - bb * rx) / det;
        x -= dx;
        y -= dy;
        if (!(fabs(dx) + fabs(dy) > 1e-14)) break;
      }
      lens_map(k, x, y, px, py, a, bb, d);
      if (fabs(px - xd) + fabs(py - yd) <= 1e-12 && lens_valid(k, x, y, a * d - bb * bb)) {
        ou = (float)((double)u + fx * (x - xd) + margin_x);
        ow = (float)((double)w + fy * (y - yd) + margin_y);
      } else {
        ou = ow = __int_as_float(0x7fc00000);
        oc = 0.0f;
      }
    }
  }
  pout[e * 3] = ou;
  pout[e * 3 + 1] = ow;
  pout[e * 3 + 2] = oc;
}

int launch_lens_pixels(bool undistort, const float* pin, float* pout, const double* calib, int64_t calib_stride,
                       const double* dist, int64_t dist_stride, double margin_x, double margin_y, int64_t B, int V, int J,
                       cudaStream_t s) {
  const int64_t total = B * V * J;
  if (total == 0) return MPL_OK;
  const unsigned grid = (unsigned)ceil_div(total, 256);
  const bool per_pose = calib_stride != 0 || dist_stride != 0;
  if (undistort) {
    if (per_pose)
      undistort_pixels_kernel<true><<<grid, 256, 0, s>>>(pin, pout, calib, calib_stride, dist, dist_stride, margin_x, margin_y,
                                                         B, V, J);
    else
      undistort_pixels_kernel<false><<<grid, 256, 0, s>>>(pin, pout, calib, 0, dist, 0, margin_x, margin_y, B, V, J);
  } else {
    if (per_pose)
      distort_pixels_kernel<true><<<grid, 256, 0, s>>>(pin, pout, calib, calib_stride, dist, dist_stride, B, V, J);
    else
      distort_pixels_kernel<false><<<grid, 256, 0, s>>>(pin, pout, calib, 0, dist, 0, B, V, J);
  }
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- random camera setups: one thread per (pose, view), fp64 ------------------------------------------------------------
// U0..U5 of (pose i, view v) come from the Philox4x64-10 stream of synth_project_kernel under key (seed, 2), with the slot
// layout of the detector-noise model (pose i owns counter blocks [i nb, (i + 1) nb), nb = ceil(6 V / 4), slot 6 v + m is
// U_m), so a pose's cameras depend only on (seed, global pose index).  openmpl_b200/synth.py (random_cameras) is the twin.
//   azimuth a = 2 pi (v + 0.8 (U0 - 0.5)) / V + 0.3 (each camera stays in its sector), horizontal distance from the look-at
//   point 4.5 (0.75 + 0.5 U1), height 0.9 + 1.2 U2, look-at point = room centre at height 0.9 shifted by 0.5 (U3 - 0.5) in x
//   and 0.5 (U4 - 0.5) in y, fx = fy = f0 (0.8 + 0.4 U5), principal point at the image centre, R the look-at rotation of
//   synth.make_rig.  Every U = 0.5 gives make_rig's camera.
__global__ void __launch_bounds__(128) synth_cameras_kernel(uint64_t seed, int64_t start, int64_t B, int V, double f0,
                                                            double w, double h, const double* __restrict__ room,
                                                            double* __restrict__ calib) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B * V) return;
  const int64_t b = e / V;
  const int v = (int)(e - b * V);
  double U[6];
  six_uniforms(seed, 2ull, start, b, V, v, U);
  double sn, cs;
  sincospi(2.0 * (v + 0.8 * (U[0] - 0.5)) / V + 0.3 / 3.14159265358979323846, &sn, &cs);  // sincos's reduction needs a stack frame
  const double dist = 4.5 * (0.75 + 0.5 * U[1]);
  const double at[3] = {0.5 * (room[0] + room[1]) + 0.5 * (U[3] - 0.5), 0.5 * (room[2] + room[3]) + 0.5 * (U[4] - 0.5), 0.9};
  const double pos[3] = {at[0] + dist * cs, at[1] + dist * sn, 0.9 + 1.2 * U[2]};
  double z[3] = {at[0] - pos[0], at[1] - pos[1], at[2] - pos[2]};
  const double zn = sqrt(z[0] * z[0] + z[1] * z[1] + z[2] * z[2]);
#pragma unroll
  for (int k = 0; k < 3; ++k) z[k] /= zn;
  const double xn = sqrt(z[1] * z[1] + z[0] * z[0]);
  const double x[3] = {z[1] / xn, -z[0] / xn, 0.0};                                    // z x (0, 0, 1)
  const double y[3] = {z[1] * x[2] - z[2] * x[1], z[2] * x[0] - z[0] * x[2], z[0] * x[1] - z[1] * x[0]};  // z x x
  const double f = f0 * (0.8 + 0.4 * U[5]);
  double* c = calib + e * 18;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    c[k] = x[k];
    c[3 + k] = y[k];
    c[6 + k] = z[k];
    c[9 + k] = pos[k];
  }
  c[12] = f;
  c[13] = f;
  c[14] = w / 2.0;
  c[15] = h / 2.0;
  c[16] = w;
  c[17] = h;
}

int launch_synth_cameras(uint64_t seed, int64_t start, int64_t B, int V, double f0, double w, double h, const double* room,
                         double* calib, cudaStream_t s) {
  const int64_t total = B * V;
  if (total == 0) return MPL_OK;
  synth_cameras_kernel<<<(unsigned)ceil_div(total, 128), 128, 0, s>>>(seed, start, B, V, f0, w, h, room, calib);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- calibration errors: one thread per (pose, view), fp64 -------------------------------------------------------------
// U0..U5 of (pose i, view v) come from the Philox4x64-10 stream under key (seed, 3), in the slot layout of synth_cameras_kernel.
// Six standard normals by Box-Muller on (U0, U1), (U2, U3), (U4, U5); R' = Exp(sigma_rot n0..2) R (a rotation in the camera
// frame), t' = t + sigma_pos n3..5 (the camera centre).  openmpl_b200/synth.py (calibration_noise) is the twin.  A thread reads
// its whole row before it writes, so calib_out may be calib when the rows coincide (stride 18 V).
__global__ void __launch_bounds__(128) synth_calib_noise_kernel(uint64_t seed, int64_t start, int64_t B, int V,
                                                                const double* calib, int64_t cstride, double sigma_rot,
                                                                double sigma_pos, double* calib_out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B * V) return;
  const int64_t b = e / V;
  const int v = (int)(e - b * V);
  const double* c = calib + b * cstride + v * 18;
  double row[18];
#pragma unroll
  for (int k = 0; k < 18; ++k) row[k] = c[k];
  double U[6], n[6];
  six_uniforms(seed, 3ull, start, b, V, v, U);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double r = sqrt(-2.0 * log(fmax(U[2 * k], 1e-12)));
    double sn, cs;
    sincospi(2.0 * U[2 * k + 1], &sn, &cs);
    n[2 * k] = r * cs;
    n[2 * k + 1] = r * sn;
  }
  if (sigma_rot != 0.0) {
    const double w[3] = {sigma_rot * n[0], sigma_rot * n[1], sigma_rot * n[2]};
    double E[9], Rn[9];
    so3_exp(w, E);
    mat3_mul(E, row, Rn);
#pragma unroll
    for (int k = 0; k < 9; ++k) row[k] = Rn[k];
  }
  if (sigma_pos != 0.0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) row[9 + k] += sigma_pos * n[3 + k];
  }
  double* o = calib_out + e * 18;
#pragma unroll
  for (int k = 0; k < 18; ++k) o[k] = row[k];
}

int launch_synth_calib_noise(uint64_t seed, int64_t start, int64_t B, int V, const double* calib, int64_t calib_stride,
                             double sigma_rot, double sigma_pos, double* calib_out, cudaStream_t s) {
  const int64_t total = B * V;
  if (total == 0) return MPL_OK;
  synth_calib_noise_kernel<<<(unsigned)ceil_div(total, 128), 128, 0, s>>>(seed, start, B, V, calib, calib_stride, sigma_rot,
                                                                          sigma_pos, calib_out);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

int launch_build_inputs(const float* pix, const double* calib, int64_t calib_stride, int64_t B, int V, int J, float* poses,
                        float* rays, float* centers, cudaStream_t s) {
  const int64_t total = B * V * J;
  if (total == 0) return MPL_OK;
  const unsigned grid = (unsigned)ceil_div(total, 256);
  if (calib_stride == 0)
    build_inputs_kernel<false><<<grid, 256, 0, s>>>(pix, calib, 0, B, V, J, poses, rays, centers);
  else
    build_inputs_kernel<true><<<grid, 256, 0, s>>>(pix, calib, calib_stride, B, V, J, poses, rays, centers);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

}  // namespace mpl
