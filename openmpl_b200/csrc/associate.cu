// Multi-person cross-view association (ABI 11; defined by this library, the reference's datasets give the grouping as
// ground truth).  The contracts are stated in include/mpl_b200.h; tests/association_oracle.py restates them in numpy and
// openmpl_b200/synth.py (synth_people) is the twin of the scene generator.
//
//   synth_people_kernel       one CTA per frame: the slot permutations (Philox key (seed, 4)) and the permuted copy
//   associate_kernel          one CTA per frame: rays, pair costs, a bitonic sort of the admissible pairs, the greedy
//                             complete-linkage pass (one thread), the ranking and the outputs
//   gather_people_kernel      one thread per (frame, row, view, joint): the member's row or zeros
//   association_score_kernel  one CTA, one warp per frame: integer counts, added to the fp64 sums once at the end
#include "kernels.cuh"
#include "shared.cuh"

namespace mpl {

constexpr int kAssocThreads = 128;  // >= the detections of a frame (P V <= 128): thread m owns detection m = s V + v
constexpr int kAssocMaxDet = 128;
constexpr int kScoreWarps = 8;

// ---- scenes out of person-ordered pixels ------------------------------------------------------------------------------
// perm[f, v] is the stable ascending argsort of the uniforms in slots v P .. v P + P - 1 of frame start + f (counter blocks
// [i nb, (i + 1) nb), nb = ceil(V P / 4), under key (seed, 4)); scene[f, s, v] = pix[f P + perm[f, v, s], v], copied as
// 32-bit words so that every bit (NaN payloads, -0) survives.
__global__ void __launch_bounds__(kAssocThreads) synth_people_kernel(uint64_t seed, int64_t start, int P, int V, int J,
                                                                     const float* __restrict__ pix, float* __restrict__ scene,
                                                                     int32_t* __restrict__ perm) {
  __shared__ double su[kAssocMaxDet];
  __shared__ int sp[kAssocMaxDet];
  const int64_t f = blockIdx.x;
  const int tid = threadIdx.x, M = P * V;
  if (tid < M) {
    const uint64_t base = (uint64_t)(start + f) * (uint64_t)((M + 3) / 4);
    uint64_t r[4];
    philox4x64_10(base + (uint64_t)(tid >> 2) + 1ull, seed, 4ull, r);  // numpy increments the counter before generating
    const int k = tid & 3;
    const uint64_t raw = k == 0 ? r[0] : (k == 1 ? r[1] : (k == 2 ? r[2] : r[3]));
    su[tid] = (double)(raw >> 11) * (1.0 / 9007199254740992.0);
  }
  __syncthreads();
  if (tid < M) {
    const int v = tid / P, k = tid - v * P;
    const double x = su[tid];
    int rank = 0;
    for (int m = 0; m < P; ++m) {
      const double y = su[v * P + m];
      rank += (y < x) || (y == x && m < k);
    }
    sp[v * P + rank] = k;
  }
  __syncthreads();
  if (tid < M) perm[f * M + tid] = sp[tid];
  const int row = 3 * J;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(pix);
  uint32_t* dst = reinterpret_cast<uint32_t*>(scene);
  for (int e = tid; e < M * row; e += blockDim.x) {
    const int sv = e / row, q = e - sv * row;              // sv = s V + v
    const int s = sv / V, v = sv - s * V;
    dst[(f * M + sv) * (int64_t)row + q] = src[((f * P + sp[v * P + s]) * V + v) * (int64_t)row + q];
  }
}

int launch_synth_people(uint64_t seed, int64_t start, int64_t F, int P, int V, int J, const float* pix, float* scene,
                        int32_t* perm, cudaStream_t s) {
  synth_people_kernel<<<(unsigned)F, kAssocThreads, 0, s>>>(seed, start, P, V, J, pix, scene, perm);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- association --------------------------------------------------------------------------------------------------------
// Distance between the lines c1 + a d1 and c2 + b d2, dc = c2 - c1 (the rule of the header).
__device__ __forceinline__ double line_distance(const double (&dc)[3], const double* d1, const double* d2) {
  const double n[3] = {d1[1] * d2[2] - d1[2] * d2[1], d1[2] * d2[0] - d1[0] * d2[2], d1[0] * d2[1] - d1[1] * d2[0]};
  const double nn = n[0] * n[0] + n[1] * n[1] + n[2] * n[2];
  const double a2 = d1[0] * d1[0] + d1[1] * d1[1] + d1[2] * d1[2];
  const double b2 = d2[0] * d2[0] + d2[1] * d2[1] + d2[2] * d2[2];
  if (nn <= 1e-24 * a2 * b2) {                             // parallel rays: the distance of c2 from the first line
    const double x[3] = {dc[1] * d1[2] - dc[2] * d1[1], dc[2] * d1[0] - dc[0] * d1[2], dc[0] * d1[1] - dc[1] * d1[0]};
    return sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]) / sqrt(a2);
  }
  return fabs(dc[0] * n[0] + dc[1] * n[1] + dc[2] * n[2]) / sqrt(nn);
}

// Median of x[0, n) (n >= 1) by rank counting in shared memory: the element of stable rank (n - 1) / 2 and the one of rank
// n / 2, averaged.  A NaN has no rank, so a list holding one gives NaN, which no threshold admits.
__device__ __forceinline__ double median_of(const double* x, int n) {
  const int i1 = (n - 1) >> 1, i2 = n >> 1;
  double lo = __longlong_as_double(0x7ff8000000000000ll), hi = lo;
  for (int i = 0; i < n; ++i) {
    const double xi = x[i];
    int r = 0;
    for (int k = 0; k < n; ++k) r += (x[k] < xi) || (x[k] == xi && k < i);
    if (r == i1) lo = xi;
    if (r == i2) hi = xi;
  }
  return i1 == i2 ? lo : 0.5 * (lo + hi);
}

// Admissible pairs of a frame: cross-view pairs of its detections (at most M (M - 1) / 2 - V P (P - 1) / 2), rounded up to a
// power of two for the bitonic sort.
static int assoc_edge_cap(int P, int V) {
  const int M = P * V, pairs = M * (M - 1) / 2 - V * (P * (P - 1) / 2);
  int c = 1;
  while (c < pairs) c <<= 1;
  return c;
}

static size_t assoc_smem(int P, int V, int J) {
  const int M = P * V;
  return (size_t)(M * J * 3 + kAssocThreads * J) * sizeof(double) + (size_t)assoc_edge_cap(P, V) * (sizeof(double) + 2);
}

__global__ void __launch_bounds__(kAssocThreads) associate_kernel(const float* __restrict__ scene, const double* __restrict__ calib,
                                                                  int64_t cstride, int P, int V, int J, float min_conf,
                                                                  int min_joints, double max_dist, int K, int cap,
                                                                  int32_t* __restrict__ members, int32_t* __restrict__ labels,
                                                                  int32_t* __restrict__ people) {
  extern __shared__ double dsm[];
  const int M = P * V, tid = threadIdx.x, T = blockDim.x;
  double* sdir = dsm;                                       // [M][J][3] ray directions of the candidate joints
  double* sdist = sdir + M * J * 3;                         // [T][J] per-thread joint distances of one pair
  double* ecost = sdist + T * J;                            // [cap] admissible pairs: cost
  uint16_t* ekey = reinterpret_cast<uint16_t*>(ecost + cap);  //            and key m1 M + m2 (m1 the lower view)
  __shared__ double sc[kMaxViews][18];
  __shared__ uint32_t cmask[kAssocMaxDet];                 // candidate joints (J <= 32)
  __shared__ uint32_t adj[kAssocMaxDet][4];                // bit m2 of row m1: cost(m1, m2) <= max_dist
  __shared__ uint32_t memb[kAssocMaxDet][4];               // members of the cluster whose representative is m
  __shared__ uint32_t vmask[kAssocMaxDet];                 // its views
  __shared__ int cl[kAssocMaxDet];                         // cluster representative of m, -1 if m is inactive
  __shared__ int pcnt[kAssocMaxDet], pmin[kAssocMaxDet], prank[kAssocMaxDet];
  __shared__ int slot[kAssocMaxDet / 2][kMaxViews];        // a frame has at most M / 2 people
  __shared__ int nedge, npeople;
  const int64_t f = blockIdx.x;
  const double* cal = calib + f * cstride;
  for (int e = tid; e < V * 18; e += T) sc[e / 18][e % 18] = cal[e];
  for (int e = tid; e < M * 4; e += T) adj[e >> 2][e & 3] = 0;
  for (int e = tid; e < (M / 2) * kMaxViews; e += T) slot[e / kMaxViews][e % kMaxViews] = -1;
  if (tid == 0) nedge = npeople = 0;
  __syncthreads();

  // candidate joints, active detections and the rays R^T ((u - cx) / fx, (v - cy) / fy, 1) of detection m = s V + v
  if (tid < M) {
    const int v = tid % V;
    const double wh[2] = {sc[v][16], sc[v][17]};
    const float* px = scene + (f * M + tid) * (int64_t)(3 * J);
    uint32_t cm = 0;
    for (int j = 0; j < J; ++j) {
      const float u = px[3 * j], w = px[3 * j + 1];
      if (!tri_candidate(px[3 * j + 2], u, w, min_conf, wh)) continue;
      cm |= 1u << j;
      const double x = ((double)u - sc[v][14]) / sc[v][12], y = ((double)w - sc[v][15]) / sc[v][13];
      double* d = sdir + (tid * J + j) * 3;
#pragma unroll
      for (int r = 0; r < 3; ++r) d[r] = sc[v][r] * x + sc[v][3 + r] * y + sc[v][6 + r];
    }
    const bool active = __popc(cm) >= min_joints;
    cmask[tid] = cm;
    cl[tid] = active ? tid : -1;
#pragma unroll
    for (int q = 0; q < 4; ++q) memb[tid][q] = active && (tid >> 5) == q ? 1u << (tid & 31) : 0u;
    vmask[tid] = active ? 1u << v : 0u;
  }
  __syncthreads();

  // pair costs: the median line distance over the shared candidate joints; the admissible pairs (cost <= max_dist) go to
  // the adjacency bits and the edge list (the list's order is fixed by the sort below)
  for (int idx = tid; idx < M * M; idx += T) {
    const int a = idx / M, b = idx - a * M;
    if (a >= b || a % V == b % V || cl[a] < 0 || cl[b] < 0) continue;
    const uint32_t shared_j = cmask[a] & cmask[b];
    const int n = __popc(shared_j);
    if (n < min_joints) continue;                         // cost +inf
    const int m1 = a % V < b % V ? a : b, m2 = a + b - m1;
    const int v1 = m1 % V, v2 = m2 % V;
    const double dc[3] = {sc[v2][9] - sc[v1][9], sc[v2][10] - sc[v1][10], sc[v2][11] - sc[v1][11]};
    double* dist = sdist + tid * J;
    int k = 0;
    for (uint32_t rest = shared_j; rest; rest &= rest - 1) {
      const int j = __ffs(rest) - 1;
      dist[k++] = line_distance(dc, sdir + (m1 * J + j) * 3, sdir + (m2 * J + j) * 3);
    }
    const double cost = median_of(dist, n);
    if (cost <= max_dist) {
      atomicOr(&adj[a][b >> 5], 1u << (b & 31));
      atomicOr(&adj[b][a >> 5], 1u << (a & 31));
      const int e = atomicAdd(&nedge, 1);
      ecost[e] = cost;
      ekey[e] = (uint16_t)(m1 * M + m2);
    }
  }
  __syncthreads();

  // bitonic sort of the admissible pairs by (cost, key), padded to a power of two with (+inf, 0xffff)
  const int ne = nedge;
  int n2 = 1;
  while (n2 < ne) n2 <<= 1;
  for (int e = ne + tid; e < n2; e += T) {
    ecost[e] = __longlong_as_double(0x7ff0000000000000ll);
    ekey[e] = 0xffff;
  }
  __syncthreads();
  for (int k = 2; k <= n2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n2; i += T) {
        const int l = i ^ j;
        if (l <= i) continue;
        const double ci = ecost[i], cj = ecost[l];
        const uint16_t ki = ekey[i], kj = ekey[l];
        const bool gt = ci > cj || (ci == cj && ki > kj);
        if (gt == ((i & k) == 0)) {
          ecost[i] = cj; ecost[l] = ci;
          ekey[i] = kj; ekey[l] = ki;
        }
      }
      __syncthreads();
    }
  }

  // greedy complete linkage, in the sorted order: merge unless one cluster already, a shared view, or a cross pair of
  // members that is not admissible
  if (tid == 0) {
    for (int e = 0; e < ne; ++e) {
      const int a = ekey[e] / M, b = ekey[e] - (ekey[e] / M) * M;
      const int ca = cl[a], cb = cl[b];
      if (ca == cb || (vmask[ca] & vmask[cb]) != 0u) continue;
      bool ok = true;
      for (int q = 0; q < 4 && ok; ++q)
        for (uint32_t rest = memb[ca][q]; rest && ok; rest &= rest - 1) {
          const int x = 32 * q + __ffs(rest) - 1;
#pragma unroll
          for (int r = 0; r < 4; ++r) ok = ok && (memb[cb][r] & ~adj[x][r]) == 0u;
        }
      if (!ok) continue;
      for (int q = 0; q < 4; ++q) {
        for (uint32_t rest = memb[cb][q]; rest; rest &= rest - 1) cl[32 * q + __ffs(rest) - 1] = ca;
        memb[ca][q] |= memb[cb][q];
        memb[cb][q] = 0u;
      }
      vmask[ca] |= vmask[cb];
      vmask[cb] = 0u;
    }
  }
  __syncthreads();

  // people: clusters of >= 2 members, ranked by member count descending, then smallest member ascending
  if (tid < M) {
    int c = 0, lo = -1;
    if (cl[tid] == tid) {
#pragma unroll
      for (int q = 3; q >= 0; --q) {
        c += __popc(memb[tid][q]);
        if (memb[tid][q]) lo = 32 * q + __ffs(memb[tid][q]) - 1;
      }
    }
    pcnt[tid] = c >= 2 ? c : 0;
    pmin[tid] = lo;
    if (c >= 2) atomicAdd(&npeople, 1);
  }
  __syncthreads();
  if (tid < M && pcnt[tid] > 0) {
    int r = 0;
    for (int q = 0; q < M; ++q) r += pcnt[q] > pcnt[tid] || (pcnt[q] == pcnt[tid] && pcnt[q] > 0 && pmin[q] < pmin[tid]);
    prank[tid] = r;
  }
  __syncthreads();
  if (tid < M) {
    const int c = cl[tid];
    int lab = -2;
    if (c >= 0) lab = pcnt[c] > 0 && prank[c] < K ? prank[c] : -1;
    labels[f * M + tid] = lab;
    if (lab >= 0) slot[lab][tid % V] = tid / V;
  }
  __syncthreads();
  for (int64_t e = tid; e < (int64_t)K * V; e += T) {
    const int k = (int)(e / V), v = (int)(e - (int64_t)k * V);
    members[f * K * V + e] = k < M / 2 ? slot[k][v] : -1;
  }
  if (tid == 0) people[f] = npeople;
}

int launch_associate_people(const float* scene, const double* calib, int64_t calib_stride, int64_t F, int P, int V, int J,
                            float min_conf, int min_joints, double max_dist, int K, int32_t* members, int32_t* labels,
                            int32_t* people, cudaStream_t s) {
  const size_t smem = assoc_smem(P, V, J);
  MPL_CUDA(cudaFuncSetAttribute(associate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  associate_kernel<<<(unsigned)F, kAssocThreads, smem, s>>>(scene, calib, calib_stride, P, V, J, min_conf, min_joints,
                                                            max_dist, K, assoc_edge_cap(P, V), members, labels, people);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- gather: out[f, k, v] = scene[f, members[f, k, v], v], zeros where there is no member --------------------------------
__global__ void __launch_bounds__(256) gather_people_kernel(const float* __restrict__ scene, const int32_t* __restrict__ members,
                                                            int64_t F, int P, int K, int V, int J, float* __restrict__ out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // (f, k, v, j)
  if (e >= F * K * V * J) return;
  const int64_t fkv = e / J, fk = fkv / V, f = fk / K;
  const int j = (int)(e - fkv * J), v = (int)(fkv - fk * V);
  const int s = members[fkv];
  uint32_t w[3] = {0u, 0u, 0u};
  if (s >= 0 && s < P) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(scene) + (((f * P + s) * V + v) * J + j) * 3;
    w[0] = src[0]; w[1] = src[1]; w[2] = src[2];
  }
  uint32_t* dst = reinterpret_cast<uint32_t*>(out) + e * 3;
  dst[0] = w[0]; dst[1] = w[1]; dst[2] = w[2];
}

int launch_gather_people(const float* scene, const int32_t* members, int64_t F, int P, int K, int V, int J, float* out,
                         cudaStream_t s) {
  const int64_t total = F * K * V * J;
  gather_people_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(scene, members, F, P, K, V, J, out);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- score: one warp per frame, integer counts per lane, one fixed-order reduction, then acc += the counts ---------------
__global__ void __launch_bounds__(kScoreWarps * 32, 1) association_score_kernel(const int32_t* __restrict__ members,
                                                                             const int32_t* __restrict__ labels,
                                                                             const int32_t* __restrict__ perm, int64_t F,
                                                                             int P, int K, int V, int32_t* __restrict__ owner,
                                                                             double* __restrict__ acc) {
  __shared__ int cnt[kScoreWarps][kAssocMaxDet];           // active detections per true person of the warp's frame
  __shared__ long long red[kScoreWarps][7];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, M = P * V;
  // associable people, non-empty rows, pure rows, complete rows, predicted pairs, correct pairs, true pairs
  long long c[7] = {0, 0, 0, 0, 0, 0, 0};
  for (int64_t f = w; f < F; f += kScoreWarps) {
    for (int p = lane; p < P; p += 32) cnt[w][p] = 0;
    __syncwarp();
    for (int m = lane; m < M; m += 32) {
      const int s = m / V, v = m - s * V;
      const int p = perm[(f * V + v) * P + s];
      if (labels[f * M + m] != -2 && p >= 0 && p < P) atomicAdd(&cnt[w][p], 1);
    }
    __syncwarp();
    for (int p = lane; p < P; p += 32) {
      const int a = cnt[w][p];
      c[0] += a >= 2;
      c[6] += a * (a - 1) / 2;
    }
    for (int64_t k = lane; k < K; k += 32) {
      const int32_t* row = members + (f * K + k) * V;
      const int32_t* pf = perm + f * V * P;
      int n = 0, best = -1, bestc = 0;
      long long same = 0;
      for (int v = 0; v < V; ++v) {
        const int s = row[v];
        if (s < 0 || s >= P) continue;
        ++n;
        const int t = pf[v * P + s];
        int ct = 0;
        for (int x = 0; x < V; ++x) {
          const int s2 = row[x];
          if (s2 < 0 || s2 >= P || pf[x * P + s2] != t) continue;
          ++ct;
          same += x > v;
        }
        if (ct > bestc || (ct == bestc && t < best)) { best = t; bestc = ct; }
      }
      owner[f * K + k] = n > 0 ? best : -1;
      if (n > 0) {
        c[1] += 1;
        c[4] += n * (n - 1) / 2;
        c[5] += same;
        if (bestc == n) {
          c[2] += 1;
          c[3] += best >= 0 && best < P && cnt[w][best] == n;
        }
      }
    }
    __syncwarp();
  }
#pragma unroll
  for (int q = 0; q < 7; ++q) {
    const long long t = warp_sum_ll(c[q]);
    if (lane == 0) red[w][q] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    acc[0] += (double)F;
#pragma unroll
    for (int q = 0; q < 7; ++q) {
      long long t = 0;
      for (int x = 0; x < kScoreWarps; ++x) t += red[x][q];
      acc[1 + q] += (double)t;
    }
  }
}

int launch_association_score(const int32_t* members, const int32_t* labels, const int32_t* perm, int64_t F, int P, int K,
                             int V, int32_t* owner, double* acc, cudaStream_t s) {
  association_score_kernel<<<1, kScoreWarps * 32, 0, s>>>(members, labels, perm, F, P, K, V, owner, acc);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

}  // namespace mpl
