// Multi-person tracking across frames (additions to ABI 11; defined by this library).  The contracts are stated in
// include/mpl_b200.h; tests/tracking_oracle.py restates the tracker and the score in numpy and openmpl_b200/synth.py
// (synth_motion) is the twin of the motion generator.
//
//   synth_motion_kernel     one thread per (sequence, frame, person) row: the closed-form motion (Philox key (seed, 5)),
//                           then synth_project's camera model and confidences (project_pixel, key (seed, 0))
//   track_people_kernel     one CTA per sequence, the track state in shared memory for the whole call; per frame one warp
//                           per (track, row) pair computes the median joint distance, a bitonic sort orders the admissible
//                           pairs, and one thread matches them greedily, ages the tracks and starts new ones
//   tracking_score_kernel   one CTA, one warp per sequence: integer counts, added to the fp64 sums once at the end
#include "kernels.cuh"
#include "shared.cuh"

namespace mpl {

constexpr int kTrackThreads = 256;
constexpr int kTrackScoreWarps = 8;
constexpr double kTwoPi = 2.0 * 3.14159265358979323846;

// ---- people that move -----------------------------------------------------------------------------------------------------
// Uniform slots of (sequence i, person p) under key (seed, 5), counter blocks [g nb, (g + 1) nb), g = i P + p,
// nb = ceil((9 + 6 (J - 1)) / 4): 0, 1 amplitude; 2, 3 frequency; 4, 5 phase (x, y); 6 height; 7 heading; 8 turn rate;
// 9 + m and 9 + 3 (J - 1) + m the Box-Muller pair of body offset m = 3 (j - 1) + k.
__global__ void __launch_bounds__(128) synth_motion_kernel(uint64_t seed, int64_t start, int64_t rows, int T, int P, int V,
                                                           int J, const double* __restrict__ calib, int64_t cstride,
                                                           const double* __restrict__ room, double fps, int conf_ones,
                                                           float* __restrict__ pix, float* __restrict__ target) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= rows) return;
  const int64_t st = b / P;                                 // s T + t
  const int p = (int)(b - st * P);
  const int64_t s = st / T;
  const int t = (int)(st - s * T);
  const int n = 3 * (J - 1);
  const uint64_t g = (uint64_t)(start + s) * (uint64_t)P + (uint64_t)p;
  const uint64_t mb = (uint64_t)((9 + 2 * n + 3) / 4);
  UniformCursor ca(g * mb, seed, 5ull), cb(g * mb, seed, 5ull);
  const double wx = room[1] - room[0], wy = room[3] - room[2];
  const double tau = (double)t / fps;
  const double ax = (0.25 + 0.25 * ca.get(0)) * wx, ay = (0.25 + 0.25 * ca.get(1)) * wy;
  const double fx = 0.03 + 0.07 * ca.get(2), fy = 0.03 + 0.07 * ca.get(3);
  const double px0 = kTwoPi * ca.get(4), py0 = kTwoPi * ca.get(5);
  double root[3];
  root[0] = 0.5 * (room[0] + room[1]) + ax * sin(kTwoPi * fx * tau + px0);
  root[1] = 0.5 * (room[2] + room[3]) + ay * sin(kTwoPi * fy * tau + py0);
  root[2] = 0.8 + 0.2 * ca.get(6);
  const double theta = kTwoPi * ca.get(7) + (ca.get(8) - 0.5) * tau;
  const double cth = cos(theta), sth = sin(theta);
  // confidences: mpl_synth_project's slots of global row r (pose r of its stream)
  const int64_t r = start * (int64_t)T * P + b;
  const uint64_t pb = (uint64_t)((3 + 2 * n + V * J + 3) / 4);
  UniformCursor cc((uint64_t)r * pb, seed);
  const double* cal = calib + b * cstride;
  float* tg = target + b * J * 3;
  float* px = pix + b * V * J * 3;
  for (int j = 0; j < J; ++j) {
    double o[3] = {0.0, 0.0, 0.0};
    if (j > 0) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const int i = (j - 1) * 3 + k;
        const double u1 = fmax(ca.get(9 + i), 1e-12), u2 = cb.get(9 + n + i);
        o[k] = 0.25 * (sqrt(-2.0 * log(u1)) * cos(kTwoPi * u2));  // Box-Muller as synth_project_kernel draws it
      }
    }
    const double X[3] = {root[0] + (cth * o[0] - sth * o[1]), root[1] + (sth * o[0] + cth * o[1]), root[2] + o[2]};
#pragma unroll
    for (int k = 0; k < 3; ++k) tg[j * 3 + k] = (float)X[k];
    for (int v = 0; v < V; ++v)
      project_pixel(cal + v * 18, X, conf_ones ? 1.0 : 0.3 + 0.7 * cc.get(3 + 2 * n + v * J + j), px + (v * J + j) * 3);
  }
}

int launch_synth_motion(uint64_t seed, int64_t start, int64_t S, int T, int P, int V, int J, const double* calib,
                        int64_t calib_stride, const double* room, double fps, int conf_ones, float* pix, float* target,
                        cudaStream_t s) {
  const int64_t rows = S * T * P;
  synth_motion_kernel<<<(unsigned)ceil_div(rows, 128), 128, 0, s>>>(seed, start, rows, T, P, V, J, calib, calib_stride, room,
                                                                     fps, conf_ones, pix, target);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- tracking ---------------------------------------------------------------------------------------------------------------
// State of one sequence, in 32-bit words: [0] the next id, [1..3] zero; then max_tracks slots of 4 + 3 J words: live, id,
// misses, the joint bitmask of the remembered positions, then the positions as fp32 [J][3].  All zeros: no live track.
__host__ __device__ __forceinline__ int track_slot_words(int J) { return 4 + 3 * J; }

size_t track_state_bytes(int max_tracks, int J) {
  return (size_t)4 * (4 + (size_t)max_tracks * track_slot_words(J));
}

// Pair list capacity: every (track, row) pair, rounded up to a power of two (>= 2) for the bitonic sort.
static int track_edge_cap(int NT, int K) {
  int c = 2;
  while (c < NT * K) c <<= 1;
  return c;
}

static size_t track_smem(int NT, int K, int J) {
  const int cap = track_edge_cap(NT, K);
  return (size_t)cap * (sizeof(double) + sizeof(uint16_t)) + track_state_bytes(NT, J) + (size_t)K * J * 3 * sizeof(float) +
         (size_t)(3 * K + NT) * sizeof(int);
}

__global__ void __launch_bounds__(kTrackThreads) track_people_kernel(const float* __restrict__ points,
                                                                     const float* __restrict__ jmask, int T, int K, int J,
                                                                     int min_joints, double max_dist, int max_age, int NT,
                                                                     int cap, int32_t* __restrict__ state,
                                                                     int32_t* __restrict__ track_id) {
  extern __shared__ double tsm[];
  double* ecost = tsm;                                       // [cap] admissible pairs: cost
  uint16_t* epair = reinterpret_cast<uint16_t*>(ecost + cap);  //          and pair index q K + k
  int32_t* st = reinterpret_cast<int32_t*>(epair + cap);       // the state (cap >= 2 keeps it 4-byte aligned)
  const int sw = track_slot_words(J), words = 4 + NT * sw;
  uint32_t* rows = reinterpret_cast<uint32_t*>(st + words);   // [K][J][3] the frame's rows, as bits
  uint32_t* rused = rows + K * J * 3;                          // [K] used joints of row k
  int* rslot = reinterpret_cast<int*>(rused + K);              // [K] slot row k matched or was born into, -1
  int* rborn = rslot + K;                                      // [K] row k started a track this frame
  int* srow = rborn + K;                                       // [NT] row slot q matched this frame, -1
  __shared__ int nedge;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5, nt = blockDim.x;
  int32_t* gst = state + (int64_t)blockIdx.x * words;
  for (int e = tid; e < words; e += nt) st[e] = gst[e];
  __syncthreads();

  for (int t = 0; t < T; ++t) {
    const int64_t fr = (int64_t)blockIdx.x * T + t;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(points) + fr * K * J * 3;
    for (int e = tid; e < K * J * 3; e += nt) rows[e] = src[e];
    for (int q = tid; q < NT; q += nt) srow[q] = -1;
    if (tid == 0) nedge = 0;
    __syncthreads();
    // used joints: finite, and mask NULL or > 0
    if (tid < K) {
      uint32_t m = 0u;
      for (int j = 0; j < J; ++j) {
        const float* x = reinterpret_cast<const float*>(rows) + (tid * J + j) * 3;
        const bool ok = isfinite(x[0]) && isfinite(x[1]) && isfinite(x[2]) &&
                        (jmask == nullptr || jmask[fr * K * J + tid * J + j] > 0.0f);
        m |= ok ? 1u << j : 0u;
      }
      rused[tid] = m;
      rslot[tid] = -1;
      rborn[tid] = 0;
    }
    __syncthreads();

    // pair costs, one warp per (slot, row): lane j holds the joint distance, the median by rank counting across the lanes
    for (int e = warp; e < NT * K; e += nw) {
      const int q = e / K, k = e - q * K;
      const int32_t* sl = st + 4 + q * sw;
      if (sl[0] == 0) continue;
      const uint32_t shared_j = rused[k] & (uint32_t)sl[3];
      const int n = __popc(shared_j);
      if (n < min_joints) continue;                            // cost +inf
      const bool valid = (shared_j >> lane) & 1u;
      double d = 0.0;
      if (valid) {
        const float* a = reinterpret_cast<const float*>(rows) + (k * J + lane) * 3;
        const float* c = reinterpret_cast<const float*>(sl + 4) + lane * 3;
        const double dx = (double)a[0] - (double)c[0], dy = (double)a[1] - (double)c[1], dz = (double)a[2] - (double)c[2];
        // explicit roundings: no fused multiply-add, so numpy's (dx dx + dy dy) + dz dz gives the same bits
        d = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
      }
      int r = 0;
      for (int i = 0; i < 32; ++i) {
        const double di = __shfl_sync(0xffffffffu, d, i);
        r += ((shared_j >> i) & 1u) && (di < d || (di == d && i < lane));
      }
      const int i1 = (n - 1) >> 1, i2 = n >> 1;
      const double lo = __shfl_sync(0xffffffffu, d, __ffs(__ballot_sync(0xffffffffu, valid && r == i1)) - 1);
      const double hi = __shfl_sync(0xffffffffu, d, __ffs(__ballot_sync(0xffffffffu, valid && r == i2)) - 1);
      const double cost = i1 == i2 ? lo : 0.5 * (lo + hi);
      if (lane == 0 && cost <= max_dist) {
        const int x = atomicAdd(&nedge, 1);
        ecost[x] = cost;
        epair[x] = (uint16_t)e;
      }
    }
    __syncthreads();

    // bitonic sort of the admissible pairs by (cost, key), key = id K + k; padding (+inf, 0xffff) sorts last
    const int ne = nedge;
    int n2 = 1;
    while (n2 < ne) n2 <<= 1;
    for (int e = ne + tid; e < n2; e += nt) {
      ecost[e] = __longlong_as_double(0x7ff0000000000000ll);
      epair[e] = 0xffff;
    }
    __syncthreads();
    for (int k = 2; k <= n2; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = tid; i < n2; i += nt) {
          const int l = i ^ j;
          if (l <= i) continue;
          const double ci = ecost[i], cj = ecost[l];
          const uint16_t pi = epair[i], pj = epair[l];
          const int64_t ki = pi == 0xffff ? INT64_MAX : (int64_t)st[4 + (pi / K) * sw + 1] * K + pi % K;
          const int64_t kj = pj == 0xffff ? INT64_MAX : (int64_t)st[4 + (pj / K) * sw + 1] * K + pj % K;
          const bool gt = ci > cj || (ci == cj && ki > kj);
          if (gt == ((i & k) == 0)) {
            ecost[i] = cj; ecost[l] = ci;
            epair[i] = pj; epair[l] = pi;
          }
        }
        __syncthreads();
      }
    }

    // greedy matching in the sorted order
    if (tid == 0) {
      for (int e = 0; e < ne; ++e) {
        const int q = epair[e] / K, k = epair[e] - q * K;
        if (srow[q] >= 0 || rslot[k] >= 0) continue;
        srow[q] = k;
        rslot[k] = q;
      }
    }
    __syncthreads();

    // matched tracks take the row's used joints and reset their misses; unmatched live tracks age and die past max_age
    for (int e = tid; e < K * J; e += nt) {
      const int k = e / J, j = e - k * J;
      if (rslot[k] < 0 || !((rused[k] >> j) & 1u)) continue;
      uint32_t* pos = reinterpret_cast<uint32_t*>(st + 4 + rslot[k] * sw + 4) + j * 3;
      const uint32_t* x = rows + (k * J + j) * 3;
      pos[0] = x[0]; pos[1] = x[1]; pos[2] = x[2];
    }
    for (int q = tid; q < NT; q += nt) {
      int32_t* sl = st + 4 + q * sw;
      if (sl[0] == 0) continue;
      if (srow[q] >= 0) {
        sl[2] = 0;
        sl[3] = (int32_t)((uint32_t)sl[3] | rused[srow[q]]);
      } else if (++sl[2] > max_age) {
        sl[0] = 0;
      }
    }
    __syncthreads();

    // births: unmatched detections in row order take the lowest free slot and the next id
    if (tid == 0) {
      int q = 0;
      for (int k = 0; k < K; ++k) {
        if (rslot[k] >= 0 || __popc(rused[k]) < min_joints) continue;
        while (q < NT && st[4 + q * sw] != 0) ++q;
        if (q == NT) break;
        int32_t* sl = st + 4 + q * sw;
        sl[0] = 1; sl[1] = st[0]++; sl[2] = 0; sl[3] = (int32_t)rused[k];
        rslot[k] = q;
        rborn[k] = 1;
      }
    }
    __syncthreads();
    for (int e = tid; e < K * J; e += nt) {
      const int k = e / J, j = e - k * J;
      if (!rborn[k]) continue;
      uint32_t* pos = reinterpret_cast<uint32_t*>(st + 4 + rslot[k] * sw + 4) + j * 3;
      const bool u = (rused[k] >> j) & 1u;
      const uint32_t* x = rows + (k * J + j) * 3;
      pos[0] = u ? x[0] : 0u; pos[1] = u ? x[1] : 0u; pos[2] = u ? x[2] : 0u;
    }
    if (tid < K) track_id[fr * K + tid] = rslot[tid] >= 0 ? st[4 + rslot[tid] * sw + 1] : -1;
    __syncthreads();
  }
  for (int e = tid; e < words; e += nt) gst[e] = st[e];
}

int launch_track_people(const float* points, const float* joint_mask, int64_t S, int64_t T, int K, int J, int min_joints,
                        double max_dist, int max_age, int max_tracks, void* state, int32_t* track_id, cudaStream_t s) {
  const size_t smem = track_smem(max_tracks, K, J);
  MPL_CUDA(cudaFuncSetAttribute(track_people_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  track_people_kernel<<<(unsigned)S, kTrackThreads, smem, s>>>(points, joint_mask, (int)T, K, J, min_joints, max_dist,
                                                               max_age, max_tracks, track_edge_cap(max_tracks, K),
                                                               static_cast<int32_t*>(state), track_id);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

// ---- score: one warp per sequence, lane per person, integer counts, one fixed-order reduction, then acc += the counts -------
__global__ void __launch_bounds__(kTrackScoreWarps * 32, 1) tracking_score_kernel(const int32_t* __restrict__ track_id,
                                                                                  const int32_t* __restrict__ owner, int64_t S,
                                                                                  int T, int K, int P,
                                                                                  double* __restrict__ acc) {
  constexpr int kN = 8;
  __shared__ long long red[kTrackScoreWarps][kN];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  // matches, rows with an id, ID switches, fragmentations, mostly tracked, mostly lost, tracks
  long long c[kN] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int64_t s = w; s < S; s += kTrackScoreWarps) {
    const int32_t* ti = track_id + s * T * K;
    const int32_t* ow = owner + s * T * K;
    int mx = -1;
    for (int64_t e = lane; e < (int64_t)T * K; e += 32) {
      mx = max(mx, ti[e]);
      c[1] += ti[e] >= 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) c[6] += (long long)mx + 1;
    for (int q = lane; q < P; q += 32) {
      int prev = 0, last = -1, m = 0;
      bool seen = false;
      for (int t = 0; t < T; ++t) {
        int h = -1;
        for (int k = 0; k < K && h < 0; ++k)
          if (ow[t * K + k] == q && ti[t * K + k] >= 0) h = ti[t * K + k];
        if (h < 0) continue;
        ++m;
        if (seen && h != prev) ++c[2];
        if (seen && last != t - 1) ++c[3];
        seen = true;
        prev = h;
        last = t;
      }
      c[0] += m;
      c[4] += 5 * m >= 4 * T;
      c[5] += 5 * m < T;
    }
  }
#pragma unroll
  for (int q = 0; q < kN; ++q) {
    const long long t = warp_sum_ll(c[q]);
    if (lane == 0) red[w][q] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    long long tot[kN];
#pragma unroll
    for (int q = 0; q < kN; ++q) {
      tot[q] = 0;
      for (int x = 0; x < kTrackScoreWarps; ++x) tot[q] += red[x][q];
    }
    const long long objects = S * (long long)T * P;
    acc[0] += (double)S;
    acc[1] += (double)(S * (long long)T);
    acc[2] += (double)objects;
    acc[3] += (double)tot[0];
    acc[4] += (double)(objects - tot[0]);
    acc[5] += (double)(tot[1] - tot[0]);
    acc[6] += (double)tot[2];
    acc[7] += (double)tot[3];
    acc[8] += (double)tot[4];
    acc[9] += (double)tot[5];
    acc[10] += (double)tot[6];
  }
}

int launch_tracking_score(const int32_t* track_id, const int32_t* owner, int64_t S, int64_t T, int K, int P, double* acc,
                          cudaStream_t s) {
  tracking_score_kernel<<<1, kTrackScoreWarps * 32, 0, s>>>(track_id, owner, S, (int)T, K, P, acc);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

}  // namespace mpl
