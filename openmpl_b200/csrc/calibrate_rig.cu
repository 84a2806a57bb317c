// Rig calibration: Levenberg-Marquardt bundle adjustment of the V extrinsics and the 3D joints of many poses of one fixed rig,
// with a Gaussian prior on the given calibration.  The problem and the LM rules are stated in include/mpl_b200.h
// (mpl_calibrate_rig); tests/rig_calibration_oracle.py restates them in numpy.
//
// Layout of one iteration (every kernel returns at once after the stop, so a fixed sequence of launches is enqueued and the
// LM control never leaves the device):
//   rig_schur_kernel    persistent, G CTAs; applies the previous accepted point step, linearises every item of its tiles
//                       and reduces its share of the reduced camera system S = A_cc + mu I - sum_i A_ci M_i^-1 A_ic and of
//                       its right-hand side into shared memory; one partial per CTA goes to the workspace
//   rig_solve_kernel    one CTA: sums the G partials in CTA order, adds the prior and mu, dense Cholesky of S (6 V <= 96),
//                       the camera step and the candidate cameras
//   rig_cost_kernel     G2 CTAs: back-substitutes each item's point step and sums the candidate's data cost per CTA
//   rig_accept_kernel   one CTA: the candidate's cost in CTA order, accept / reject, mu, the stop test
// Determinism: no floating-point atomics; every sum has a fixed order; G and G2 depend on (B, V, J) only.
#include "kernels.cuh"
#include "so3.cuh"

namespace mpl {

constexpr int kRigThreads = 256;
constexpr int kRigTileViews = 256;    // items x views of one Schur tile: T = 256 / V items
constexpr int kRigTerms = 45;         // doubles per (item, view) in the tile: Y (3 x 6), H_cc upper (21), r (6)
constexpr int kRigRecExtra = 8;       // scalars at the end of a partial record
constexpr int kRigCostTile = 256;     // items per CTA pass of rig_cost_kernel

struct RigCtrl {
  double mu, C, Cdata, wsum, cand_prior, step_norm, cnorm, C0, Cdata0;
  int done, have_step, pending, iters, accepted, items;
  double obs;
};

struct RigCams {                      // per view: current (om, c, R, Jl), candidate (omn, cn, Rn), the camera step dc
  double om[kMaxViews][3], c[kMaxViews][3], R[kMaxViews][9], Jl[kMaxViews][9];
  double omn[kMaxViews][3], cn[kMaxViews][3], Rn[kMaxViews][9];
  double dc[6 * kMaxViews];
};

struct RigWs {
  RigCtrl* ctrl;
  RigCams* cams;
  uint32_t* used;                     // [B J] used-view mask of each item, 0 for a pair that is not an item
  double* X;                          // [B J 3] current points
  double* Xn;                         // [B J 3] candidate points
  double* part;                       // [G][rec] Schur / init partials
  double* cpart;                      // [G2] candidate data cost partials
};

static inline int rig_n(int V) { return 6 * V; }
__host__ __device__ __forceinline__ int rig_ns(int V) { return 6 * V * (6 * V + 1) / 2; }
__device__ __forceinline__ int64_t ceil_div_dev(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int rig_rec(int V) { return rig_ns(V) + rig_n(V) + kRigRecExtra; }
static inline int rig_tile(int V) { return kRigTileViews / V; }
static inline int rig_grid(int64_t items, int V) {
  const int64_t t = ceil_div(items, rig_tile(V));
  return (int)(t < kNumSMs ? t : kNumSMs);
}
static inline int rig_grid2(int64_t items) {
  const int64_t t = ceil_div(items, kRigCostTile);
  return (int)(t < 4 * kNumSMs ? t : 4 * kNumSMs);
}

static size_t rig_carve(int64_t B, int V, int J, RigWs* w, void* base) {
  const int64_t BJ = B * J;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes, 256); return o; };
  const size_t o_ctrl = take(sizeof(RigCtrl)), o_cams = take(sizeof(RigCams)), o_used = take((size_t)BJ * 4),
               o_X = take((size_t)BJ * 24), o_Xn = take((size_t)BJ * 24),
               o_part = take((size_t)rig_grid(BJ, V) * rig_rec(V) * 8), o_cpart = take((size_t)rig_grid2(BJ) * 8);
  if (w != nullptr) {
    char* b = reinterpret_cast<char*>(base);
    w->ctrl = reinterpret_cast<RigCtrl*>(b + o_ctrl);
    w->cams = reinterpret_cast<RigCams*>(b + o_cams);
    w->used = reinterpret_cast<uint32_t*>(b + o_used);
    w->X = reinterpret_cast<double*>(b + o_X);
    w->Xn = reinterpret_cast<double*>(b + o_Xn);
    w->part = reinterpret_cast<double*>(b + o_part);
    w->cpart = reinterpret_cast<double*>(b + o_cpart);
  }
  return off;
}

size_t rig_workspace_bytes(int64_t B, int V, int J) { return rig_carve(B, V, J, nullptr, nullptr); }

// One observation of X through camera (R, c, K): the residual r = pi(R (X - c)) - (u, v), the 2 x 3 Jacobians Dx = d pi / dX
// and Dw = d pi / d omega = -(d pi / dy) [y]x Jl (d pi / dc = -Dx).  Returns false where the depth y2 is not > 0 or not finite.
__device__ __forceinline__ bool rig_view(const double* R, const double* c, const double* Jl, const double* K, const double (&X)[3],
                                         double u, double v, double (&r)[2], double (&Dx)[2][3], double (&Dw)[2][3]) {
  const double d[3] = {X[0] - c[0], X[1] - c[1], X[2] - c[2]};
  double y[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) y[k] = R[3 * k] * d[0] + R[3 * k + 1] * d[1] + R[3 * k + 2] * d[2];
  if (!(y[2] > 0.0) || isinf(y[2])) return false;
  const double iz = 1.0 / y[2];
  const double px = K[0] * y[0] * iz, py = K[1] * y[1] * iz;
  r[0] = px + K[2] - u;
  r[1] = py + K[3] - v;
  // d pi / dy = [[fx iz, 0, -px iz], [0, fy iz, -py iz]]
  const double P[2][3] = {{K[0] * iz, 0.0, -px * iz}, {0.0, K[1] * iz, -py * iz}};
#pragma unroll
  for (int a = 0; a < 2; ++a) {
#pragma unroll
    for (int k = 0; k < 3; ++k) Dx[a][k] = P[a][0] * R[k] + P[a][1] * R[3 + k] + P[a][2] * R[6 + k];
    // (d pi / dy) [y]x, [y]x = [[0, -y2, y1], [y2, 0, -y0], [-y1, y0, 0]]
    const double Q[3] = {P[a][1] * y[2] - P[a][2] * y[1], P[a][2] * y[0] - P[a][0] * y[2], P[a][0] * y[1] - P[a][1] * y[0]};
#pragma unroll
    for (int k = 0; k < 3; ++k) Dw[a][k] = -(Q[0] * Jl[k] + Q[1] * Jl[3 + k] + Q[2] * Jl[6 + k]);
  }
  return true;
}

// Squared pixel error of X through (R, c, K); +inf where the depth is not > 0 or not finite.
__device__ __forceinline__ double rig_err2(const double* R, const double* c, const double* K, const double (&X)[3], double u,
                                           double v) {
  const double d[3] = {X[0] - c[0], X[1] - c[1], X[2] - c[2]};
  double y[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) y[k] = R[3 * k] * d[0] + R[3 * k + 1] * d[1] + R[3 * k + 2] * d[2];
  if (!(y[2] > 0.0) || isinf(y[2])) return __longlong_as_double(0x7ff0000000000000ll);
  const double iz = 1.0 / y[2];
  const double du = K[0] * y[0] * iz + K[2] - u, dv = K[1] * y[1] * iz + K[3] - v;
  return du * du + dv * dv;
}

// 3 x 3 Cholesky of A + mu I (A upper: 00 01 02 11 12 22) into L (l00 l10 l11 l20 l21 l22); false on a pivot that is not
// finite and > 0.
__device__ __forceinline__ bool chol3(const double (&A)[6], double mu, double (&L)[6]) {
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  const double m00 = A[0] + mu;
  if (!(m00 > 0.0 && m00 < inf)) return false;
  L[0] = sqrt(m00);
  L[1] = A[1] / L[0];
  L[3] = A[2] / L[0];
  const double m11 = A[3] + mu - L[1] * L[1];
  if (!(m11 > 0.0 && m11 < inf)) return false;
  L[2] = sqrt(m11);
  L[4] = (A[4] - L[3] * L[1]) / L[2];
  const double m22 = A[5] + mu - L[3] * L[3] - L[4] * L[4];
  if (!(m22 > 0.0 && m22 < inf)) return false;
  L[5] = sqrt(m22);
  return true;
}
__device__ __forceinline__ void fsub3(const double (&L)[6], double a0, double a1, double a2, double (&y)[3]) {  // L y = a
  y[0] = a0 / L[0];
  y[1] = (a1 - L[1] * y[0]) / L[2];
  y[2] = (a2 - L[3] * y[0] - L[4] * y[1]) / L[5];
}
__device__ __forceinline__ void bsub3(const double (&L)[6], const double (&y)[3], double (&x)[3]) {  // L^T x = y
  x[2] = y[2] / L[5];
  x[1] = (y[1] - L[4] * x[2]) / L[2];
  x[0] = (y[0] - L[1] * x[1] - L[3] * x[2]) / L[0];
}

// Index of (p, q), p <= q < n, in the row-major upper triangle.
__host__ __device__ __forceinline__ int tri_index(int p, int q, int n) { return p * n - p * (p - 1) / 2 + (q - p); }

// Fixed-order block sum of x over kRigThreads threads (valid in thread 0).  Every thread must call it.
__device__ __forceinline__ double block_sum(double x, double* red) {
  red[threadIdx.x] = x;
  __syncthreads();
  for (int s = kRigThreads / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  const double r = red[0];
  __syncthreads();
  return r;
}

// Per-view camera tables in shared memory: R (9), Jl (9), c (3), K = (fx, fy, cx, cy).
struct RigSmemCams {
  double R[kMaxViews][9], Jl[kMaxViews][9], c[kMaxViews][3], K[kMaxViews][4];
};

__device__ __forceinline__ void load_intrinsics(const double* calib, int V, RigSmemCams& sc) {
  for (int e = threadIdx.x; e < V * 4; e += blockDim.x) sc.K[e / 4][e % 4] = calib[(e / 4) * 18 + 12 + e % 4];
}

// ---- start: items, their used views, the starting cost, sum conf^2 and the diagonal of A (for mu0) -------------------------
// Grid and tiles of rig_schur_kernel.  Record: [ns, ns + n) camera diagonal of the data part of A_cc; scalars at ns + n:
// cost, sum w, items, observations, max point diagonal.
__global__ void __launch_bounds__(kRigThreads) rig_init_kernel(const float* __restrict__ pix, const double* __restrict__ calib,
                                                               int64_t B, int V, int J, float min_conf,
                                                               const int32_t* __restrict__ view_mask,
                                                               const float* __restrict__ init, double inv_s2, RigWs ws) {
  extern __shared__ __align__(16) double rsm[];
  __shared__ RigSmemCams sc;
  __shared__ double red[kRigThreads];
  const int n = 6 * V, ns = rig_ns(V), T = kRigTileViews / V;
  double* sdiag = rsm;                                   // [n] CTA sum
  double* stile = rsm + n;                               // [T][n]
  const int tid = threadIdx.x;
  for (int e = tid; e < V * 9; e += blockDim.x) {
    const int v = e / 9, k = e % 9;
    sc.R[v][k] = calib[v * 18 + k];
    sc.Jl[v][k] = (k % 4 == 0) ? 1.0 : 0.0;
  }
  for (int e = tid; e < V * 3; e += blockDim.x) sc.c[e / 3][e % 3] = calib[(e / 3) * 18 + 9 + e % 3];
  load_intrinsics(calib, V, sc);
  for (int e = tid; e < n; e += blockDim.x) sdiag[e] = 0.0;
  double cost = 0.0, wsum = 0.0, nit = 0.0, nobs = 0.0, pmax = 0.0;
  const int64_t BJ = B * J, tiles = ceil_div_dev(BJ, T);
  for (int64_t tl = blockIdx.x; tl < tiles; tl += gridDim.x) {
    __syncthreads();
    const int64_t i = tl * T + tid;
    if (tid < T) {
      double* row = stile + (size_t)tid * n;
      for (int e = 0; e < n; ++e) row[e] = 0.0;
      if (i < BJ) {
        const int64_t b = i / J;
        const int j = (int)(i - b * J);
        const double X[3] = {(double)init[i * 3], (double)init[i * 3 + 1], (double)init[i * 3 + 2]};
        unsigned m = 0;
        for (int v = 0; v < V; ++v) {
          const float* p = pix + (((b * V + v) * J) + j) * 3;
          const double u = p[0], w = p[1], wh[2] = {calib[v * 18 + 16], calib[v * 18 + 17]};
          if (p[2] > min_conf && 0.0 < u && u < wh[0] - 1.0 && 0.0 < w && w < wh[1] - 1.0) m |= 1u << v;
        }
        if (view_mask != nullptr) m &= (unsigned)view_mask[i];
        bool item = isfinite(X[0]) && isfinite(X[1]) && isfinite(X[2]) && __popc(m) >= 2;
        double ci = 0.0, wi = 0.0, A0 = 0.0, A3 = 0.0, A5 = 0.0;
        if (item) {
          for (unsigned mm = m; mm; mm &= mm - 1) {
            const int v = __ffs(mm) - 1;
            const float* p = pix + (((b * V + v) * J) + j) * 3;
            double r[2], Dx[2][3], Dw[2][3];
            if (!rig_view(sc.R[v], sc.c[v], sc.Jl[v], sc.K[v], X, p[0], p[1], r, Dx, Dw)) { item = false; break; }
            const double cf = p[2], wv = cf * cf * inv_s2;
            ci += wv * (r[0] * r[0] + r[1] * r[1]);
            wi += cf * cf;
            A0 += wv * (Dx[0][0] * Dx[0][0] + Dx[1][0] * Dx[1][0]);
            A3 += wv * (Dx[0][1] * Dx[0][1] + Dx[1][1] * Dx[1][1]);
            A5 += wv * (Dx[0][2] * Dx[0][2] + Dx[1][2] * Dx[1][2]);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
              row[6 * v + k] = wv * (Dw[0][k] * Dw[0][k] + Dw[1][k] * Dw[1][k]);
              row[6 * v + 3 + k] = wv * (Dx[0][k] * Dx[0][k] + Dx[1][k] * Dx[1][k]);   // d pi / dc = -Dx
            }
          }
        }
        if (!item) {
          m = 0;
          for (int e = 0; e < n; ++e) row[e] = 0.0;
        } else {
          cost += ci;
          wsum += wi;
          nit += 1.0;
          nobs += (double)__popc(m);
          pmax = fmax(pmax, fmax(A0, fmax(A3, A5)));
          ws.X[i * 3] = X[0];
          ws.X[i * 3 + 1] = X[1];
          ws.X[i * 3 + 2] = X[2];
        }
        ws.used[i] = m;
      }
    }
    __syncthreads();
    for (int e = tid; e < n; e += blockDim.x) {
      double s = sdiag[e];
      for (int t = 0; t < T; ++t) s += stile[(size_t)t * n + e];
      sdiag[e] = s;
    }
  }
  __syncthreads();
  double* rec = ws.part + (size_t)blockIdx.x * (ns + n + kRigRecExtra);
  for (int e = tid; e < n; e += blockDim.x) rec[ns + e] = sdiag[e];
  cost = block_sum(cost, red);
  wsum = block_sum(wsum, red);
  nit = block_sum(nit, red);
  nobs = block_sum(nobs, red);
  red[tid] = pmax;
  __syncthreads();
  if (tid == 0) {
    double mx = 0.0;
    for (int t = 0; t < kRigThreads; ++t) mx = fmax(mx, red[t]);
    double* s = rec + ns + n;
    s[0] = cost; s[1] = wsum; s[2] = nit; s[3] = nobs; s[4] = mx;
  }
}

// Camera state from omega: R = Exp(omega) R0 (R0 copied when omega is exactly 0) and Jl(omega).
__device__ __forceinline__ void rig_camera(const double* calib, int v, const double (&om)[3], double* R, double* Jl) {
  if (om[0] == 0.0 && om[1] == 0.0 && om[2] == 0.0) {
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = calib[v * 18 + k];
  } else {
    double E[9], Rn[9];
    so3_exp(om, E);
    mat3_mul(E, calib + v * 18, Rn);
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = Rn[k];
  }
  if (Jl != nullptr) {
    double L[9];
    so3_left_jacobian(om, L);
#pragma unroll
    for (int k = 0; k < 9; ++k) Jl[k] = L[k];
  }
}

__global__ void rig_init_finish_kernel(const double* __restrict__ calib, int V, int G, double inv_rot2, double inv_pos2,
                                       RigWs ws) {
  const int n = 6 * V, ns = rig_ns(V), rec = ns + n + kRigRecExtra;
  __shared__ double mxs[6 * kMaxViews];
  const int tid = threadIdx.x;
  if (tid < n) {
    double s = 0.0;
    for (int g = 0; g < G; ++g) s += ws.part[(size_t)g * rec + ns + tid];
    mxs[tid] = s + ((tid % 6) < 3 ? inv_rot2 : inv_pos2);
  }
  if (tid < V) {
    RigCams* cm = ws.cams;
    const double z[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      cm->om[tid][k] = 0.0;
      cm->c[tid][k] = calib[tid * 18 + 9 + k];
    }
    rig_camera(calib, tid, z, cm->R[tid], cm->Jl[tid]);
  }
  __syncthreads();
  if (tid == 0) {
    double cost = 0.0, wsum = 0.0, nit = 0.0, nobs = 0.0, mx = 0.0;
    for (int g = 0; g < G; ++g) {
      const double* s = ws.part + (size_t)g * rec + ns + n;
      cost += s[0]; wsum += s[1]; nit += s[2]; nobs += s[3];
      mx = fmax(mx, s[4]);
    }
    for (int e = 0; e < n; ++e) mx = fmax(mx, mxs[e]);
    RigCtrl* c = ws.ctrl;
    c->mu = 1e-3 * mx;
    c->C = c->C0 = cost;                                 // the prior is 0 at the given calibration
    c->Cdata = c->Cdata0 = cost;
    c->wsum = wsum;
    c->items = (int)nit;
    c->obs = nobs;
    c->done = nit == 0.0;
    c->have_step = c->pending = c->iters = c->accepted = 0;
    c->step_norm = c->cnorm = c->cand_prior = 0.0;
  }
}

// ---- one iteration ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kRigThreads) rig_schur_kernel(const float* __restrict__ pix, const double* __restrict__ calib,
                                                                int64_t B, int V, int J, double inv_s2, RigWs ws) {
  if (ws.ctrl->done) return;
  extern __shared__ __align__(16) double rsm[];
  __shared__ RigSmemCams sc;
  __shared__ uint32_t sused[kRigTileViews / 2];
  __shared__ int sbad;
  const int n = 6 * V, ns = rig_ns(V), T = kRigTileViews / V, tid = threadIdx.x;
  double* sacc = rsm;                                    // [ns + n]: S upper, then the RHS sum of r
  double* stile = rsm + ns + n;                          // [T][V][kRigTerms]
  int* spq = reinterpret_cast<int*>(stile + (size_t)T * V * kRigTerms);   // [ns] packed (p, q)
  const double mu = ws.ctrl->mu;
  const bool pending = ws.ctrl->pending != 0;
  for (int e = tid; e < V * 9; e += blockDim.x) {
    sc.R[e / 9][e % 9] = ws.cams->R[e / 9][e % 9];
    sc.Jl[e / 9][e % 9] = ws.cams->Jl[e / 9][e % 9];
  }
  for (int e = tid; e < V * 3; e += blockDim.x) sc.c[e / 3][e % 3] = ws.cams->c[e / 3][e % 3];
  load_intrinsics(calib, V, sc);
  for (int e = tid; e < ns + n; e += blockDim.x) sacc[e] = 0.0;
  for (int p = 0; p < n; ++p)
    for (int q = p + tid; q < n; q += blockDim.x) spq[tri_index(p, q, n)] = p | (q << 8);
  if (tid == 0) sbad = 0;
  const int64_t BJ = B * J, tiles = ceil_div_dev(BJ, T);
  for (int64_t tl = blockIdx.x; tl < tiles; tl += gridDim.x) {
    __syncthreads();
    const int64_t i = tl * T + tid;
    if (tid < T) {
      uint32_t m = i < BJ ? ws.used[i] : 0u;
      if (m) {
        const int64_t b = i / J;
        const int j = (int)(i - b * J);
        double X[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          X[k] = pending ? ws.Xn[i * 3 + k] : ws.X[i * 3 + k];
          if (pending) ws.X[i * 3 + k] = X[k];
        }
        double A[6] = {0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};
        for (unsigned mm = m; mm; mm &= mm - 1) {
          const int v = __ffs(mm) - 1;
          const float* p = pix + (((b * V + v) * J) + j) * 3;
          double r[2], Dx[2][3], Dw[2][3];
          rig_view(sc.R[v], sc.c[v], sc.Jl[v], sc.K[v], X, p[0], p[1], r, Dx, Dw);   // items: finite depth at every accepted X
          const double cf = p[2], wv = cf * cf * inv_s2;
          double* t = stile + ((size_t)tid * V + v) * kRigTerms;
          // camera Jacobian columns: omega (Dw), c (-Dx)
          double Dc[2][6];
#pragma unroll
          for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int k = 0; k < 3; ++k) { Dc[a][k] = Dw[a][k]; Dc[a][3 + k] = -Dx[a][k]; }
          int e = 0;
#pragma unroll
          for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int bb = a; bb < 3; ++bb, ++e) A[e] += wv * (Dx[0][a] * Dx[0][bb] + Dx[1][a] * Dx[1][bb]);
            g[a] += wv * (Dx[0][a] * r[0] + Dx[1][a] * r[1]);
#pragma unroll
            for (int k = 0; k < 6; ++k) t[a * 6 + k] = wv * (Dx[0][a] * Dc[0][k] + Dx[1][a] * Dc[1][k]);   // A_ic
          }
          e = 0;
#pragma unroll
          for (int a = 0; a < 6; ++a) {
#pragma unroll
            for (int bb = a; bb < 6; ++bb, ++e) t[18 + e] = wv * (Dc[0][a] * Dc[0][bb] + Dc[1][a] * Dc[1][bb]);
            t[39 + a] = wv * (Dc[0][a] * r[0] + Dc[1][a] * r[1]);                                          // g_c
          }
        }
        double L[6];
        if (!chol3(A, mu, L)) {
          sbad = 1;
          m = 0;
        } else {
          double z[3];
          fsub3(L, g[0], g[1], g[2], z);
          for (unsigned mm = m; mm; mm &= mm - 1) {
            const int v = __ffs(mm) - 1;
            double* t = stile + ((size_t)tid * V + v) * kRigTerms;
#pragma unroll
            for (int k = 0; k < 6; ++k) {
              double y[3];
              fsub3(L, t[k], t[6 + k], t[12 + k], y);      // Y = L^-1 A_ic
              t[k] = y[0];
              t[6 + k] = y[1];
              t[12 + k] = y[2];
              t[39 + k] -= y[0] * z[0] + y[1] * z[1] + y[2] * z[2];   // r = g_c - Y^T z
            }
          }
        }
      }
      sused[tid] = m;
    }
    __syncthreads();
    const int ntile = (int)(BJ - tl * T < T ? BJ - tl * T : T);
    for (int e = tid; e < ns + n; e += blockDim.x) {
      double s = sacc[e];
      if (e < ns) {
        const int pq = spq[e], p = pq & 255, q = pq >> 8;
        const int va = p / 6, pa = p - 6 * va, vb = q / 6, qb = q - 6 * vb;
        const int hidx = 18 + tri_index(pa, qb, 6);
        for (int t = 0; t < ntile; ++t) {
          const uint32_t m = sused[t];
          if (((m >> va) & (m >> vb) & 1u) == 0u) continue;
          const double* ya = stile + ((size_t)t * V + va) * kRigTerms;
          const double* yb = stile + ((size_t)t * V + vb) * kRigTerms;
          double x = -(ya[pa] * yb[qb] + ya[6 + pa] * yb[6 + qb] + ya[12 + pa] * yb[12 + qb]);
          if (va == vb) x += ya[hidx];
          s += x;
        }
      } else {
        const int p = e - ns, va = p / 6, pa = p - 6 * va;
        for (int t = 0; t < ntile; ++t)
          if ((sused[t] >> va) & 1u) s += stile[((size_t)t * V + va) * kRigTerms + 39 + pa];
      }
      sacc[e] = s;
    }
  }
  __syncthreads();
  double* rec = ws.part + (size_t)blockIdx.x * (ns + n + kRigRecExtra);
  for (int e = tid; e < ns + n; e += blockDim.x) rec[e] = sacc[e];
  if (tid == 0) rec[ns + n] = sbad;
}

constexpr int kRigSolveThreads = 512;

__global__ void __launch_bounds__(kRigSolveThreads) rig_solve_kernel(const double* __restrict__ calib, int V, int G,
                                                                     double inv_rot2, double inv_pos2, RigWs ws) {
  RigCtrl* ctrl = ws.ctrl;
  if (ctrl->done) return;
  RigCams* cm = ws.cams;
  extern __shared__ __align__(16) double Sm[];         // [n][n + 1], lower triangle
  __shared__ double rhs[6 * kMaxViews];
  __shared__ int bad;
  const int n = 6 * V, ns = rig_ns(V), rec = ns + n + kRigRecExtra, tid = threadIdx.x, ld = n + 1;
  auto S = [&](int i, int j) -> double& { return Sm[i * ld + j]; };
  const double mu = ctrl->mu;
  if (tid == 0) {
    int b = 0;
    for (int g = 0; g < G; ++g) b |= ws.part[(size_t)g * rec + ns + n] != 0.0;
    bad = b;
  }
  for (int e = tid; e < ns + n; e += blockDim.x) {
    double s = 0.0;
    for (int g = 0; g < G; ++g) s += ws.part[(size_t)g * rec + e];
    if (e < ns) {
      int p = 0;
      while (tri_index(p + 1, p + 1, n) <= e) ++p;
      const int q = p + (e - tri_index(p, p, n));
      if (p == q) s += ((p % 6) < 3 ? inv_rot2 : inv_pos2) + mu;
      S(q, p) = s;                                     // lower triangle
    } else {
      const int p = e - ns, v = p / 6, k = p % 6;
      const double gp = k < 3 ? cm->om[v][k] * inv_rot2 : (cm->c[v][k - 3] - calib[v * 18 + 9 + k - 3]) * inv_pos2;
      rhs[p] = -(s + gp);
    }
  }
  __syncthreads();
  // right-looking Cholesky S = L L^T in the lower triangle
  for (int k = 0; k < n && !bad; ++k) {
    if (tid == 0) {
      const double d = S(k, k);
      if (!(d > 0.0 && d < __longlong_as_double(0x7ff0000000000000ll))) bad = 1;
      else S(k, k) = sqrt(d);
    }
    __syncthreads();
    if (bad) break;
    const double lkk = S(k, k);
    for (int i = k + 1 + tid; i < n; i += blockDim.x) S(i, k) /= lkk;
    __syncthreads();
    const int m = n - k - 1;
    for (int e = tid; e < m * m; e += blockDim.x) {
      const int i = k + 1 + e / m, j = k + 1 + e % m;
      if (j <= i) S(i, j) -= S(i, k) * S(j, k);
    }
    __syncthreads();
  }
  __syncthreads();
  if (bad) {
    if (tid == 0) ctrl->have_step = 0;
    return;
  }
  // forward and back substitution by one warp, lane-strided dot products reduced in a fixed xor tree
  if (tid < 32) {
    for (int k = 0; k < n; ++k) {
      double s = 0.0;
      for (int j = tid; j < k; j += 32) s += S(k, j) * rhs[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (tid == 0) rhs[k] = (rhs[k] - s) / S(k, k);
      __syncwarp();
    }
    for (int k = n - 1; k >= 0; --k) {
      double s = 0.0;
      for (int j = k + 1 + tid; j < n; j += 32) s += S(j, k) * rhs[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (tid == 0) rhs[k] = (rhs[k] - s) / S(k, k);
      __syncwarp();
    }
  }
  __syncthreads();
  if (tid < n) cm->dc[tid] = rhs[tid];
  if (tid < V) {
    double om[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      om[k] = cm->om[tid][k] + rhs[6 * tid + k];
      cm->omn[tid][k] = om[k];
      cm->cn[tid][k] = cm->c[tid][k] + rhs[6 * tid + 3 + k];
    }
    rig_camera(calib, tid, om, cm->Rn[tid], nullptr);
  }
  if (tid == 0) {
    double dn = 0.0, cn = 0.0, pr = 0.0;
    for (int p = 0; p < n; ++p) dn += rhs[p] * rhs[p];
    for (int v = 0; v < V; ++v)
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        cn += cm->c[v][k] * cm->c[v][k];
        const double om = cm->om[v][k] + rhs[6 * v + k], dc = cm->c[v][k] + rhs[6 * v + 3 + k] - calib[v * 18 + 9 + k];
        pr += om * om * inv_rot2 + dc * dc * inv_pos2;
      }
    ctrl->step_norm = sqrt(dn);
    ctrl->cnorm = sqrt(cn);
    ctrl->cand_prior = pr;
    ctrl->have_step = 1;
  }
}

__global__ void __launch_bounds__(kRigThreads) rig_cost_kernel(const float* __restrict__ pix, const double* __restrict__ calib,
                                                               int64_t B, int V, int J, double inv_s2, RigWs ws) {
  const RigCtrl* ctrl = ws.ctrl;
  if (ctrl->done || !ctrl->have_step) return;
  __shared__ RigSmemCams sc;                             // current cameras: the linearisation point
  __shared__ double sRn[kMaxViews][9], scn[kMaxViews][3], sdc[6 * kMaxViews];
  __shared__ double red[kRigThreads];
  const int tid = threadIdx.x;
  for (int e = tid; e < V * 9; e += blockDim.x) {
    sc.R[e / 9][e % 9] = ws.cams->R[e / 9][e % 9];
    sc.Jl[e / 9][e % 9] = ws.cams->Jl[e / 9][e % 9];
    sRn[e / 9][e % 9] = ws.cams->Rn[e / 9][e % 9];
  }
  for (int e = tid; e < V * 3; e += blockDim.x) {
    sc.c[e / 3][e % 3] = ws.cams->c[e / 3][e % 3];
    scn[e / 3][e % 3] = ws.cams->cn[e / 3][e % 3];
  }
  for (int e = tid; e < 6 * V; e += blockDim.x) sdc[e] = ws.cams->dc[e];
  load_intrinsics(calib, V, sc);
  __syncthreads();
  const double mu = ctrl->mu;
  const int64_t BJ = B * J;
  double cost = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * kRigCostTile + tid; i < BJ; i += (int64_t)gridDim.x * kRigCostTile) {
    const uint32_t m = ws.used[i];
    if (!m) continue;
    const int64_t b = i / J;
    const int j = (int)(i - b * J);
    const double X[3] = {ws.X[i * 3], ws.X[i * 3 + 1], ws.X[i * 3 + 2]};
    double A[6] = {0, 0, 0, 0, 0, 0}, h[3] = {0, 0, 0};
    for (unsigned mm = m; mm; mm &= mm - 1) {
      const int v = __ffs(mm) - 1;
      const float* p = pix + (((b * V + v) * J) + j) * 3;
      double r[2], Dx[2][3], Dw[2][3];
      rig_view(sc.R[v], sc.c[v], sc.Jl[v], sc.K[v], X, p[0], p[1], r, Dx, Dw);
      const double cf = p[2], wv = cf * cf * inv_s2;
      const double* d = sdc + 6 * v;
      double lin[2];                                     // r + Dw d_omega - Dx d_c
#pragma unroll
      for (int a = 0; a < 2; ++a)
        lin[a] = r[a] + (Dw[a][0] * d[0] + Dw[a][1] * d[1] + Dw[a][2] * d[2]) - (Dx[a][0] * d[3] + Dx[a][1] * d[4] + Dx[a][2] * d[5]);
      int e = 0;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int bb = a; bb < 3; ++bb, ++e) A[e] += wv * (Dx[0][a] * Dx[0][bb] + Dx[1][a] * Dx[1][bb]);
        h[a] += wv * (Dx[0][a] * lin[0] + Dx[1][a] * lin[1]);
      }
    }
    double L[6], Xn[3];
    if (!chol3(A, mu, L)) {                              // not reached: rig_schur_kernel rejected the step already
      cost = __longlong_as_double(0x7ff0000000000000ll);
      continue;
    }
    double y[3], dx[3];
    fsub3(L, -h[0], -h[1], -h[2], y);
    bsub3(L, y, dx);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      Xn[k] = X[k] + dx[k];
      ws.Xn[i * 3 + k] = Xn[k];
    }
    for (unsigned mm = m; mm; mm &= mm - 1) {
      const int v = __ffs(mm) - 1;
      const float* p = pix + (((b * V + v) * J) + j) * 3;
      const double cf = p[2];
      cost += cf * cf * inv_s2 * rig_err2(sRn[v], scn[v], sc.K[v], Xn, p[0], p[1]);
    }
  }
  cost = block_sum(cost, red);
  if (tid == 0) ws.cpart[blockIdx.x] = cost;
}

__global__ void rig_accept_kernel(const double* __restrict__ calib, int V, int G2, int max_iters, RigWs ws) {
  RigCtrl* ctrl = ws.ctrl;
  if (ctrl->done) return;
  __shared__ int acc;
  const int tid = threadIdx.x;
  if (tid == 0) {
    const int k = ++ctrl->iters;
    int a = 0;
    if (ctrl->have_step) {
      double cd = 0.0;
      for (int g = 0; g < G2; ++g) cd += ws.cpart[g];
      const double cn = cd + ctrl->cand_prior;
      if (cn < ctrl->C) {
        a = 1;
        ctrl->C = cn;
        ctrl->Cdata = cd;
        ctrl->mu /= 10.0;
        ctrl->accepted += 1;
      } else {
        ctrl->mu *= 10.0;
      }
      if (ctrl->step_norm <= 1e-10 * (ctrl->cnorm + 1e-10)) ctrl->done = 1;
    } else {
      ctrl->mu *= 10.0;
    }
    ctrl->pending = a;
    if (k >= max_iters) ctrl->done = 1;
    acc = a;
  }
  __syncthreads();
  if (acc && tid < V) {
    RigCams* cm = ws.cams;
    double om[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      om[k] = cm->omn[tid][k];
      cm->om[tid][k] = om[k];
      cm->c[tid][k] = cm->cn[tid][k];
    }
    rig_camera(calib, tid, om, cm->R[tid], cm->Jl[tid]);
  }
}

__global__ void __launch_bounds__(256) rig_final_kernel(const double* __restrict__ calib, int64_t BJ, int V, const float* init,
                                                        double s2, RigWs ws, double* __restrict__ calib_out, float* points,
                                                        double* __restrict__ report) {
  const RigCtrl* ctrl = ws.ctrl;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (points != nullptr && i < BJ) {
    if (ws.used[i]) {
      const double* X = (ctrl->pending ? ws.Xn : ws.X) + i * 3;
#pragma unroll
      for (int k = 0; k < 3; ++k) points[i * 3 + k] = (float)X[k];
    } else if (points != init) {
#pragma unroll
      for (int k = 0; k < 3; ++k) points[i * 3 + k] = init[i * 3 + k];
    }
  }
  if (blockIdx.x == 0) {
    const int t = threadIdx.x;
    if (t < V) {
      const RigCams* cm = ws.cams;
      const double* c0 = calib + t * 18;
      double* o = calib_out + t * 18;
      for (int k = 0; k < 9; ++k) o[k] = cm->R[t][k];
      for (int k = 0; k < 3; ++k) o[9 + k] = cm->c[t][k];
      for (int k = 12; k < 18; ++k) o[k] = c0[k];
    }
    if (t == 0) {
      const bool any = ctrl->items > 0;
      report[0] = ctrl->items;
      report[1] = ctrl->obs;
      report[2] = ctrl->C0;
      report[3] = ctrl->C;
      report[4] = any ? sqrt(ctrl->Cdata0 * s2 / ctrl->wsum) : 0.0;
      report[5] = any ? sqrt(ctrl->Cdata * s2 / ctrl->wsum) : 0.0;
      report[6] = ctrl->iters;
      report[7] = ctrl->accepted;
    }
  }
}

static size_t rig_schur_smem(int V) {
  const int n = 6 * V, ns = rig_ns(V);
  return (size_t)(ns + n) * 8 + (size_t)rig_tile(V) * V * kRigTerms * 8 + (size_t)ns * 4;
}
static size_t rig_init_smem(int V) { return (size_t)(6 * V) * 8 * (1 + rig_tile(V)); }

int launch_calibrate_rig(const float* pix, const double* calib, int64_t B, int V, int J, float min_conf,
                         const int32_t* view_mask, const float* init, double sigma_px, double sigma_rot, double sigma_pos,
                         int max_iters, double* calib_out, float* points, double* report, void* workspace, cudaStream_t s) {
  RigWs ws;
  rig_carve(B, V, J, &ws, workspace);
  const int64_t BJ = B * J;
  const int G = rig_grid(BJ, V), G2 = rig_grid2(BJ);
  const double inv_s2 = 1.0 / (sigma_px * sigma_px), inv_rot2 = 1.0 / (sigma_rot * sigma_rot),
               inv_pos2 = 1.0 / (sigma_pos * sigma_pos);
  const size_t ss = rig_schur_smem(V), si = rig_init_smem(V), sv = (size_t)(6 * V) * (6 * V + 1) * 8;
  MPL_CUDA(cudaFuncSetAttribute(rig_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sv));
  MPL_CUDA(cudaFuncSetAttribute(rig_schur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ss));
  MPL_CUDA(cudaFuncSetAttribute(rig_init_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)si));
  rig_init_kernel<<<G, kRigThreads, si, s>>>(pix, calib, B, V, J, min_conf, view_mask, init, inv_s2, ws);
  MPL_LAUNCH_CHECK();
  rig_init_finish_kernel<<<1, 128, 0, s>>>(calib, V, G, inv_rot2, inv_pos2, ws);
  MPL_LAUNCH_CHECK();
  for (int k = 0; k < max_iters; ++k) {
    rig_schur_kernel<<<G, kRigThreads, ss, s>>>(pix, calib, B, V, J, inv_s2, ws);
    MPL_LAUNCH_CHECK();
    rig_solve_kernel<<<1, kRigSolveThreads, sv, s>>>(calib, V, G, inv_rot2, inv_pos2, ws);
    MPL_LAUNCH_CHECK();
    rig_cost_kernel<<<G2, kRigThreads, 0, s>>>(pix, calib, B, V, J, inv_s2, ws);
    MPL_LAUNCH_CHECK();
    rig_accept_kernel<<<1, 32, 0, s>>>(calib, V, G2, max_iters, ws);
    MPL_LAUNCH_CHECK();
  }
  rig_final_kernel<<<(unsigned)ceil_div(BJ, 256), 256, 0, s>>>(calib, BJ, V, init, sigma_px * sigma_px, ws, calib_out, points,
                                                               report);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

}  // namespace mpl
