// K3: the FPT projection GEMMs (QKV, proj, fc1, fc2 of multiview_mpl.py:26-36,48-66 batched over B*V rows) on the
// 5th-generation tensor cores: Y[M,N] = epilogue(A[M,K] . W[N,K]^T + bias).
//
// Persistent, warp-specialised, hand-written tcgen05 kernel:
//   warp 0     TMA producer   cp.async.bulk.tensor 2D tiles (128B swizzle) into a ring of shared-memory stages
//   warp 1     MMA issuer     one thread issues tcgen05.mma (kind::f16, bf16 / fp16 operands), accumulators in TMEM.
//                             KIND 1 ("split", the fp32-grade mode): both operands arrive as two bf16 planes, hi = bf16(x)
//                             and lo = bf16(x - hi), and every k-step issues hi.hi + hi.lo + lo.hi into the same
//                             accumulator (2^-16 relative operand error instead of 2^-9, at a third of the bf16 rate)
//   warp 2     TMEM allocator 512 columns = two 256-column accumulator stages (MMA of tile i+1 overlaps epilogue of i)
//   warps 4-11 epilogue       tcgen05.ld -> registers -> bias / GELU -> 128B-swizzled staging tile in shared memory ->
//                             TMA store (bf16 / fp32) or TMA reduce-add (the fp32 residual stream is updated in L2,
//                             never read by the SM).  Two warps per TMEM lane quarter, 64 columns per step.
//                             bf16 mode folds the LayerNorms in: LN-apply epilogues (EPI 4 / 5) for QKV / fc1 and
//                             residual-emit epilogues (EPI 6 / 7) for proj / fc2, see GemmLn below.
//   warp 3     residual producer (EPI 6 / 7 only): TMA-loads the old residual boxes (two bf16 planes) into a ring of
//                             shared-memory slots, running ahead of the epilogue warps across tile boundaries
// A CTA pair (cluster 2x1x1, cta_group::2) computes each 256 x 256 output tile, each CTA staging half of A and half of W,
// which halves the shared-memory and L2 operand traffic per MMA.
// Every FPT width is a multiple of 17 (D = 1088 = 17*64): ragged N tiles use a narrower UMMA N (multiple of 16) and
// the K tail is zero-filled by TMA, so no padding copies are needed.
#include <cuda.h>

#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <mutex>
#include <type_traits>

#include "kernels.cuh"
#include "ptx.cuh"

namespace mpl {

namespace {

constexpr int CG = 2;            // CTAs per output tile (a CTA pair)
constexpr int BM = 128;          // accumulator rows per CTA (TMEM lanes)
constexpr int BN = 256;          // accumulator columns per tile
constexpr int KB_BYTES = 128;    // bytes of K per stage row = one 128B swizzle span
constexpr int UMMA_K_BYTES = 32; // bytes of K per tcgen05.mma
// Shared-memory budget of the LayerNorm-fused bf16 kernels.  Defaults: all of shared memory.  The smaller settings (5 / 1 / 4:
// ~193 KB, room for CTAs of a light kernel beside the persistent GEMM CTA) were measured with an experimental schedule, since
// removed, that ran two pose chunks on two streams: no gain, see profiles/r2_experiments.md.
#ifndef MPL_LN_STAGES
#define MPL_LN_STAGES 6      // QKV / fc1 operand stages
#endif
#ifndef MPL_E6_SLOTS_EVEN
#define MPL_E6_SLOTS_EVEN 2  // proj: residual slots of an even-group warp
#endif
#ifndef MPL_E7_STAGES
#define MPL_E7_STAGES 5      // fc2 operand stages
#endif
constexpr int NUM_EPI_WARPS = 8;   // two per TMEM lane quarter: even / odd 64-column groups
constexpr int TMEM_COLS = 512;

template <int EPI = 0, int KIND = 0>
struct Cfg {
  static constexpr int OPS = (KIND == 1) ? 2 : 1;           // operand planes per matrix (split mode: hi + lo)
  static constexpr int A_BYTES = BM * KB_BYTES;             // 16 KB
  static constexpr int B_ROWS = BN / CG;                    // W rows staged per CTA
  static constexpr int B_BYTES = B_ROWS * KB_BYTES;         // 16 KB
  static constexpr int STAGE_BYTES = OPS * (A_BYTES + B_BYTES);  // 32 KB (split: 64 KB)
  // The residual-emit epilogues keep the old residual in TMA-fed shared-memory slots of 8 KB (a 32-row x 64-column box of each
  // bf16 plane) that are updated in place and stored back from the same slot.  Slots are PRIVATE to an epilogue warp (its
  // mbarrier phases are then observed in order by construction -- a shared ring lets a warp wait for generation n + 1 of a
  // slot whose generation n it never saw complete, and a parity wait cannot tell those apart).  A tile has 3 or 4 groups of 64
  // columns: the even-group warps always take two, the odd-group warps one or two.  The slots are paid for with operand
  // stages: the short-K proj (EPI 6) is epilogue / HBM bound -> 4 stages, two slots per even-group warp + one per odd-group
  // warp (12); the long-K fc2 (EPI 7) is MMA bound -> 5 stages, one slot per warp (8; a second group waits for its box).
  static constexpr bool RESID = (KIND == 0) && (EPI == 6 || EPI == 7);
  static constexpr int EPI_WARPS = NUM_EPI_WARPS;
  static constexpr int THREADS = (4 + EPI_WARPS) * 32;
  // Register cap.  The LayerNorm-fused bf16 kernels (the bench path) need no more than 112 registers (no spills).  The cap
  // (42 k of the SM's 64 k) was set for a since removed two-stream chunk schedule, to leave room for CTAs of a light kernel
  // beside the persistent GEMM CTA, and is kept because the shipped build is measured with it.  The other instantiations
  // take what a single CTA per SM may use.
#ifndef MPL_LN_MAXREG
#define MPL_LN_MAXREG 112
#endif
  static constexpr int MAXREG = (KIND == 0 && EPI >= 4) ? MPL_LN_MAXREG : 168;
  static constexpr int SLOTS_EVEN = !RESID ? 0 : (EPI == 6 ? MPL_E6_SLOTS_EVEN : 1);  // slots of an even-group warp (odd-group warps: 1)
  static constexpr int RING_SLOTS = !RESID ? 0 : 4 * SLOTS_EVEN + 4;
  static constexpr int SLOT_BYTES = 8192;
  static constexpr int RING_BYTES = RING_SLOTS * SLOT_BYTES;
  static constexpr int STAGES = (KIND == 1) ? 3 : (EPI == 6) ? 4 : (EPI == 7) ? MPL_E7_STAGES : (EPI >= 4 ? MPL_LN_STAGES : 6);
  static constexpr int STAGING_BYTES = RESID ? 0 : EPI_WARPS * 4096;  // per epilogue warp: one 32-row x 128-byte output box
  // slot and mbarrier phase of the n-th residual box (n = 0, 1, ...) of epilogue warp (lane quarter q, group parity `odd`)
  static constexpr uint32_t SE = SLOTS_EVEN ? SLOTS_EVEN : 1;
  __host__ __device__ static constexpr uint32_t slot_of(int q, int odd, uint32_t n) {
    return odd ? (uint32_t)(4 * SLOTS_EVEN + q) : (uint32_t)(SLOTS_EVEN * q) + n % SE;
  }
  __host__ __device__ static constexpr uint32_t phase_of(int odd, uint32_t n) { return (odd ? n : n / SE) & 1u; }
  static constexpr int BAR_BYTES = 512;
  static constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + STAGING_BYTES + RING_BYTES + BAR_BYTES;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB of shared memory a CTA may use");
};

// Output columns are dealt to T tiles in whole 64-column groups, as evenly as possible: the first r tiles take q + 1 groups,
// the others q (the last one clipped at N).  N = 1088 (17 groups) -> 256 | 256 | 192 | 192 | 192, N = 2176 -> 7 x 256 + 2 x 192:
// no narrow tail tile (a 64-wide tile costs far more than a quarter of a 256-wide one) and every tile starts on a
// 128-byte boundary of the bf16 output row.
struct TileSplit {
  int T, q, r;
};
__host__ __device__ __forceinline__ void tile_cols(const TileSplit& ts, int i, int N, int& n0, int& n_size, bool& wide) {
  wide = i < ts.r;
  n0 = 64 * (i * ts.q + (i < ts.r ? i : ts.r));
  const int w = 64 * (ts.q + (wide ? 1 : 0));
  n_size = (w < N - n0) ? w : N - n0;
}

// K-major, 128B-swizzled operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart (SBO), version 1 (sm_100)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);        // start address
  d |= (uint64_t)1 << 16;                            // leading byte offset (unused for swizzled K-major) = 1
  d |= (uint64_t)(1024 >> 4) << 32;                  // stride byte offset
  d |= (uint64_t)1 << 46;                            // descriptor version
  d |= (uint64_t)2 << 61;                            // SWIZZLE_128B
  return d;
}

// kind::f16 instruction descriptor: fp32 accumulate, K-major A and B
__device__ __forceinline__ uint32_t make_idesc(int m, int n, bool fp16 = false) {
  const uint32_t fmt = fp16 ? 0u : 1u;  // kind::f16: F16 = 0, BF16 = 1
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// EPI: 0 bias -> operand dtype (split mode: two bf16 planes), 1 bias + GELU -> operand dtype, 2 Y(fp32) += acc + bias, 3 bias -> fp32,
//      4 / 5 = 0 / 1 with LayerNorm folded in (see GemmLn), 6 / 7 residual update that also emits the next LayerNorm's inputs
//      (6: shared-memory prefetch ring of the old residual, 7: register prefetch).
//
// LayerNorm fused around the projections (bf16 mode).  LN(x) W^T + b = rstd * (x W'^T - mu * colsum(W')) + b' with
// W' = W diag(gamma), b' = b + W beta.  The residual stream x lives in HBM as TWO bf16 planes, hi = bf16(x) and
// lo = bf16(x - hi) (16 significand bits).  The consumer GEMM (QKV, fc1; EPI 4 / 5) multiplies the hi plane (the RAW
// residual rows rounded to bf16) by W' and applies the per-row (mu, rstd) in its epilogue; the producer GEMM of that
// residual (proj, fc2; EPI 6 / 7) computes x_new = hi + lo + acc + bias in its epilogue, writes both planes back in place
// (TMA in, TMA out: 8 bytes per element instead of the 12 of an fp32 stream plus a bf16 copy) and per-row partial
// (sum, sum of squares) of its column slice into a fixed slot -> no LayerNorm kernel, no atomics, bitwise reproducible.
struct GemmLn {
  const float* colsum;      // [N]  sum_k bf16(W'[n,k])                       (EPI 4 / 5)
  const float2* stats_in;   // [slots_in][stats_ld] partial (sum x, sum x^2) per row, slot-major: a warp's 32 rows of one
                            // slot are one coalesced 256-byte access                           (EPI 4 / 5)
  float2* stats_out;        // [slots_out][stats_ld]                                            (EPI 6 / 7)
  int64_t stats_ld;         // rows per slot plane (M rounded up to a multiple of 256)
  int slots_in, slots_out;
  float inv_k, eps;         // 1 / LayerNorm width (= K of the consumer), LayerNorm eps
  int flags;                // bit 1: A and W are fp16 (not bf16); bit 2: the 16-bit output is fp16 and GELU runs in packed half2
};

// accumulator chunk (32 columns of this lane's row) -> + bias (-> GELU) as fp32; LNF: LayerNorm row statistics applied
template <int KIND, int EPI>
__device__ __forceinline__ void epilogue_math(const uint32_t (&v)[32], const float* __restrict__ bias, int n, int N, float (&f)[32],
                                              const float* __restrict__ colsum = nullptr, float mu = 0.f, float rstd = 1.f) {
  // columns >= N (ragged last tile) are clipped by the TMA store; their bias reads are clamped into the array
  constexpr bool LNF = (EPI == 4 || EPI == 5);
#pragma unroll
  for (int i = 0; i < 32; i += 4) {
    const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + min(n + i, N - 4)));
    if constexpr (LNF) {
      const float4 c4 = __ldg(reinterpret_cast<const float4*>(colsum + min(n + i, N - 4)));
      f[i] = fmaf(rstd, fmaf(-mu, c4.x, __uint_as_float(v[i])), b4.x);
      f[i + 1] = fmaf(rstd, fmaf(-mu, c4.y, __uint_as_float(v[i + 1])), b4.y);
      f[i + 2] = fmaf(rstd, fmaf(-mu, c4.z, __uint_as_float(v[i + 2])), b4.z);
      f[i + 3] = fmaf(rstd, fmaf(-mu, c4.w, __uint_as_float(v[i + 3])), b4.w);
    } else {
      f[i] = __uint_as_float(v[i]) + b4.x;
      f[i + 1] = __uint_as_float(v[i + 1]) + b4.y;
      f[i + 2] = __uint_as_float(v[i + 2]) + b4.z;
      f[i + 3] = __uint_as_float(v[i + 3]) + b4.w;
    }
  }
  if constexpr (EPI == 1 || EPI == 5) {
#pragma unroll
    for (int i = 0; i < 32; ++i) f[i] = (KIND == 0) ? gelu_tanh_fit(f[i]) : gelu_erf(f[i]);  // split mode: exact erf form
  }
}

// one lane's 32 fp32 values -> its 128-byte row of a 32-row SWIZZLE_128B box (16-byte chunk j lands at j ^ (row & 7))
__device__ __forceinline__ void stage_row_f32(uint32_t box, int lane, const float (&f)[32]) {
  const uint32_t rowaddr = box + lane * 128;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    ptx::st_shared_v4(rowaddr + ((j ^ (lane & 7)) << 4), __float_as_uint(f[4 * j]), __float_as_uint(f[4 * j + 1]),
                      __float_as_uint(f[4 * j + 2]), __float_as_uint(f[4 * j + 3]));
}
// 32 fp32 values -> bf16, chunks j0 .. j0+3 of the lane's 128-byte row (a 64-column bf16 box takes two calls)
__device__ __forceinline__ void stage_row_bf16(uint32_t box, int lane, int j0, const float (&f)[32]) {
  const uint32_t rowaddr = box + lane * 128;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    __nv_bfloat162 p0 = __floats2bfloat162_rn(f[8 * j], f[8 * j + 1]);
    __nv_bfloat162 p1 = __floats2bfloat162_rn(f[8 * j + 2], f[8 * j + 3]);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(f[8 * j + 4], f[8 * j + 5]);
    __nv_bfloat162 p3 = __floats2bfloat162_rn(f[8 * j + 6], f[8 * j + 7]);
    ptx::st_shared_v4(rowaddr + (((j0 + j) ^ (lane & 7)) << 4), *reinterpret_cast<uint32_t*>(&p0),
                      *reinterpret_cast<uint32_t*>(&p1), *reinterpret_cast<uint32_t*>(&p2), *reinterpret_cast<uint32_t*>(&p3));
  }
}

// split-plane output: stores bf16(f) like stage_row_bf16 and leaves the rounding remainder f - bf16(f) in f, so a second
// call stages the lo plane
__device__ __forceinline__ void stage_row_bf16_rem(uint32_t box, int lane, int j0, float (&f)[32]) {
  const uint32_t rowaddr = box + lane * 128;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t p[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(f[8 * j + 2 * i], f[8 * j + 2 * i + 1]);
      p[i] = *reinterpret_cast<const uint32_t*>(&h);
      f[8 * j + 2 * i] -= __uint_as_float(p[i] << 16);
      f[8 * j + 2 * i + 1] -= __uint_as_float(p[i] & 0xffff0000u);
    }
    ptx::st_shared_v4(rowaddr + (((j0 + j) ^ (lane & 7)) << 4), p[0], p[1], p[2], p[3]);
  }
}

// fp16 output path (fc1 -> fc2 hidden activations kept in fp16: 3 more mantissa bits than bf16, and the GELU runs as packed
// half2 arithmetic): 32 fp32 values -> half2 pairs (saturating) -> optional tanh-fit erf-GELU -> chunks j0 .. j0+3 of the row
template <bool GELU>
__device__ __forceinline__ void stage_row_f16(uint32_t box, int lane, int j0, const float (&f)[32]) {
  const uint32_t rowaddr = box + lane * 128;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t p[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(p[i]) : "f"(f[8 * j + 2 * i + 1]), "f"(f[8 * j + 2 * i]));
      if (GELU) p[i] = gelu_tanh_fit_h2(p[i]);
    }
    ptx::st_shared_v4(rowaddr + (((j0 + j) ^ (lane & 7)) << 4), p[0], p[1], p[2], p[3]);
  }
}

template <int KIND, int EPI>
__global__ void __maxnreg__((Cfg<EPI, KIND>::MAXREG))
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmA2,
                    const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ CUtensorMap tmY2,
                    const float* __restrict__ bias, int64_t M, int N, int K, const TileSplit ts, const GemmLn ln) {
  // tmA2 / tmY2: the lo planes of the split mode (KIND 1) and of the residual stream (EPI 6 / 7).  tmB2: the lo plane of W in
  // split mode; otherwise the W box of the narrow tiles (q groups; tmB serves the wide ones, q + 1 groups)
  using C = Cfg<EPI, KIND>;
  constexpr bool SPLIT = (KIND == 1);
  constexpr bool RESID = C::RESID;
  constexpr int BK = KB_BYTES / 2;  // K elements per stage (16-bit operands)
  extern __shared__ uint8_t smem_raw[];
  // 128B-swizzled tiles need 1024-byte aligned bases
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t staging_base = smem_base + C::STAGES * C::STAGE_BYTES;  // 1024-aligned: stage sizes are multiples of 1 KB
  const uint32_t ring_base = staging_base + C::STAGING_BYTES;
  const uint32_t bar_base = ring_base + C::RING_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (C::STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * C::STAGES + 4);
  auto rfull_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + 5 + s); };
  auto rempty_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + 5 + C::RING_SLOTS + s); };
  static_assert(8 * (2 * C::STAGES + 5 + 2 * C::RING_SLOTS) <= C::BAR_BYTES, "barrier area too small");
  uint8_t* smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(
      smem_gen + C::STAGES * C::STAGE_BYTES + C::STAGING_BYTES + C::RING_BYTES + 8 * (2 * C::STAGES + 4));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = ptx::cluster_ctarank();
  const bool is_leader = cta_rank == 0;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    ptx::prefetch_tensormap(&tmY);
    ptx::prefetch_tensormap(&tmB2);
    if constexpr (SPLIT || RESID) {
      ptx::prefetch_tensormap(&tmA2);
      ptx::prefetch_tensormap(&tmY2);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      ptx::mbar_init(full_bar(s), 1);   // the leader's arrive.expect_tx covers the bytes of both CTAs of a pair
      ptx::mbar_init(empty_bar(s), 1);  // one tcgen05.commit
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(tfull_bar(s), 1);        // one tcgen05.commit
      ptx::mbar_init(tempty_bar(s), C::EPI_WARPS * CG);  // one arrive per epilogue warp of every CTA of the pair
    }
    for (int s = 0; s < C::RING_SLOTS; ++s) {
      ptx::mbar_init(rfull_bar(s), 1);   // the residual producer's arrive.expect_tx
      ptx::mbar_init(rempty_bar(s), 1);  // the consuming epilogue warp's release
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int n_tiles = ts.T;
  // W rows one CTA stages per k-block for a wide / narrow tile (split mode has no narrow box: its tmB2 is the lo plane)
  const int wide_rows = 64 * (ts.q + (ts.r > 0 ? 1 : 0)) / CG;
  const int narrow_rows = SPLIT ? wide_rows : 64 * ts.q / CG;
  const int64_t m_tiles = (M + (int64_t)BM * CG - 1) / ((int64_t)BM * CG);
  const int64_t total_tiles = m_tiles * n_tiles;
  const int64_t first_tile = blockIdx.x / CG;
  const int64_t tile_stride = gridDim.x / CG;
  const int num_kb = (K + BK - 1) / BK;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t leader_full0 = ptx::mapa(full_bar(0), 0);
      for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride) {
        const int64_t m_blk = tile / n_tiles;
        const int n_blk = (int)(tile % n_tiles);
        int nt0, n_size;
        bool wide;
        tile_cols(ts, n_blk, N, nt0, n_size, wide);
        const int32_t m0 = (int32_t)(m_blk * BM * CG + cta_rank * BM);
        const int32_t n0 = nt0 + (int32_t)cta_rank * (n_size / CG);
        const bool use_narrow = !SPLIT && !wide;
        const CUtensorMap* tb = use_narrow ? &tmB2 : &tmB;
        const uint32_t stage_tx = (uint32_t)(C::OPS * (C::A_BYTES + (use_narrow ? narrow_rows : wide_rows) * KB_BYTES));
        // The A rows of a tile come from HBM exactly once (the n-tiles of one row block run concurrently on
        // neighbouring CTAs and share them through L2).  Whoever will open the next row block pulls its A rows into
        // L2 now, one tile ahead, so those first-touch misses do not stall the operand ring.
        const int64_t next_tile = tile + tile_stride;
        const bool prefetch_next = next_tile < total_tiles && (next_tile % n_tiles) == 0;
        const int32_t next_m0 = (int32_t)((next_tile / n_tiles) * BM * CG + cta_rank * BM);
        for (int kb = 0; kb < num_kb; ++kb) {
          if (prefetch_next) {
            ptx::tma_prefetch_l2_2d(&tmA, kb * BK, next_m0);
            if constexpr (SPLIT) ptx::tma_prefetch_l2_2d(&tmA2, kb * BK, next_m0);
          }
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t a_dst = smem_base + stage * C::STAGE_BYTES;  // [A hi][A lo][W hi][W lo] in split mode
          const uint32_t b_dst = a_dst + C::OPS * C::A_BYTES;
          const uint32_t lbar = leader_full0 + 8u * stage;
          // the peer's bytes may land before this expect_tx: the phase still cannot complete without this arrive
          if (is_leader) ptx::mbar_arrive_expect_tx(full_bar(stage), 2 * stage_tx);
          ptx::tma_load_2d_pair(a_dst, &tmA, lbar, kb * BK, m0);
          ptx::tma_load_2d_pair(b_dst, tb, lbar, kb * BK, n0);
          if constexpr (SPLIT) {
            ptx::tma_load_2d_pair(a_dst + C::A_BYTES, &tmA2, lbar, kb * BK, m0);
            ptx::tma_load_2d_pair(b_dst + C::B_BYTES, &tmB2, lbar, kb * BK, n0);
          }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================== MMA issuer ========================================
    // The whole warp walks the loops convergently (barrier waits, descriptor arithmetic on warp-uniform values -> uniform
    // registers, no per-instruction ELECT / R2UR chains); one elected lane issues the tcgen05.mma / commit instructions.
    // Operand descriptors advance by adding to the 14-bit (address >> 4) field: +2 per 32-byte UMMA K step.
    if (is_leader) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint64_t desc0 = make_smem_desc(smem_base);
      for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride) {
        const int n_blk = (int)(tile % n_tiles);
        int nt0, n_size;
        bool wide;
        tile_cols(ts, n_blk, N, nt0, n_size, wide);
        const uint32_t idesc = make_idesc(BM * CG, n_size, (ln.flags & 2) != 0);
        ptx::mbar_wait(tempty_bar(acc), acc_phase ^ 1u);  // epilogue has drained this accumulator stage
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(full_bar(stage), phase);
          ptx::tc_fence_after();
          const uint64_t adesc0 = desc0 + (uint64_t)((stage * C::STAGE_BYTES) >> 4);
          const uint64_t bdesc0 = adesc0 + (uint64_t)((C::OPS * C::A_BYTES) >> 4);
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < KB_BYTES / UMMA_K_BYTES; ++k) {
              const uint64_t adesc = adesc0 + (uint64_t)(k * (UMMA_K_BYTES >> 4));
              const uint64_t bdesc = bdesc0 + (uint64_t)(k * (UMMA_K_BYTES >> 4));
              if constexpr (SPLIT) {
                // small cross terms first, the hi.hi product last (the lo.lo term, 2^-18 relative, is dropped)
                const uint64_t adesc2 = adesc + (uint64_t)(C::A_BYTES >> 4);
                const uint64_t bdesc2 = bdesc + (uint64_t)(C::B_BYTES >> 4);
                ptx::umma<0>(d_tmem, adesc, bdesc2, idesc, (kb | k) != 0 ? 1u : 0u);
                ptx::umma<0>(d_tmem, adesc2, bdesc, idesc, 1u);
                ptx::umma<0>(d_tmem, adesc, bdesc, idesc, 1u);
              } else {
                ptx::umma<0>(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
              }
            }
            ptx::umma_commit_pair(empty_bar(stage), 0x3);
            if (kb == num_kb - 1) ptx::umma_commit_pair(tfull_bar(acc), 0x3);
          }
          __syncwarp();
          if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 3) {
    // ===================================== residual producer (EPI 6 / 7) =====================
    // Boxes are requested in (tile, 64-column group g, 32-row quarter q) order, each into a slot of the epilogue warp
    // (q, g & 1) that will consume it; the producer runs as far ahead as free slots allow -- across tile boundaries, i.e. the
    // old residual of the next tile streams in while its accumulator is still being computed.
    if constexpr (RESID) {
      if (lane == 0) {
        uint32_t cnt[2] = {0u, 0u};  // boxes handed to an even- / odd-group warp so far (the same for every quarter)
        for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride) {
          const int64_t m_blk = tile / n_tiles;
          const int n_blk = (int)(tile % n_tiles);
          int nt0, n_size;
          bool wide;
          tile_cols(ts, n_blk, N, nt0, n_size, wide);
          const int ng = (n_size + 63) >> 6;
          const int32_t row_base = (int32_t)(m_blk * BM * CG + cta_rank * BM);
          for (int g = 0; g < ng; ++g) {
            const int odd = g & 1;
            const uint32_t n = cnt[odd]++;
            const uint32_t ph = C::phase_of(odd, n);
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
              const uint32_t slot = C::slot_of(q, odd, n);
              ptx::mbar_wait(rempty_bar(slot), ph ^ 1u);
              const uint32_t dst = ring_base + slot * C::SLOT_BYTES;
              ptx::mbar_arrive_expect_tx(rfull_bar(slot), C::SLOT_BYTES);
              ptx::tma_load_2d(dst, &tmY, rfull_bar(slot), nt0 + 64 * g, row_base + 32 * q);
              ptx::tma_load_2d(dst + 4096, &tmY2, rfull_bar(slot), nt0 + 64 * g, row_base + 32 * q);
            }
          }
        }
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ===================================== epilogue ==========================================
    const int q = warp & 3;            // TMEM lane quarter this warp may read (warp id % 4)
    const int half = (warp - 4) >> 2;  // 0: even 64-column groups, 1: odd groups (residual-emit: group index mod 4)
    constexpr bool OUT_BF16 = (KIND == 0) && (EPI == 0 || EPI == 1 || EPI == 4 || EPI == 5);
    constexpr bool OUT_SPLIT = SPLIT && (EPI == 0 || EPI == 1);  // two bf16 planes (hi through tmY, lo through tmY2)
    constexpr bool LNF = (EPI == 4 || EPI == 5);
    const uint32_t box = staging_base + (uint32_t)(warp - 4) * 4096u;
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t leader_tempty0 = ptx::mapa(tempty_bar(0), 0);
    uint32_t box_count = 0;  // RESID: residual boxes this warp has consumed so far (selects its slot and mbarrier phase)
    int held_slot = -1;      // RESID: slot whose TMA stores may still be reading shared memory
    for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride) {
      const int64_t m_blk = tile / n_tiles;
      const int n_blk = (int)(tile % n_tiles);
      int ncol0, n_size;
      bool wide;
      tile_cols(ts, n_blk, N, ncol0, n_size, wide);
      const int32_t row0 = (int32_t)(m_blk * BM * CG + cta_rank * BM + q * 32);  // first row of this warp's 32-row box
      const int64_t my_row = (int64_t)row0 + lane;
      const bool row_ok = my_row < M;
      float mu = 0.f, rstd = 1.f;
      if constexpr (LNF) {
        // LayerNorm statistics of this lane's row from the producer's per-slice partial sums (fixed order: reproducible)
        float s1 = 0.f, s2 = 0.f;
        if (row_ok) {
          const float2* sp = ln.stats_in + my_row;
          for (int i0 = 0; i0 < ln.slots_in; i0 += 16) {  // 16 independent loads in flight, summed in slot order
            float2 t[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) t[i] = (i0 + i < ln.slots_in) ? sp[(i0 + i) * ln.stats_ld] : make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 16; ++i) { s1 += t[i].x; s2 += t[i].y; }
          }
        }
        mu = s1 * ln.inv_k;
        rstd = rsqrtf(fmaxf(fmaf(-mu, mu, s2 * ln.inv_k), 0.f) + ln.eps);
      }
      if constexpr (RESID) {
        // Residual update x_new = (hi + lo) + acc + bias on two bf16 planes.  The old planes arrive by TMA in the ring slot
        // (128B-swizzled 32-row x 64-column boxes, so this lane's row is eight conflict-free 16-byte chunks per plane --
        // the same one-row-per-lane layout the accumulator has, no transposition); the new planes overwrite them in place
        // and leave by TMA from the same slot.  Rows past M and columns past N are zero-filled on the way in and clipped
        // on the way out by the tensor maps.  The row statistics are per-lane sums: no shuffles.
        const int ng = (n_size + 63) >> 6;
        float2 s1 = make_float2(0.f, 0.f), s2 = s1;  // (even, odd) column partial sums
        ptx::mbar_wait(tfull_bar(acc), acc_phase);
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
        for (int g = half; g < ng; g += 2, ++box_count) {
          const uint32_t slot = C::slot_of(q, half, box_count), ph = C::phase_of(half, box_count);
          if (held_slot >= 0) {  // hand the previous slot back before waiting for the next one (no hold-and-wait)
            if (lane == 0) {
              ptx::bulk_wait_read<0>();
              ptx::mbar_arrive(rempty_bar(held_slot));
            }
            held_slot = -1;
          }
          ptx::mbar_wait(rfull_bar(slot), ph);
          const uint32_t rowh = ring_base + slot * C::SLOT_BYTES + (uint32_t)lane * 128u;
          const uint32_t rowl = rowh + 4096u;
          const int gcol = ncol0 + 64 * g;
#pragma unroll
          for (int hb = 0; hb < 2; ++hb) {
            uint32_t va[32];
            ptx::tmem_ld_32x32(taddr + 64 * g + 32 * hb, va);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const int j = 4 * hb + jj;
              const int col = gcol + 8 * j;
              const uint32_t sw = (uint32_t)((j ^ (lane & 7)) << 4);
              uint32_t h[4], l[4];
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(h[0]), "=r"(h[1]), "=r"(h[2]), "=r"(h[3]) : "r"(rowh + sw));
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(l[0]), "=r"(l[1]), "=r"(l[2]), "=r"(l[3]) : "r"(rowl + sw));
              const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + min(col, N - 4)));
              const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + min(col + 4, N - 4)));
              const float2 bb[4] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y), make_float2(b1.z, b1.w)};
              // element pairs on packed f32x2 instructions (half the FADD / FFMA count of the scalar form)
              float2 v[4];
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                const float2 xo = __fadd2_rn(make_float2(__uint_as_float(h[w] << 16), __uint_as_float(h[w] & 0xffff0000u)),
                                             make_float2(__uint_as_float(l[w] << 16), __uint_as_float(l[w] & 0xffff0000u)));
                const float2 ab = __fadd2_rn(make_float2(__uint_as_float(va[8 * jj + 2 * w]), __uint_as_float(va[8 * jj + 2 * w + 1])), bb[w]);
                v[w] = __fadd2_rn(ab, xo);
              }
              if (col < N) {  // (whole 8-column chunks: N % 8 == 0) columns past N carry stale accumulator values
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                  s1 = __fadd2_rn(s1, v[w]);
                  s2 = __ffma2_rn(v[w], v[w], s2);
                }
              }
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                const __nv_bfloat162 hh = __float22bfloat162_rn(v[w]);
                h[w] = *reinterpret_cast<const uint32_t*>(&hh);
                const float2 rem = __fadd2_rn(v[w], make_float2(-__uint_as_float(h[w] << 16), -__uint_as_float(h[w] & 0xffff0000u)));
                const __nv_bfloat162 ll = __float22bfloat162_rn(rem);
                l[w] = *reinterpret_cast<const uint32_t*>(&ll);
              }
              ptx::st_shared_v4(rowh + sw, h[0], h[1], h[2], h[3]);
              ptx::st_shared_v4(rowl + sw, l[0], l[1], l[2], l[3]);
            }
          }
          ptx::fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            ptx::tma_store_2d(&tmY, ring_base + slot * C::SLOT_BYTES, gcol, row0);
            ptx::tma_store_2d(&tmY2, ring_base + slot * C::SLOT_BYTES + 4096u, gcol, row0);
            ptx::bulk_commit();
          }
          held_slot = (int)slot;
        }
        if (held_slot >= 0) {  // nothing is held across tiles: the producer prefetches the next tile's boxes meanwhile
          if (lane == 0) {
            ptx::bulk_wait_read<0>();
            ptx::mbar_arrive(rempty_bar(held_slot));
          }
          held_slot = -1;
        }
        // per-row partial statistics of this warp's column slice (rows past M land in the padding of the slot plane)
        ln.stats_out[(2 * n_blk + half) * ln.stats_ld + my_row] = make_float2(s1.x + s1.y, s2.x + s2.y);
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_cluster(leader_tempty0 + 8u * acc);
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        continue;
      }
      ptx::mbar_wait(tfull_bar(acc), acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
      for (int c = half * 64; c < n_size; c += 128) {
        if constexpr (OUT_BF16) {
          // one 64-column bf16 box per step, filled in two 32-column halves (one accumulator chunk in registers at a time:
          // ~100 registers per thread, see Cfg::MAXREG)
          constexpr bool GELU = (EPI == 1 || EPI == 5);
          const bool f16_out = (ln.flags & 4) != 0;
          if (lane == 0) ptx::bulk_wait_read<0>();  // the previous store has finished reading the box
          __syncwarp();
#pragma unroll
          for (int hb = 0; hb < 2; ++hb) {
            uint32_t va[32];
            ptx::tmem_ld_32x32(taddr + c + 32 * hb, va);
            ptx::tmem_ld_wait();
            float fa[32];
            if (GELU && f16_out) {  // activation deferred to the packed-half2 stage
              epilogue_math<KIND, EPI == 5 ? 4 : 0>(va, bias, ncol0 + c + 32 * hb, N, fa, ln.colsum, mu, rstd);
              stage_row_f16<GELU>(box, lane, 4 * hb, fa);
            } else {
              epilogue_math<KIND, EPI>(va, bias, ncol0 + c + 32 * hb, N, fa, ln.colsum, mu, rstd);
              if (f16_out) stage_row_f16<false>(box, lane, 4 * hb, fa);
              else stage_row_bf16(box, lane, 4 * hb, fa);
            }
          }
          ptx::fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            ptx::tma_store_2d(&tmY, box, ncol0 + c, row0);
            ptx::bulk_commit();
          }
          continue;
        }
        uint32_t va[32], vb[32];
        ptx::tmem_ld_32x32(taddr + c, va);
        ptx::tmem_ld_32x32(taddr + c + 32, vb);
        ptx::tmem_ld_wait();
        if constexpr (OUT_SPLIT) {
          // one 64-column group per step, as two bf16 boxes: hi plane, then the rounding remainder as the lo plane
          float fa[32], fb[32];
          epilogue_math<KIND, EPI>(va, bias, ncol0 + c, N, fa);
          epilogue_math<KIND, EPI>(vb, bias, ncol0 + c + 32, N, fb);
#pragma unroll
          for (int plane = 0; plane < 2; ++plane) {
            if (lane == 0) ptx::bulk_wait_read<0>();  // the previous store has finished reading the box
            __syncwarp();
            stage_row_bf16_rem(box, lane, 0, fa);
            stage_row_bf16_rem(box, lane, 4, fb);
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              ptx::tma_store_2d(plane ? &tmY2 : &tmY, box, ncol0 + c, row0);
              ptx::bulk_commit();
            }
          }
        } else {
          // two 32-column fp32 boxes per step, one after the other through the same staging box
#pragma unroll
          for (int hbox = 0; hbox < 2; ++hbox) {
            if (c + 32 * hbox >= n_size) break;
            float f[32];
            epilogue_math<KIND, EPI>(hbox ? vb : va, bias, ncol0 + c + 32 * hbox, N, f);
            if (lane == 0) ptx::bulk_wait_read<0>();
            __syncwarp();
            stage_row_f32(box, lane, f);
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              if constexpr (EPI == 2) ptx::tma_reduce_add_2d(&tmY, box, ncol0 + c + 32 * hbox, row0);
              else ptx::tma_store_2d(&tmY, box, ncol0 + c + 32 * hbox, row0);
              ptx::bulk_commit();
            }
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_cluster(leader_tempty0 + 8u * acc);
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (lane == 0) ptx::bulk_wait_all();  // every output tile has landed before the CTA retires
    __syncwarp();
  }

  ptx::tc_fence_before();
  ptx::cluster_sync();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, TMEM_COLS);
  }
}


// =====================================================================================================================
// QKV projection + cross-view attention in ONE kernel (bf16 mode, LayerNorm folded, view tokens with hd = 136, V = 2 .. 8)
// -- multiview_mpl.py:48-64.  The q|k|v tensor (6.5 KB per row, written and re-read once per block application: a quarter
// of all DRAM traffic of the step) never exists: an output tile is one HEAD of 256 rows, 3 * 136 + 8 = 416 accumulator
// columns [q | k | v | pad] (W rows permuted / zero-padded per head at pack time and stored so that each CTA of the pair
// reads its 208 rows contiguously; two N = 208 UMMAs per K step).  The V views of a pose are V adjacent TMEM lanes = V
// adjacent lanes of an epilogue warp.  Epilogue of a warp (lane quarter, half of the head dims):
//   A  read q, k, v of its dims out of TMEM, apply the folded LayerNorm + bias, keep q in registers (bf16 pairs; the softmax
//      scale * log2 e is folded into the q rows of W), park k and v in shared memory (bf16) -> the accumulator is RELEASED
//      here, the next tile's MMAs run under everything below;
//   B  partial scores of its dims: every lane reads the k rows of the V views of ITS pose (the V lanes of a pose read the
//      same address: one broadcast wavefront per load), packed f32x2 FMAs; the two warps of a quarter exchange the partial
//      sums through shared memory (64-thread named barrier); softmax over the V keys in registers;
//   C  o = sum_j p_j v_j for its dims, bf16, into the (now free) k rows of the quarter;
//   D  one TMA store of the quarter's 32 x 136 output box.
// =====================================================================================================================
constexpr int FA_HD = 136, FA_NT = 416, FA_UW = 208;         // head dim, padded q|k|v tile width, UMMA N
constexpr int FA_B_ROWS = FA_NT / 2;                          // W rows per CTA and stage
constexpr int FA_A_BYTES = BM * KB_BYTES, FA_B_BYTES = FA_B_ROWS * KB_BYTES;
constexpr int FA_STAGE_BYTES = FA_A_BYTES + FA_B_BYTES;       // 43 008
constexpr int FA_STAGES = 3;
constexpr int FA_PITCH = FA_HD * 2;                           // bytes per row of the output box, and of the k / v rows for hd = 136 (272)
constexpr int FA_PITCH2 = 288;                                // k / v row pitch for hd = 68: two heads at byte offsets 0 and 144
constexpr int FA_KV_BYTES = 2 * BM * FA_PITCH2;               // k rows then v rows of the CTA's 128 rows
constexpr int FA_D0 = 72;                                     // dims of epilogue half 0 ([0, 72)); half 1 takes [72, 136)
constexpr int FA_PART_BYTES = 2 * BM * 8 * 4;                 // partial scores [half][row][<= 8 views]
constexpr int FA_BC_WARP_BYTES = 3 * FA_D0 * 8;               // per epilogue warp: (bias, colsum) of its 3 x 72 columns of the head
constexpr int FA_BC_BYTES = NUM_EPI_WARPS * FA_BC_WARP_BYTES;
constexpr int FA_SMEM_BYTES = 1024 + FA_STAGES * FA_STAGE_BYTES + FA_KV_BYTES + FA_PART_BYTES + FA_BC_BYTES + 256;
static_assert(FA_STAGE_BYTES % 1024 == 0 && FA_SMEM_BYTES <= 232448, "fused QKV + attention kernel: shared-memory budget");

struct FusedAttnArgs {
  const float* bias;       // [H * 416] folded bias, logical column order [q | k | v | pad] per head
  const float* colsum;     // [H * 416]
  const float2* stats;     // [slots][stats_ld]
  int64_t stats_ld;
  int slots;
  float inv_k, eps;
  int64_t M;
  int K, H;
};

__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// HD = 136: a tile is one head, the two epilogue warps of a lane quarter split its dims 72 / 64 and exchange partial scores.
// HD = 68 (the "chosen" architecture, D = 544): a tile is a PAIR of heads -- accumulator columns [208 e, 208 e + 204) = q | k | v
// of head 2 t + e, one N = 208 UMMA each -- and the two epilogue warps of a quarter take one head each, all 68 dims.
template <int V, int HD>
__global__ void __launch_bounds__(NUM_EPI_WARPS * 32 + 128, 1)
qkv_attn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmO, const FusedAttnArgs a) {
  // The views of a pose are adjacent lanes of one warp (= 32 TMEM lanes = one quarter of the CTA's rows): a quarter holds
  // PQ whole poses = RQ rows.  V = 2, 4, 8 fill it; for the other view counts the row tiling is pose aligned instead of
  // 128 aligned: every quarter is its own 32-row TMA box starting RQ rows after the previous one, its last 32 - RQ rows
  // (and lanes) are the first rows of the next quarter again and are ignored.
  static_assert(V >= 2 && V <= 8, "2 to 8 views");
  static_assert(HD == 136 || HD == 68, "136-wide heads, or pairs of 68-wide heads");
  constexpr int PQ = 32 / V, RQ = PQ * V;
  constexpr bool PAIR = HD == 68;
  constexpr int KVP = PAIR ? FA_PITCH2 : FA_PITCH;  // bytes per k / v row
  constexpr int BK = KB_BYTES / 2;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t kv_base = smem_base + FA_STAGES * FA_STAGE_BYTES;  // k rows [128][272 B], then v rows
  const uint32_t part_base = kv_base + FA_KV_BYTES;
  const uint32_t bc_base = part_base + FA_PART_BYTES;
  const uint32_t bar_base = bc_base + FA_BC_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (FA_STAGES + s); };
  const uint32_t tfull_bar = bar_base + 8u * (2 * FA_STAGES);
  const uint32_t tempty_bar = bar_base + 8u * (2 * FA_STAGES + 1);
  const uint32_t tmem_slot = bar_base + 8u * (2 * FA_STAGES + 2);
  uint8_t* smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(
      smem_gen + FA_STAGES * FA_STAGE_BYTES + FA_KV_BYTES + FA_PART_BYTES + FA_BC_BYTES + 8 * (2 * FA_STAGES + 2));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = ptx::cluster_ctarank();
  const bool is_leader = cta_rank == 0;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    ptx::prefetch_tensormap(&tmO);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < FA_STAGES; ++s) {
      ptx::mbar_init(full_bar(s), 1);
      ptx::mbar_init(empty_bar(s), 1);
    }
    ptx::mbar_init(tfull_bar, 1);
    ptx::mbar_init(tempty_bar, NUM_EPI_WARPS * 2);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int64_t m_tiles = (a.M + 8 * RQ - 1) / (8 * RQ);
  const int64_t total_tiles = m_tiles * a.H;
  const int64_t first_tile = blockIdx.x / 2, tile_stride = gridDim.x / 2;
  const int num_kb = (a.K + BK - 1) / BK;

  if (warp == 0) {
    // ---- TMA producer: A rows of this CTA (4 quarters x 32 rows x 64 K elements) + its 208 W rows of the head ----
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t leader_full0 = ptx::mapa(full_bar(0), 0);
      for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride) {
        const int64_t m_blk = tile / a.H;
        const int head = (int)(tile % a.H);
        const int32_t m0 = (int32_t)((m_blk * 2 + cta_rank) * 4 * RQ);
        const int32_t n0 = head * FA_NT + (int32_t)cta_rank * FA_B_ROWS;
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t a_dst = smem_base + stage * FA_STAGE_BYTES, b_dst = a_dst + FA_A_BYTES;
          const uint32_t lbar = leader_full0 + 8u * stage;
          if (is_leader) ptx::mbar_arrive_expect_tx(full_bar(stage), 2 * FA_STAGE_BYTES);
          if constexpr (RQ == 32) {
            ptx::tma_load_2d_pair(a_dst, &tmA, lbar, kb * BK, m0);
          } else {
#pragma unroll
            for (int q = 0; q < 4; ++q)  // 32-row boxes: whole swizzle atoms of 8 rows, the same layout as one 128-row box
              ptx::tma_load_2d_pair(a_dst + (uint32_t)(q * 32 * KB_BYTES), &tmA, lbar, kb * BK, m0 + q * RQ);
          }
          ptx::tma_load_2d_pair(b_dst, &tmB, lbar, kb * BK, n0);
          if (++stage == FA_STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---- MMA issuer: two N = 208 UMMAs per K step into the single 416-column accumulator ----
    if (is_leader) {
      int stage = 0;
      uint32_t phase = 0, acc_phase = 0;
      const uint64_t desc0 = make_smem_desc(smem_base);
      const uint32_t idesc = make_idesc(2 * BM, FA_UW);
      for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride) {
        ptx::mbar_wait(tempty_bar, acc_phase ^ 1u);  // the epilogue warps have read the previous tile out of TMEM
        ptx::tc_fence_after();
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(full_bar(stage), phase);
          ptx::tc_fence_after();
          const uint64_t adesc0 = desc0 + (uint64_t)((stage * FA_STAGE_BYTES) >> 4);
          const uint64_t bdesc0 = adesc0 + (uint64_t)(FA_A_BYTES >> 4);
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < KB_BYTES / UMMA_K_BYTES; ++k) {
#pragma unroll
              for (int u = 0; u < 2; ++u)  // W rows [104 u, 104 u + 104) of both CTAs = accumulator columns [208 u, 208 u + 208)
                ptx::umma<0>(tmem_base + (uint32_t)(u * FA_UW), adesc0 + (uint64_t)(k * (UMMA_K_BYTES >> 4)),
                             bdesc0 + (uint64_t)(k * (UMMA_K_BYTES >> 4) + u * ((FA_UW / 2 * KB_BYTES) >> 4)), idesc,
                             (kb | k) != 0 ? 1u : 0u);
            }
            ptx::umma_commit_pair(empty_bar(stage), 0x3);
            if (kb == num_kb - 1) ptx::umma_commit_pair(tfull_bar, 0x3);
          }
          __syncwarp();
          if (++stage == FA_STAGES) { stage = 0; phase ^= 1u; }
        }
        acc_phase ^= 1u;
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ---- epilogue ----
    const int q4 = warp & 3, half = (warp - 4) >> 2;
    // dims [d_lo, d_lo + nd) of the head this warp works on: nchunks whole 8-dim chunks (+ a 4-dim tail for 68-wide heads)
    const int d_lo = (!PAIR && half) ? FA_D0 : 0;
    const int nd = PAIR ? 68 : (half ? FA_HD - FA_D0 : FA_D0), nchunks = nd / 8;
    const uint32_t cbase = PAIR ? (uint32_t)(half * FA_UW) : 0u;  // accumulator column of the head
    const uint32_t hoff = PAIR ? (uint32_t)(half * (FA_PITCH2 / 2)) : 0u;  // byte offset of the head inside a k / v row
    const int lrow = q4 * 32 + lane;                       // CTA-local row of this lane
    const int prow0 = q4 * 32 + min(lane / V, PQ - 1) * V;  // first row (view 0) of this lane's pose (lanes >= RQ: idle)
    const uint32_t k_row = kv_base + (uint32_t)lrow * KVP + hoff, v_row = k_row + BM * KVP;
    const uint32_t k_pose = kv_base + (uint32_t)prow0 * KVP + hoff, v_pose = k_pose + BM * KVP;
    // the quarter's dense output box (RQ rows of 272 B) takes the place of its k rows once the scores are done
    const uint32_t o_box = kv_base + (uint32_t)(q4 * 32) * KVP;
    const uint32_t o_row = o_box + (uint32_t)lane * FA_PITCH + (PAIR ? (uint32_t)(half * HD * 2) : 0u);
    const uint32_t leader_tempty = ptx::mapa(tempty_bar, 0);
    uint32_t acc_phase = 0;
    for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride) {
      const int64_t m_blk = tile / a.H;
      const int head = (int)(tile % a.H);
      const int32_t row0 = (int32_t)(((m_blk * 2 + cta_rank) * 4 + q4) * RQ);
      const int64_t my_row = (int64_t)row0 + lane;
      float mu = 0.f, rstd = 1.f;
      {
        float s1 = 0.f, s2 = 0.f;
        if (lane < RQ && my_row < a.M) {
          const float2* sp = a.stats + my_row;
          for (int i = 0; i < a.slots; ++i) { const float2 t = sp[i * a.stats_ld]; s1 += t.x; s2 += t.y; }
        }
        mu = s1 * a.inv_k;
        rstd = rsqrtf(fmaxf(fmaf(-mu, mu, s2 * a.inv_k), 0.f) + a.eps);
      }
      // (bias, colsum) of this warp's 3 x nd columns of the head -> its shared-memory scratch, while the MMAs of the tile run
      // (the accumulator is single-buffered: everything between its completion and its release is serial time)
      const uint32_t bc = bc_base + (uint32_t)(warp - 4) * FA_BC_WARP_BYTES;
      for (int idx = lane; idx < 3 * nd / 2; idx += 32) {  // per pair of dims: (bias d, bias d+1, colsum d, colsum d+1)
        const int part = idx / (nd / 2), d = 2 * (idx - part * (nd / 2));
        const int n = head * FA_NT + (int)cbase + part * HD + d_lo + d;
        const float2 b2 = __ldg(reinterpret_cast<const float2*>(a.bias + n)), c2 = __ldg(reinterpret_cast<const float2*>(a.colsum + n));
        ptx::st_shared_v4(bc + (uint32_t)idx * 16u, __float_as_uint(b2.x), __float_as_uint(b2.y), __float_as_uint(c2.x), __float_as_uint(c2.y));
      }
      // the previous tile's output box (it lives in the k rows of this quarter) has left shared memory
      if (half == 0 && lane == 0) ptx::bulk_wait_read<0>();
      named_bar_sync(1 + q4, 64);
      ptx::mbar_wait(tfull_bar, acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16);
      // ---- A: TMEM -> folded LayerNorm + bias -> q in registers, k / v rows in shared memory (bf16) ----
      const float2 rstd2 = make_float2(rstd, rstd), nmu2 = make_float2(-mu, -mu);
      uint32_t qreg[FA_D0 / 2];
#pragma unroll
      for (int part = 0; part < 3; ++part) {
        uint32_t r0[32], r1[32], r2[8];
        const uint32_t col0 = cbase + (uint32_t)(part * HD + d_lo);
        ptx::tmem_ld_32x32(taddr + col0, r0);
        ptx::tmem_ld_32x32(taddr + col0 + 32, r1);
        if constexpr (PAIR) {
          ptx::tmem_ld_32x4(taddr + col0 + 64, r2);
        } else {
          if (half == 0) ptx::tmem_ld_32x8(taddr + col0 + 64, r2);
        }
        ptx::tmem_ld_wait();
        // NP dim pairs starting at dim 8 c: LayerNorm-apply, bias, bf16 pairs (packed f32x2 arithmetic)
        auto chunk = [&](const uint32_t* r, int c, auto np) {
          constexpr int NP = decltype(np)::value;
          uint32_t w[NP];
#pragma unroll
          for (int i = 0; i < NP; ++i) {
            float4 t;  // (bias d, bias d+1, colsum d, colsum d+1) of dims d = 2i, 2i + 1 of the chunk
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(t.x), "=f"(t.y), "=f"(t.z), "=f"(t.w)
                         : "r"(bc + (uint32_t)((part * nd + 8 * c + 2 * i) * 8)));
            const float2 acc2 = make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
            const float2 f2v = __ffma2_rn(rstd2, __ffma2_rn(nmu2, make_float2(t.z, t.w), acc2), make_float2(t.x, t.y));
            const __nv_bfloat162 p = __float22bfloat162_rn(f2v);
            w[i] = *reinterpret_cast<const uint32_t*>(&p);
          }
          if (part == 0) {
#pragma unroll
            for (int i = 0; i < NP; ++i) qreg[4 * c + i] = w[i];
          } else {
            const uint32_t dst = (part == 1 ? k_row : v_row) + (uint32_t)(d_lo + 8 * c) * 2u;
            if constexpr (NP == 4) ptx::st_shared_v4(dst, w[0], w[1], w[2], w[3]);
            else ptx::st_shared_v2(dst, w[0], w[1]);
          }
        };
#pragma unroll
        for (int c = 0; c < 4; ++c) chunk(&r0[8 * c], c, std::integral_constant<int, 4>{});
#pragma unroll
        for (int c = 0; c < 4; ++c) chunk(&r1[8 * c], 4 + c, std::integral_constant<int, 4>{});
        if constexpr (PAIR) {
          chunk(r2, 8, std::integral_constant<int, 2>{});
        } else {
          if (half == 0) chunk(r2, 8, std::integral_constant<int, 4>{});
        }
      }
      // the accumulator is free: the next tile's MMAs run under the rest of this epilogue
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_cluster(leader_tempty);
      acc_phase ^= 1u;
      // ---- B: (partial) scores over this warp's dims ----
      float2 s2[V];
#pragma unroll
      for (int j = 0; j < V; ++j) s2[j] = make_float2(0.f, 0.f);
      auto bf_lo = [](uint32_t w) { return __uint_as_float(w << 16); };
      auto bf_hi = [](uint32_t w) { return __uint_as_float(w & 0xffff0000u); };
#pragma unroll
      for (int c = 0; c < FA_D0 / 8; ++c) {
        if (c < nchunks) {
          float2 q2[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) q2[i] = make_float2(bf_lo(qreg[4 * c + i]), bf_hi(qreg[4 * c + i]));
#pragma unroll
          for (int j = 0; j < V; ++j) {
            uint32_t kw[4];
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(kw[0]), "=r"(kw[1]), "=r"(kw[2]), "=r"(kw[3])
                         : "r"(k_pose + (uint32_t)j * KVP + (uint32_t)(d_lo + 8 * c) * 2u));
#pragma unroll
            for (int i = 0; i < 4; ++i) s2[j] = __ffma2_rn(q2[i], make_float2(bf_lo(kw[i]), bf_hi(kw[i])), s2[j]);
          }
        }
      }
      if constexpr (PAIR) {  // dims 64 .. 67
        float2 q2[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) q2[i] = make_float2(bf_lo(qreg[32 + i]), bf_hi(qreg[32 + i]));
#pragma unroll
        for (int j = 0; j < V; ++j) {
          uint32_t kw[2];
          asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(kw[0]), "=r"(kw[1]) : "r"(k_pose + (uint32_t)j * KVP + 128u));
#pragma unroll
          for (int i = 0; i < 2; ++i) s2[j] = __ffma2_rn(q2[i], make_float2(bf_lo(kw[i]), bf_hi(kw[i])), s2[j]);
        }
      }
      float p[V];
      if constexpr (!PAIR) {
        const uint32_t mine = part_base + (uint32_t)((half * BM + lrow) * 8) * 4u;
#pragma unroll
        for (int j = 0; j < V; ++j) asm volatile("st.shared.f32 [%0], %1;" ::"r"(mine + 4u * j), "f"(s2[j].x + s2[j].y) : "memory");
      }
      named_bar_sync(1 + q4, 64);  // both warps of the quarter are done reading its k rows (and the partial sums are in place)
      {
        float mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < V; ++j) {
          if constexpr (PAIR) {
            p[j] = s2[j].x + s2[j].y;
          } else {
            float s0, s1;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(s0) : "r"(part_base + (uint32_t)((lrow) * 8 + j) * 4u));
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(s1) : "r"(part_base + (uint32_t)((BM + lrow) * 8 + j) * 4u));
            p[j] = s0 + s1;  // fixed order: bitwise the same in both warps
          }
          mx = fmaxf(mx, p[j]);
        }
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < V; ++j) { p[j] = exp2f(p[j] - mx); sum += p[j]; }
        const float inv = 1.0f / sum;
#pragma unroll
        for (int j = 0; j < V; ++j) p[j] *= inv;
      }
      // ---- C: o = sum_j p_j v_j over this warp's dims, into the quarter's output box (its k rows: free since the barrier) ----
#pragma unroll
      for (int c = 0; c < FA_D0 / 8; ++c) {
        if (c < nchunks) {
          float2 o2[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) o2[i] = make_float2(0.f, 0.f);
#pragma unroll
          for (int j = 0; j < V; ++j) {
            uint32_t vw[4];
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(vw[0]), "=r"(vw[1]), "=r"(vw[2]), "=r"(vw[3])
                         : "r"(v_pose + (uint32_t)j * KVP + (uint32_t)(d_lo + 8 * c) * 2u));
            const float2 pj = make_float2(p[j], p[j]);
#pragma unroll
            for (int i = 0; i < 4; ++i) o2[i] = __ffma2_rn(pj, make_float2(bf_lo(vw[i]), bf_hi(vw[i])), o2[i]);
          }
          uint32_t w[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const __nv_bfloat162 t = __float22bfloat162_rn(o2[i]);
            w[i] = *reinterpret_cast<const uint32_t*>(&t);
          }
          const uint32_t dst = o_row + (uint32_t)(d_lo + 8 * c) * 2u;
          if constexpr (PAIR) {  // head 1 starts 136 B into the row: 8-byte aligned only
            ptx::st_shared_v2(dst, w[0], w[1]);
            ptx::st_shared_v2(dst + 8u, w[2], w[3]);
          } else {
            ptx::st_shared_v4(dst, w[0], w[1], w[2], w[3]);
          }
        }
      }
      if constexpr (PAIR) {  // dims 64 .. 67
        float2 o2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
        for (int j = 0; j < V; ++j) {
          uint32_t vw[2];
          asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(vw[0]), "=r"(vw[1]) : "r"(v_pose + (uint32_t)j * KVP + 128u));
          const float2 pj = make_float2(p[j], p[j]);
#pragma unroll
          for (int i = 0; i < 2; ++i) o2[i] = __ffma2_rn(pj, make_float2(bf_lo(vw[i]), bf_hi(vw[i])), o2[i]);
        }
        const __nv_bfloat162 t0 = __float22bfloat162_rn(o2[0]), t1 = __float22bfloat162_rn(o2[1]);
        ptx::st_shared_v2(o_row + 128u, *reinterpret_cast<const uint32_t*>(&t0), *reinterpret_cast<const uint32_t*>(&t1));
      }
      // ---- D: the quarter's RQ x 136 output box leaves by TMA ----
      ptx::fence_proxy_async();
      named_bar_sync(1 + q4, 64);
      if (half == 0 && lane == 0) {
        ptx::tma_store_2d(&tmO, o_box, head * FA_HD, row0);
        ptx::bulk_commit();
      }
    }
    if (half == 0 && lane == 0) ptx::bulk_wait_all();
    __syncwarp();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// pack: W [3D, D] fp32, LayerNorm gamma / beta folded, q rows scaled by qscale -> W'' [tiles * 416, D] bf16 in the PHYSICAL row
// order of the kernel (per tile: CTA 0 rows {[0,104) | [208,312)}, CTA 1 rows {[104,208) | [312,416)} of the logical column
// order), colsum / bias [tiles * 416] fp32 in LOGICAL order.  Logical columns of a tile: hd = 136: [q | k | v | 8 pad] of head
// t; hd = 68: [q | k | v | 4 pad] of head 2 t, then the same of head 2 t + 1.
__global__ void __launch_bounds__(256) qkv_attn_pack_kernel(const float* __restrict__ W, const float* __restrict__ b,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           __nv_bfloat16* __restrict__ Wp, float* __restrict__ colsum,
                                                           float* __restrict__ bias_f, int tiles, int HD, int D, float qscale,
                                                           const int* __restrict__ kperm) {
  const int pr = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // physical row
  if (pr >= tiles * FA_NT) return;
  const int lane = threadIdx.x & 31;
  const int tile = pr / FA_NT, within = pr % FA_NT;
  const int r = within / (FA_NT / 2), rem = within % (FA_NT / 2);
  const int u = rem / (FA_UW / 2), i = rem % (FA_UW / 2);
  const int logical = u * FA_UW + r * (FA_UW / 2) + i;
  int part, d, head;
  if (HD == FA_HD) {
    part = logical / FA_HD, d = logical % FA_HD, head = tile;
  } else {
    const int e = logical / FA_UW, l2 = logical % FA_UW;
    part = l2 / HD, d = l2 % HD, head = 2 * tile + e;
  }
  const bool live = part < 3;
  const int src = part * D + head * HD + d;
  const float sc = (part == 0) ? qscale : 1.0f;
  float cs = 0.f, bb = 0.f;
  for (int k = lane; k < D; k += 32) {
    const int ks = kperm ? kperm[k] : k;  // source channel of packed input channel k
    const float w = live ? W[(int64_t)src * D + ks] : 0.f;
    const __nv_bfloat16 rw = __float2bfloat16_rn(w * gamma[ks] * sc);
    Wp[(int64_t)pr * D + k] = rw;
    cs += __bfloat162float(rw);
    bb = fmaf(w, beta[ks], bb);
  }
  cs = warp_sum(cs);
  bb = warp_sum(bb);
  if (lane == 0) {
    colsum[tile * FA_NT + logical] = cs;
    bias_f[tile * FA_NT + logical] = live ? ((b != nullptr ? b[src] : 0.f) + bb) * sc : 0.f;
  }
}

// ---- host side ---------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// [rows, K] row-major matrix, box = 128 bytes of K x box_rows rows, 128B swizzle, out-of-bounds -> zeros
int make_tmap(CUtensorMap* map, const void* ptr, int64_t rows, int K, int esz, int box_rows, int box_cols = 0, bool swizzle = true,
              int64_t pitch = 0) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return MPL_ERR_CUDA;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)(pitch ? pitch : K) * esz};  // pitch: a [rows, K] window of wider rows
  const cuuint32_t box[2] = {(cuuint32_t)(box_cols ? box_cols : KB_BYTES / esz), (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(map, esz == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld K=%d esz=%d box_rows=%d ptr=%p)", (int)r,
              (long long)rows, K, esz, box_rows, ptr);
    return MPL_ERR_CUDA;
  }
  return MPL_OK;
}

struct GemmMaps {
  CUtensorMap a, b, y, a2, b2, y2;
};

template <int KIND, int EPI>
int launch_one(const GemmMaps& tm, const float* bias, int64_t M, int N, int K, const TileSplit& ts, const GemmLn& ln,
               cudaStream_t s) {
  using C = Cfg<EPI, KIND>;
  auto kern = gemm_tcgen05_kernel<KIND, EPI>;
  // per instantiation and device (function attributes live in the device's context); a benign race: two threads may both set it
  static std::atomic<unsigned char> attr_set[64];
  int dev = 0;
  MPL_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !attr_set[dev].load(std::memory_order_acquire)) {
    MPL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    if (dev >= 0 && dev < 64) attr_set[dev].store(1, std::memory_order_release);
  }
  const int64_t m_tiles = ceil_div(M, (int64_t)BM * CG);
  const int64_t total = m_tiles * ts.T;
  const int64_t max_groups = kNumSMs / CG;
  const unsigned groups = (unsigned)(total < max_groups ? total : max_groups);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(groups * CG);
  cfg.blockDim = dim3(C::THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MPL_CUDA(cudaLaunchKernelEx(&cfg, kern, tm.a, tm.b, tm.y, tm.a2, tm.b2, tm.y2, bias, M, N, K, ts, ln));
  return MPL_OK;
}

template <int KIND>
int launch_epi(int epi, const GemmMaps& tm, const float* bias, int64_t M, int N, int K, const TileSplit& bn, const GemmLn& ln,
               cudaStream_t s) {
  switch (epi) {
    case 0: return launch_one<KIND, 0>(tm, bias, M, N, K, bn, ln, s);
    case 1: return launch_one<KIND, 1>(tm, bias, M, N, K, bn, ln, s);
    case 2: return launch_one<KIND, 2>(tm, bias, M, N, K, bn, ln, s);
    case 3: return launch_one<KIND, 3>(tm, bias, M, N, K, bn, ln, s);
    default: break;
  }
  if constexpr (KIND == 0) {  // the LayerNorm-fused epilogues exist for single-plane bf16 / fp16 operands only
    switch (epi) {
      case 4: return launch_one<KIND, 4>(tm, bias, M, N, K, bn, ln, s);
      case 5: return launch_one<KIND, 5>(tm, bias, M, N, K, bn, ln, s);
      case 6: return launch_one<KIND, 6>(tm, bias, M, N, K, bn, ln, s);
      case 7: return launch_one<KIND, 7>(tm, bias, M, N, K, bn, ln, s);
      default: break;
    }
  }
  set_error("launch_gemm_tcgen05: epilogue %d is not available for this operand type", epi);
  return MPL_ERR_UNSUPPORTED;
}

// Output tiles: whole 64-column groups dealt evenly to ceil(groups / 4) tiles of at most 256 columns (see TileSplit).
// Measured on B200 before the even split existed: N = 1088 as 4 x 256 + 64 beat 5 x 192 + 128 by 8 % (fewer re-reads of A
// per output column) and 4 x 224 + 192 beat 4 x 256 + 64 by another 9 % (no narrow tail tile) -- the even split has both.
TileSplit split_tiles(int N) {
  const int G = (N + 63) / 64;
  TileSplit ts;
  ts.T = (G + 3) / 4;
  ts.q = G / ts.T;
  ts.r = G % ts.T;
  return ts;
}

}  // namespace

static int qkv_attn_tiles(int D, int H) { return D == H * FA_HD ? H : H / 2; }  // head tiles: one 136-wide head or two 68-wide ones

bool qkv_attn_supports(int D, int H, int tokens) {
  const bool shape = H >= 1 && (D == H * FA_HD || (D == H * (FA_HD / 2) && H % 2 == 0));
  return shape && tokens >= 2 && tokens <= 8 && ((int64_t)D * 2) % 16 == 0;
}
size_t qkv_attn_weight_elems(int D, int H) { return (size_t)qkv_attn_tiles(D, H) * FA_NT * D; }
int qkv_attn_vec_len(int D, int H) { return qkv_attn_tiles(D, H) * FA_NT; }

int launch_qkv_attn_pack(const float* W, const float* b, const float* gamma, const float* beta, void* Wp, float* colsum,
                         float* bias_f, int H, int D, float scale, cudaStream_t s, const int* kperm) {
  const int tiles = qkv_attn_tiles(D, H), rows = tiles * FA_NT;
  qkv_attn_pack_kernel<<<(unsigned)ceil_div(rows, 8), 256, 0, s>>>(W, b, gamma, beta, reinterpret_cast<__nv_bfloat16*>(Wp), colsum,
                                                                 bias_f, tiles, D / H, D, scale * 1.4426950408889634f, kperm);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

int launch_qkv_attn(const void* xb, const void* Wp, const float* bias_f, const float* colsum, const void* stats, int slots,
                    float eps, void* att, int64_t M, int D, int H, int V, cudaStream_t s) {
  if (M == 0) return MPL_OK;
  if (!qkv_attn_supports(D, H, V) || M % V != 0) {
    set_error("launch_qkv_attn: needs D = H * 136 (or H * 68, H even), 2 <= V <= 8 and whole poses (D=%d H=%d V=%d)", D, H, V);
    return MPL_ERR_UNSUPPORTED;
  }
  const int tiles = qkv_attn_tiles(D, H);
  const bool pair = tiles != H;
  CUtensorMap tmA, tmB, tmO;
  const int rq = (32 / V) * V;  // rows of a lane quarter: whole poses
  MPL_TRY(make_tmap(&tmA, xb, M, D, 2, rq == 32 ? BM : 32));
  MPL_TRY(make_tmap(&tmB, Wp, (int64_t)tiles * FA_NT, D, 2, FA_B_ROWS));
  MPL_TRY(make_tmap(&tmO, att, M, D, 2, rq, FA_HD, /*swizzle=*/false));
  FusedAttnArgs a{};
  a.bias = bias_f;
  a.colsum = colsum;
  a.stats = reinterpret_cast<const float2*>(stats);
  a.stats_ld = (int64_t)align_up((size_t)M, 256);
  a.slots = slots;
  a.inv_k = 1.0f / (float)D;
  a.eps = eps;
  a.M = M;
  a.K = D;
  a.H = tiles;
  typedef void (*Kern)(CUtensorMap, CUtensorMap, CUtensorMap, FusedAttnArgs);
  static const Kern kerns[2][7] = {
      {qkv_attn_kernel<2, 136>, qkv_attn_kernel<3, 136>, qkv_attn_kernel<4, 136>, qkv_attn_kernel<5, 136>, qkv_attn_kernel<6, 136>,
       qkv_attn_kernel<7, 136>, qkv_attn_kernel<8, 136>},
      {qkv_attn_kernel<2, 68>, qkv_attn_kernel<3, 68>, qkv_attn_kernel<4, 68>, qkv_attn_kernel<5, 68>, qkv_attn_kernel<6, 68>,
       qkv_attn_kernel<7, 68>, qkv_attn_kernel<8, 68>}};
  const int vi = V - 2, hi = pair ? 1 : 0;
  const Kern kern = kerns[hi][vi];
  static std::atomic<unsigned char> attr_set[64][2][7];
  int dev = 0;
  MPL_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !attr_set[dev][hi][vi].load(std::memory_order_acquire)) {
    MPL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, FA_SMEM_BYTES));
    if (dev >= 0 && dev < 64) attr_set[dev][hi][vi].store(1, std::memory_order_release);
  }
  const int64_t total = ceil_div(M, (int64_t)8 * rq) * tiles;
  const unsigned groups = (unsigned)std::min<int64_t>(total, kNumSMs / 2);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(groups * 2);
  cfg.blockDim = dim3(NUM_EPI_WARPS * 32 + 128);
  cfg.dynamicSmemBytes = FA_SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MPL_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmO, a));
  return MPL_OK;
}


bool gemm_tcgen05_supports(int N, int K, int dtype) {
  (void)dtype;  // both tensor-core modes stage bf16 planes
  return N >= 16 && N % 16 == 0 && K >= 1 && ((int64_t)K * 2) % 16 == 0;
}

int gemm_ln_slots(int N) { return 2 * split_tiles(N).T; }  // one slot per (tile, epilogue warp of a lane quarter)

int launch_gemm_tcgen05(const void* A, const void* W, const float* bias, void* Y, int64_t M, int N, int K, int dtype,
                        int epilogue, int out_fp32, cudaStream_t s, const GemmLnArgs* lnargs) {
  if (M == 0) return MPL_OK;
  GemmLn ln{};
  if (epilogue >= EPI_LN_BIAS) {
    if (lnargs == nullptr || dtype != MPL_PREC_BF16) {
      set_error("launch_gemm_tcgen05: LayerNorm-fused epilogues need bf16 operands and GemmLnArgs");
      return MPL_ERR_INVALID_ARGUMENT;
    }
    ln.colsum = lnargs->colsum;
    ln.stats_in = reinterpret_cast<const float2*>(lnargs->stats_in);
    ln.stats_out = reinterpret_cast<float2*>(lnargs->stats_out);
    ln.slots_in = lnargs->slots_in;
    ln.stats_ld = (int64_t)align_up((size_t)M, 256);
    ln.slots_out = gemm_ln_slots(N);
    ln.inv_k = 1.0f / (float)K;
    ln.eps = lnargs->eps;
    ln.flags = (lnargs->ab_fp16 ? 2 : 0) | (lnargs->out_fp16 ? 4 : 0);
    if (epilogue == EPI_RESIDUAL_EMIT && (N % 16 != 0 || ln.stats_out == nullptr || lnargs->x_lo == nullptr)) {
      set_error("launch_gemm_tcgen05: residual-emit epilogue needs N %% 16 == 0, a statistics buffer and the lo plane of the residual");
      return MPL_ERR_INVALID_ARGUMENT;
    }
    if (epilogue != EPI_RESIDUAL_EMIT && (ln.colsum == nullptr || ln.stats_in == nullptr || ln.slots_in < 1)) {
      set_error("launch_gemm_tcgen05: LayerNorm-apply epilogue needs column sums and row statistics");
      return MPL_ERR_INVALID_ARGUMENT;
    }
  }
  if (dtype != MPL_PREC_BF16 && dtype != MPL_PREC_TF32) {
    set_error("launch_gemm_tcgen05: dtype must be MPL_PREC_BF16 or MPL_PREC_TF32");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (!gemm_tcgen05_supports(N, K, dtype)) {
    set_error("tcgen05 projection needs N %% 16 == 0 and a 16-byte aligned row pitch (N=%d K=%d)", N, K);
    return MPL_ERR_UNSUPPORTED;
  }
  if (bias == nullptr) {
    set_error("launch_gemm_tcgen05: bias must not be null");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  const bool split = dtype == MPL_PREC_TF32;  // the fp32-grade mode: operands are two bf16 planes (hi, lo), [2][rows][K]
  int epi = epilogue;
  if (epilogue == EPI_BIAS && out_fp32) epi = 3;
  // output boxes: 32 rows x 128 bytes (64 bf16 or 32 fp32 columns), 128B swizzle like the staging writes
  // residual-emit: short K (proj) is epilogue / HBM bound -> 4 operand stages + 12 residual slots (EPI 6);
  // long K (fc2) is MMA bound -> 5 stages + 8 slots (EPI 7)
  if (epi == 6 && K > 1536) epi = 7;
  const bool resid = epi == 6 || epi == 7;
  const bool out_bf16 = epi == 0 || epi == 1 || epi == 4 || epi == 5 || resid;
  const TileSplit ts = split_tiles(N);
  const int wide_rows = 64 * (ts.q + (ts.r > 0 ? 1 : 0)) / CG, narrow_rows = 64 * ts.q / CG;
  GemmMaps tm;
  MPL_TRY(make_tmap(&tm.a, A, M, K, 2, BM));
  MPL_TRY(make_tmap(&tm.b, W, N, K, 2, wide_rows));
  const int64_t ldy = (resid && lnargs->ldy > 0) ? lnargs->ldy : 0;  // residual planes wider than the N columns updated
  if (ldy != 0 && (ldy < N || (ldy * 2) % 16 != 0)) {
    set_error("launch_gemm_tcgen05: residual row pitch %lld does not fit N=%d", (long long)ldy, N);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  MPL_TRY(make_tmap(&tm.y, Y, M, N, out_bf16 ? 2 : 4, 32, out_bf16 ? 64 : 32, true, ldy));
  tm.a2 = tm.a;
  tm.y2 = tm.y;
  if (split) {
    MPL_TRY(make_tmap(&tm.a2, reinterpret_cast<const __nv_bfloat16*>(A) + M * (int64_t)K, M, K, 2, BM));
    MPL_TRY(make_tmap(&tm.b2, reinterpret_cast<const __nv_bfloat16*>(W) + (int64_t)N * K, N, K, 2, wide_rows));
    if (out_bf16) MPL_TRY(make_tmap(&tm.y2, reinterpret_cast<__nv_bfloat16*>(Y) + M * (int64_t)N, M, N, 2, 32, 64));
  } else {
    MPL_TRY(make_tmap(&tm.b2, W, N, K, 2, narrow_rows));  // the W box of the narrow tiles
    if (resid) MPL_TRY(make_tmap(&tm.y2, lnargs->x_lo, M, N, 2, 32, 64, true, ldy));  // Y = the hi plane, x_lo = the lo plane
  }
  return split ? launch_epi<1>(epi, tm, bias, M, N, K, ts, ln, s) : launch_epi<0>(epi, tm, bias, M, N, K, ts, ln, s);
}

}  // namespace mpl
