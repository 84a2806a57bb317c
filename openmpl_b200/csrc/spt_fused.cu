// K2: the Spatial Pose Transformer as ONE kernel (multiview_mpl.py:400-412 with Block/Attention/Mlp :21-92).
//
// The SPT is latency / issue work, not FLOPs: 17 tokens x 32 channels per (pose, view) set, head_dim 4, depth+1 block
// applications.  Launched layer by layer it is ~14 small kernels per application and re-reads the residual stream
// from HBM every time; here a CTA keeps 14 sets resident for the whole stack, two CTAs per SM:
//   * 14 sets x 17 tokens = 238 rows = 15 MMA row tiles of 16 -> 8 warps x 2 tiles (the last warp's second tile is a
//     phantom), so every weight fragment read from shared memory feeds two MMAs (the v1 kernel, one tile per warp,
//     was bound by the LSU pipe); the two resident CTAs run out of phase, so the attention phase of one (LSU + MUFU)
//     overlaps the MMA / GELU phases of the other (one 544-thread CTA per SM issued only 48 % of the cycles).
//     8 warps rather than 9 x 16 sets (the first shape of this kernel): two 256-thread CTAs get 128 registers per
//     thread instead of 96 and stop spilling -- 3-5 % faster in every mode (profiles/r2_experiments.md);
//   * the residual stream lives in registers as mma.sync C fragments (32 fp32 per lane) across all applications;
//   * LayerNorm is computed on the fragments (quad shuffles, one pass, gamma / beta folded into the following weights
//     and biases at pack time); the four Linears are fp16 mma.sync m16n8k16 with fp32
//     accumulation (fp16 rather than bf16 operands: 3 more mantissa bits, and every operand here is O(1) after
//     LayerNorm; conversions saturate), weights pre-packed in fragment order, double-buffered via cp.async;
//   * q|k|v of the 32 sets are staged once in shared memory as fp16 with the channels of each head PAIR interleaved
//     (word = (head 2p, head 2p+1) at one head-dim), so that the 17x17 softmax of two heads runs in packed half2
//     arithmetic straight from 16-byte shared-memory loads: one thread per two token rows x two head pairs (every
//     k / v vector read serves both rows), two passes (max, then exp2 / sum / PV) with the scores kept in registers.  The interleave costs nothing: it is a row
//     permutation of the QKV weight and a column permutation of the proj weight, applied when the layer is packed;
//     softmax scale * log2(e) is folded into the q rows the same way;
//   * the attention output overwrites the (already consumed) q slot of its own row and is the A operand of proj;
//   * erf-GELU via a tanh-form fit (see gelu_tanh_fit), residual adds and the final Spatial_norm stay in fp32.
// HBM traffic per set: 17*32*4 B in + out, nothing in between.
#include <algorithm>
#include <atomic>

#include <cuda_fp16.h>

#include "kernels.cuh"

namespace mpl {

namespace {

constexpr int J = 17, D = 32, HID = 64, HEADS = 8;
// This file is compiled twice (openmpl_b200/build.py): the primary object with the shape below, and -DMPL_SPT_ALT with the
// first shape of the kernel (16 sets on 9 warps), which exports only launch_fpt_kp_fused_alt -- the keypoint-token FPT of
// V = 5 or 8 views packs whole poses into 16 sets (15 and 16 of them) far better than into 14 (10 and 8).
#ifdef MPL_SPT_ALT
#define MPL_SPT_SETS 16
#define MPL_SPT_WARPS 9
#endif
#ifndef MPL_SPT_SETS  // build-time experiment knob (MPL_SPT_DEFS, openmpl_b200/build.py)
#define MPL_SPT_SETS 14
#define MPL_SPT_WARPS 8
#endif
constexpr int SETS = MPL_SPT_SETS, ROWS = SETS * J, WARPS = MPL_SPT_WARPS, THREADS = WARPS * 32;  // 238 rows in 256 threads
static_assert(ROWS <= WARPS * 32 && SETS * 18 <= THREADS + 17, "two row tiles per warp, 18 attention threads per set");
constexpr int SROWS = WARPS * 32;  // staging rows incl. the phantom tile of the last warp (rows 238..255)
constexpr int QP = 104;     // fp16 row pitch of the q|k|v staging buffer (96 + 8): 52 words -> rows g = 0..7 start on banks
                            // {0,20,8,28,16,4,24,12}: conflict-free half2 C-fragment stores, A-fragment loads and 16 B row loads
constexpr int QPW = QP / 2;

// fragment-packed layer blob (32-bit words): B fragments of the four weight matrices, then the four bias vectors as C
// operands: per output tile column nt and quad lane t the 16-byte group (b[8nt+2t], b[8nt+2t+1], same, same) -- one
// LDS.128 lands in an aligned register quad that the first MMA of the tile takes as its C operand as is.  The LayerNorm
// weights are not stored: gamma / beta are folded into the QKV / fc1 weights and biases (spt_pack_kernel).
constexpr int OFF_QKV = 0, OFF_PROJ = 1536, OFF_FC1 = 2048, OFF_FC2 = 3072, FRAG_WORDS = 4096;
constexpr int F_QKVB = 0, F_PROJB = 192, F_FC1B = 256, F_FC2B = 384;
constexpr int VEC_WORDS = 448, LAYER_WORDS = FRAG_WORDS + VEC_WORDS;  // 4544 words = 18176 bytes
// The packed blob of a layer continues with the LO fragments: fp16(w - fp16(w)) of the same four matrices in the same order.
// Only the PRECISE kernel (the fp32-grade tensor-core mode) loads them: it splits every MMA operand into fp16 hi + lo and
// accumulates hi.hi + lo.hi + hi.lo (22 significand bits per operand instead of 11).
constexpr int LAYER_WORDS_FULL = LAYER_WORDS + FRAG_WORDS;  // 8640 words = 34560 bytes: stride of a layer in the blob
constexpr int QPF = 104;    // PRECISE: fp32 row pitch of the q|k|v staging buffer (96 + 8 words: 8-byte C-fragment stores of a
                            // half-warp, rows g = 0..3, land on 32 distinct banks)

template <bool PRECISE> struct Smem {
  static constexpr int LAYER = PRECISE ? LAYER_WORDS_FULL : LAYER_WORDS;  // words loaded per layer
  static constexpr int W_BYTES = 2 * LAYER * 4;                            // double-buffered
  static constexpr int QKV_BYTES = PRECISE ? SROWS * QPF * 4 : SROWS * QP * 2;
  static constexpr int TOTAL = W_BYTES + QKV_BYTES;                        // 96 256 B (two CTAs per SM) / 188 928 B (one)
};

// staging position (within a 32-wide q, k or v third) of channel c = 8p + 4e + d (head 2p+e, head-dim d): 8p + 2d + e
__host__ __device__ constexpr int chan_of_pos(int pos) { return (pos & ~7) + 4 * (pos & 1) + ((pos & 7) >> 1); }

__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// fp32 pair -> fp16 hi pair + fp16 lo pair (lo = the rounding remainder of hi)
__device__ __forceinline__ void split_f16(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = pack_f16(a, b);
  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  lo = pack_f16(a - hf.x, b - hf.y);
}

__device__ __forceinline__ void mma_f16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// first k-step of a tile: D = A.B + (bx, by, bx, by) -- the bias quad enters as the C operand, no accumulator initialisation
__device__ __forceinline__ void mma_f16_16816_bias(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1, const float4& c) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(c.x), "f"(c.y), "f"(c.z), "f"(c.w));
}

__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}

// LayerNorm (eps 1e-6, biased variance) of the two rows a lane co-owns, straight to fp16 A fragments (2 k-tiles of 16).
// Only the normalisation happens here: gamma is folded into the columns of the following weight matrix and beta into its
// bias when the layer is packed (spt_pack_kernel), so a row costs one FMA per element: y = x * rstd - mean * rstd.
__device__ __forceinline__ void ln_to_afrag(const float (&x)[4][4], uint32_t (&a)[2][4]) {
  // one pass: sum and sum of squares together (32 values of O(1): E[x^2] - mean^2 in fp32 is far inside the fp16 operand
  // rounding that follows), the four quad reductions issued back to back
  float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    s0 += x[nt][0] + x[nt][1];
    s1 += x[nt][2] + x[nt][3];
    q0 = fmaf(x[nt][0], x[nt][0], fmaf(x[nt][1], x[nt][1], q0));
    q1 = fmaf(x[nt][2], x[nt][2], fmaf(x[nt][3], x[nt][3], q1));
  }
  s0 = quad_sum(s0); s1 = quad_sum(s1); q0 = quad_sum(q0); q1 = quad_sum(q1);
  const float m0 = s0 * (1.0f / D), m1 = s1 * (1.0f / D);
  const float r0 = rsqrtf(fmaxf(fmaf(-m0, m0, q0 * (1.0f / D)), 0.f) + 1e-6f);
  const float r1 = rsqrtf(fmaxf(fmaf(-m1, m1, q1 * (1.0f / D)), 0.f) + 1e-6f);
  const float n0 = -m0 * r0, n1 = -m1 * r1;
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    a[nt >> 1][(nt & 1) * 2 + 0] = pack_f16(fmaf(x[nt][0], r0, n0), fmaf(x[nt][1], r0, n0));
    a[nt >> 1][(nt & 1) * 2 + 1] = pack_f16(fmaf(x[nt][2], r1, n1), fmaf(x[nt][3], r1, n1));
  }
}

// the same with every A-fragment register split into hi + lo (PRECISE)
__device__ __forceinline__ void ln_to_afrag_split(const float (&x)[4][4], uint32_t (&ah)[2][4], uint32_t (&al)[2][4]) {
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) { s0 += x[nt][0] + x[nt][1]; s1 += x[nt][2] + x[nt][3]; }
  const float m0 = quad_sum(s0) * (1.0f / D), m1 = quad_sum(s1) * (1.0f / D);
  float q0 = 0.f, q1 = 0.f;  // two-pass variance like nn.LayerNorm: this path is fp32-grade
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    const float d0 = x[nt][0] - m0, d1 = x[nt][1] - m0, d2 = x[nt][2] - m1, d3 = x[nt][3] - m1;
    q0 = fmaf(d0, d0, fmaf(d1, d1, q0));
    q1 = fmaf(d2, d2, fmaf(d3, d3, q1));
  }
  const float r0 = rsqrtf(quad_sum(q0) * (1.0f / D) + 1e-6f), r1 = rsqrtf(quad_sum(q1) * (1.0f / D) + 1e-6f);
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    split_f16((x[nt][0] - m0) * r0, (x[nt][1] - m0) * r0, ah[nt >> 1][(nt & 1) * 2 + 0], al[nt >> 1][(nt & 1) * 2 + 0]);
    split_f16((x[nt][2] - m1) * r1, (x[nt][3] - m1) * r1, ah[nt >> 1][(nt & 1) * 2 + 1], al[nt >> 1][(nt & 1) * 2 + 1]);
  }
}

// one output tile column (8 features) for both row tiles of the warp: acc = bias, then KT k-steps; every B fragment
// read from the packed blob feeds two MMAs
template <int KT>
__device__ __forceinline__ void gemm_tile2(float (&c0)[4], float (&c1)[4], const uint32_t (&a0)[KT][4], const uint32_t (&a1)[KT][4],
                                           const uint32_t* __restrict__ wfrag, int nt, const float* __restrict__ bias, int lane,
                                           int t) {
  const float4 b4 = *reinterpret_cast<const float4*>(bias + 16 * nt + 4 * t);
  {
    const uint2 b = *reinterpret_cast<const uint2*>(wfrag + ((nt * KT) * 32 + lane) * 2);
    mma_f16_16816_bias(c0, a0[0], b.x, b.y, b4);
    mma_f16_16816_bias(c1, a1[0], b.x, b.y, b4);
  }
#pragma unroll
  for (int kt = 1; kt < KT; ++kt) {
    const uint2 b = *reinterpret_cast<const uint2*>(wfrag + ((nt * KT + kt) * 32 + lane) * 2);
    mma_f16_16816(c0, a0[kt], b.x, b.y);
    mma_f16_16816(c1, a1[kt], b.x, b.y);
  }
}

// split form (PRECISE): per k-step hi.hi + lo.hi + hi.lo into the same fp32 accumulators; wlo = the LO fragments of the
// same matrix (FRAG_WORDS + VEC_WORDS words behind the hi fragments)
template <int KT>
__device__ __forceinline__ void gemm_tile2_split(float (&c0)[4], float (&c1)[4], const uint32_t (&a0h)[KT][4], const uint32_t (&a0l)[KT][4],
                                                 const uint32_t (&a1h)[KT][4], const uint32_t (&a1l)[KT][4],
                                                 const uint32_t* __restrict__ wfrag, int nt, const float* __restrict__ bias, int lane,
                                                 int t) {
  const uint32_t* __restrict__ wlo = wfrag + LAYER_WORDS;
  const float4 b4 = *reinterpret_cast<const float4*>(bias + 16 * nt + 4 * t);
#pragma unroll
  for (int kt = 0; kt < KT; ++kt) {
    const uint2 bh = *reinterpret_cast<const uint2*>(wfrag + ((nt * KT + kt) * 32 + lane) * 2);
    const uint2 bl = *reinterpret_cast<const uint2*>(wlo + ((nt * KT + kt) * 32 + lane) * 2);
    if (kt == 0) {
      mma_f16_16816_bias(c0, a0h[0], bl.x, bl.y, b4);
      mma_f16_16816_bias(c1, a1h[0], bl.x, bl.y, b4);
    } else {
      mma_f16_16816(c0, a0h[kt], bl.x, bl.y);
      mma_f16_16816(c1, a1h[kt], bl.x, bl.y);
    }
    mma_f16_16816(c0, a0l[kt], bh.x, bh.y);
    mma_f16_16816(c1, a1l[kt], bh.x, bh.y);
    mma_f16_16816(c0, a0h[kt], bh.x, bh.y);
    mma_f16_16816(c1, a1h[kt], bh.x, bh.y);
  }
}

struct SptArgs {
  const float* x_in;                  // [V, B, J, 32] joint embeddings (null: the embedding is computed here, io.embed)
  float* x_out;                       // [V, B, J, 32] after the stack and Spatial_norm (null: tokens are written here, io.token)
  const uint32_t* wpack[kMaxViews];   // per view stack: [depth][LAYER_WORDS_FULL]
  const float* sn_w;
  const float* sn_b;
  const float* conf;                  // [V, B, J] or null: confidence_as_attention_uncertainty_weight (unfused embed only)
  int64_t B;
  int depth;
  int conf_weighted;                  // the confidence-weighted extra pass per block is live
  int group;                          // GROUPED: sets attending together (V views of a pose); 1 in the SPT
  int rows_used;                      // rows of a CTA tile that carry data: ROWS, or (SETS / group) * group * 17 when GROUPED
  int final_norm;                     // apply Spatial_norm at the end (SPT) or store the residual as is (GROUPED)
  SptIo io;                           // fused K1 embedding in front, fused FPT token build behind
};

// confidence of token row `gr` of `view` straight from the pose record (x, y, conf)
__device__ __forceinline__ float pose_conf(const SptArgs& a, int view, int64_t gr) {
  const int64_t b = gr / J;
  const int j = (int)(gr - b * J);
  return __ldg(a.io.embed.poses[view] + b * a.io.embed.pose_stride + j * 3 + 2);
}

template <int WORDS>
__device__ __forceinline__ void load_layer_async(uint32_t* dst, const uint32_t* src) {
  constexpr int CHUNKS = WORDS * 4 / 16;  // 1136 (2160 with the lo fragments) x 16 bytes
  for (int i = threadIdx.x; i < CHUNKS; i += THREADS) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst + i * 4);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + i * 4) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}
__device__ __forceinline__ void wait_async_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ __half2 h2(uint32_t u) { return *reinterpret_cast<__half2*>(&u); }
__device__ __forceinline__ uint32_t u32(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ __half2 ex2_h2(__half2 x) {
  uint32_t r;
  asm("ex2.approx.f16x2 %0, %1;" : "=r"(r) : "r"(u32(x)));
  return h2(r);
}

// (measured with the 9-warp shape: __maxnreg__(112) removes the spills but only one CTA then fits per SM -> 16.3 ms instead
// of 13.2 ms per step; the 8-warp shape gets its 128 registers with two CTAs resident)
// PRECISE (tf32 mode): softmax / PV arithmetic in fp32 on the fp16-staged q, k, v and the exact erf GELU -- every
// rounding left is a 2^-11 operand rounding, the same class as kind::tf32's; bf16 mode takes the packed-half2 forms.
// GROUPED: the same block stack as the keypoint-token FPT (FPT_blocks_view_keypoint_tokens: tokens = V * 17 joints of one
// pose, width 32, one weight stack, multiview_mpl.py:261-266,416-423,496-497): `group` = V consecutive 17-row sets attend
// together, so the whole V * J-token set of a pose lives in this CTA's shared memory for all depth + 1 block applications
// (V <= 16: one pose of up to 238 tokens per CTA in the 14-set tile at V = 9..14, 255 / 272 tokens in the 16-set tile at
// V = 15 / 16);
// keys are walked in two passes (max, then exp2 / sum / PV with the scores recomputed), fp16 partial
// sums flushed into fp32 every 17 keys.  Rows come from and go back to the fp32 token buffer in place.
template <bool PRECISE, bool GROUPED>
__device__ __forceinline__ void spt_fused_body(const SptArgs& args);

// packed-half2 forms: two CTAs of 8 warps per SM (128 registers each); PRECISE: one CTA per SM with up to 255 registers
// (it takes 238; the 9-warp shape was capped at 168 -- the register file is handed out in units of four warps, 9 count as
// 12 -- and spilled ~740 bytes)
template <bool GROUPED>
__global__ void __launch_bounds__(THREADS, 2) spt_fused_kernel_fast(const SptArgs args) { spt_fused_body<false, GROUPED>(args); }
__global__ void __launch_bounds__(THREADS, 1) spt_fused_kernel_precise(const SptArgs args) { spt_fused_body<true, false>(args); }

template <bool PRECISE, bool GROUPED>
__device__ __forceinline__ void spt_fused_body(const SptArgs& args) {
  static_assert(!(PRECISE && GROUPED), "the grouped (keypoint-token FPT) form exists for the packed-half2 arithmetic only");
  using SM = Smem<PRECISE>;
  constexpr int LW = SM::LAYER;
  extern __shared__ __align__(16) uint8_t smem[];
  uint32_t* wbuf = reinterpret_cast<uint32_t*>(smem);
  uint32_t* qkv_w = reinterpret_cast<uint32_t*>(smem + SM::W_BYTES);  // fp16 staging viewed as half2 words, row pitch QPW
  float* qkv_f = reinterpret_cast<float*>(smem + SM::W_BYTES);        // PRECISE: fp32 staging, row pitch QPF

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int view = blockIdx.y;
  const int64_t tile = blockIdx.x;
  const int64_t rows_in_view = args.B * J;
  const int64_t view_row0 = (int64_t)view * rows_in_view;
  const uint32_t* wsrc = args.wpack[view];

  load_layer_async<LW>(wbuf, wsrc);

  // residual stream: C-fragment layout per row tile mt: x[mt][nt][0..1] = row r0 cols 8nt+2t,+1 ; [2..3] = row r0 + 8
  float x[2][4][4];
  int lr[2];        // CTA-local first row (r0) of each tile
  bool ok[2][2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    lr[mt] = warp * 32 + mt * 16 + g;
    const int64_t gr0 = tile * args.rows_used + lr[mt], gr1 = gr0 + 8;
    ok[mt][0] = lr[mt] < args.rows_used && gr0 < rows_in_view;
    ok[mt][1] = lr[mt] + 8 < args.rows_used && gr1 < rows_in_view;
    if (args.x_in != nullptr) {
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        float2 v0 = make_float2(0.f, 0.f), v1 = make_float2(0.f, 0.f);
        if (ok[mt][0]) v0 = *reinterpret_cast<const float2*>(args.x_in + (view_row0 + gr0) * D + 8 * nt + 2 * t);
        if (ok[mt][1]) v1 = *reinterpret_cast<const float2*>(args.x_in + (view_row0 + gr1) * D + 8 * nt + 2 * t);
        x[mt][nt][0] = v0.x; x[mt][nt][1] = v0.y; x[mt][nt][2] = v1.x; x[mt][nt][3] = v1.y;
      }
    } else {
      // K1 joint embedding fused in front (multiview_mpl.py:349-398): x = W_e (x, y[, conf]) + b_e [+/* conf embedding]
      // + Spatial_pos_embed [+ learnable 3D position], computed straight into the C-fragment layout
      const EmbedArgs& e = args.io.embed;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int64_t gr = h ? gr1 : gr0;
        float px = 0.f, py = 0.f, pc = 0.f;
        int j = 0;
        if (ok[mt][h]) {
          const int64_t b = gr / J;
          j = (int)(gr - b * J);
          const float* pp = e.poses[view] + b * e.pose_stride + j * 3;
          px = __ldg(pp); py = __ldg(pp + 1); pc = __ldg(pp + 2);
        }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int c = 8 * nt + 2 * t + i;
            const float* W = e.We[view] + c * e.in_ch;
            float val = fmaf(__ldg(W + 1), py, fmaf(__ldg(W), px, __ldg(e.be[view] + c)));
            if (e.in_ch == 3) val = fmaf(__ldg(W + 2), pc, val);
            if (e.add_conf || e.mult_conf) {
              const float ce = fmaf(__ldg(e.Wc[view] + c), pc, __ldg(e.bc[view] + c));
              if (e.add_conf) val += ce;
              if (e.mult_conf) val *= ce;
            }
            val += __ldg(e.Ps[view] + j * D + c);
            if (e.spatial_pos_mode == 1) val += __ldg(e.pos3d + j * e.pos3d_ld + c);
            x[mt][nt][2 * h + i] = ok[mt][h] ? val : 0.f;
          }
        }
      }
    }
  }

  // attention role of this thread: TWO token rows of one set (rows 2rs, 2rs+1; the 9th slot of a set holds row 16 alone)
  // x two head pairs (hh, hh + 2): every k / v vector read from shared memory serves both rows.  18 threads per set.
  const int aset = threadIdx.x / 18, arem = threadIdx.x % 18, ars = arem >> 1, ahh = arem & 1;
  const int ra = aset * J + 2 * ars;
  const bool two = ars < 8;
  const int rb = two ? ra + 1 : ra;
  const int aset0 = aset * J;  // first row of the set
  float aconf_a = 1.0f, aconf_b = 1.0f;
  if (args.conf_weighted) {
    const int64_t ga = tile * args.rows_used + ra, gb = tile * args.rows_used + rb;
    if (ga < rows_in_view) aconf_a = args.conf != nullptr ? __ldg(args.conf + view_row0 + ga) : pose_conf(args, view, ga);
    if (gb < rows_in_view) aconf_b = args.conf != nullptr ? __ldg(args.conf + view_row0 + gb) : pose_conf(args, view, gb);
  }

  for (int layer = 0; layer < args.depth; ++layer) {
    wait_async_all();
    __syncthreads();  // this layer's weights have landed; every warp is done with the other buffer
    const uint32_t* w = wbuf + (layer & 1) * LW;
    const float* wv = reinterpret_cast<const float*>(w + FRAG_WORDS);
    if (layer + 1 < args.depth) load_layer_async<LW>(wbuf + ((layer + 1) & 1) * LW, wsrc + (size_t)(layer + 1) * LAYER_WORDS_FULL);

    // block applications of this layer (multiview_mpl.py:405-410): [confidence-weighted], [last layer: once more], plain
    const int n_apps = (args.conf_weighted ? 1 : 0) + (layer == args.depth - 1 ? 2 : 1);
    for (int app = 0; app < n_apps; ++app) {
      const bool weighted = args.conf_weighted && app == 0;
      // ---- LN1 + QKV -> fp16 staging (q pre-scaled by scale * log2 e through the packed weights) ----
      if constexpr (PRECISE) {
        uint32_t a0h[2][4], a0l[2][4], a1h[2][4], a1l[2][4];
        ln_to_afrag_split(x[0], a0h, a0l);
        ln_to_afrag_split(x[1], a1h, a1l);
#pragma unroll
        for (int nt = 0; nt < 12; ++nt) {
          float c0[4], c1[4];
          gemm_tile2_split<2>(c0, c1, a0h, a0l, a1h, a1l, w + OFF_QKV, nt, wv + F_QKVB, lane, t);
          *reinterpret_cast<float2*>(qkv_f + lr[0] * QPF + 8 * nt + 2 * t) = make_float2(c0[0], c0[1]);
          *reinterpret_cast<float2*>(qkv_f + (lr[0] + 8) * QPF + 8 * nt + 2 * t) = make_float2(c0[2], c0[3]);
          *reinterpret_cast<float2*>(qkv_f + lr[1] * QPF + 8 * nt + 2 * t) = make_float2(c1[0], c1[1]);
          *reinterpret_cast<float2*>(qkv_f + (lr[1] + 8) * QPF + 8 * nt + 2 * t) = make_float2(c1[2], c1[3]);
        }
      } else {
        uint32_t a0[2][4], a1[2][4];
        ln_to_afrag(x[0], a0);
        ln_to_afrag(x[1], a1);
#pragma unroll
        for (int nt = 0; nt < 12; ++nt) {
          float c0[4], c1[4];
          gemm_tile2<2>(c0, c1, a0, a1, w + OFF_QKV, nt, wv + F_QKVB, lane, t);
          qkv_w[lr[0] * QPW + 4 * nt + t] = pack_f16(c0[0], c0[1]);
          qkv_w[(lr[0] + 8) * QPW + 4 * nt + t] = pack_f16(c0[2], c0[3]);
          qkv_w[lr[1] * QPW + 4 * nt + t] = pack_f16(c1[0], c1[1]);
          qkv_w[(lr[1] + 8) * QPW + 4 * nt + t] = pack_f16(c1[2], c1[3]);
        }
      }
      __syncthreads();
      // ---- attention: softmax(q k^T * scale) v over the 17 tokens of the row's set; two heads per half2 lane pair ----
      if constexpr (GROUPED) {
        if (aset * J < args.rows_used) {
          const int g0row = (aset / args.group) * args.group * J;  // first row of the pose's token set
          const int nkeys = args.group * J;
          uint4* rowpa = reinterpret_cast<uint4*>(qkv_w + ra * QPW);
          uint4* rowpb = reinterpret_cast<uint4*>(qkv_w + rb * QPW);
          const uint4* setp = reinterpret_cast<const uint4*>(qkv_w + g0row * QPW);
          constexpr int RP4 = QPW / 4;
#pragma unroll 1
          for (int pp = 0; pp < 2; ++pp) {
            const int p = ahh + 2 * pp;
            const uint4 qa = rowpa[p], qb = rowpb[p];
            __half2 mxa = __float2half2_rn(-60000.f), mxb = mxa;
            for (int j = 0; j < nkeys; ++j) {
              const uint4 k = setp[j * RP4 + 4 + p];
              __half2 s0 = __hmul2(h2(qa.x), h2(k.x)), s1 = __hmul2(h2(qb.x), h2(k.x));
              s0 = __hfma2(h2(qa.y), h2(k.y), s0); s1 = __hfma2(h2(qb.y), h2(k.y), s1);
              s0 = __hfma2(h2(qa.z), h2(k.z), s0); s1 = __hfma2(h2(qb.z), h2(k.z), s1);
              s0 = __hfma2(h2(qa.w), h2(k.w), s0); s1 = __hfma2(h2(qb.w), h2(k.w), s1);
              mxa = __hmax2(mxa, s0);
              mxb = __hmax2(mxb, s1);
            }
            float2 fsa = make_float2(0.f, 0.f), fsb = fsa;
            float2 oa[4], ob[4];
#pragma unroll
            for (int d = 0; d < 4; ++d) { oa[d] = make_float2(0.f, 0.f); ob[d] = oa[d]; }
            for (int j0 = 0; j0 < nkeys; j0 += J) {
              const __half2 z = __float2half2_rn(0.f);
              __half2 suma = z, a0 = z, a1 = z, a2 = z, a3 = z, sumb = z, b0 = z, b1 = z, b2 = z, b3 = z;
#pragma unroll
              for (int jj = 0; jj < J; ++jj) {
                const int j = j0 + jj;
                const uint4 k = setp[j * RP4 + 4 + p];
                const uint4 v = setp[j * RP4 + 8 + p];
                __half2 s0 = __hmul2(h2(qa.x), h2(k.x)), s1 = __hmul2(h2(qb.x), h2(k.x));
                s0 = __hfma2(h2(qa.y), h2(k.y), s0); s1 = __hfma2(h2(qb.y), h2(k.y), s1);
                s0 = __hfma2(h2(qa.z), h2(k.z), s0); s1 = __hfma2(h2(qb.z), h2(k.z), s1);
                s0 = __hfma2(h2(qa.w), h2(k.w), s0); s1 = __hfma2(h2(qb.w), h2(k.w), s1);
                const __half2 ea = ex2_h2(__hsub2(s0, mxa)), eb = ex2_h2(__hsub2(s1, mxb));
                suma = __hadd2(suma, ea); sumb = __hadd2(sumb, eb);
                a0 = __hfma2(ea, h2(v.x), a0); b0 = __hfma2(eb, h2(v.x), b0);
                a1 = __hfma2(ea, h2(v.y), a1); b1 = __hfma2(eb, h2(v.y), b1);
                a2 = __hfma2(ea, h2(v.z), a2); b2 = __hfma2(eb, h2(v.z), b2);
                a3 = __hfma2(ea, h2(v.w), a3); b3 = __hfma2(eb, h2(v.w), b3);
              }
              auto flush = [](float2& acc, __half2 h) { const float2 f = __half22float2(h); acc.x += f.x; acc.y += f.y; };
              flush(fsa, suma); flush(oa[0], a0); flush(oa[1], a1); flush(oa[2], a2); flush(oa[3], a3);
              flush(fsb, sumb); flush(ob[0], b0); flush(ob[1], b1); flush(ob[2], b2); flush(ob[3], b3);
            }
            {
              const float i0 = 1.0f / fsa.x, i1 = 1.0f / fsa.y;
              uint4 o;
              o.x = pack_f16(oa[0].x * i0, oa[0].y * i1); o.y = pack_f16(oa[1].x * i0, oa[1].y * i1);
              o.z = pack_f16(oa[2].x * i0, oa[2].y * i1); o.w = pack_f16(oa[3].x * i0, oa[3].y * i1);
              rowpa[p] = o;
            }
            if (two) {
              const float i0 = 1.0f / fsb.x, i1 = 1.0f / fsb.y;
              uint4 o;
              o.x = pack_f16(ob[0].x * i0, ob[0].y * i1); o.y = pack_f16(ob[1].x * i0, ob[1].y * i1);
              o.z = pack_f16(ob[2].x * i0, ob[2].y * i1); o.w = pack_f16(ob[3].x * i0, ob[3].y * i1);
              rowpb[p] = o;
            }
          }
        }
      } else       if constexpr (PRECISE) {
        // fp32 staging: word = one value; a head pair p owns words 8p .. 8p+7 = (dim 0: head 2p, head 2p+1), (dim 1: ..), ..
        float4* rowps[2] = {reinterpret_cast<float4*>(qkv_f + ra * QPF), reinterpret_cast<float4*>(qkv_f + rb * QPF)};
        const float rsc[2] = {weighted ? aconf_a : 1.0f, weighted ? aconf_b : 1.0f};
        const float4* setp = reinterpret_cast<const float4*>(qkv_f + aset0 * QPF);
        constexpr int RP4 = QPF / 4;  // row pitch in float4 units (26)
#pragma unroll 1
        for (int pp = 0; pp < 2; ++pp) {
          const int p = ahh + 2 * pp;
#pragma unroll 1
          for (int rr = 0; rr < 2; ++rr) {
            if (rr == 1 && !two) break;
            const float4 qa = rowps[rr][2 * p], qb = rowps[rr][2 * p + 1];  // (d0h0, d0h1, d1h0, d1h1), (d2h0, d2h1, d3h0, d3h1)
            float s0[J], s1[J];
            float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
            for (int j = 0; j < J; ++j) {
              const float4 ka = setp[j * RP4 + 8 + 2 * p], kb = setp[j * RP4 + 9 + 2 * p];
              s0[j] = fmaf(qb.z, kb.z, fmaf(qb.x, kb.x, fmaf(qa.z, ka.z, qa.x * ka.x)));
              s1[j] = fmaf(qb.w, kb.w, fmaf(qb.y, kb.y, fmaf(qa.w, ka.w, qa.y * ka.y)));
              m0 = fmaxf(m0, s0[j]);
              m1 = fmaxf(m1, s1[j]);
            }
            float sum0 = 0.f, sum1 = 0.f;
            float4 oa = make_float4(0.f, 0.f, 0.f, 0.f), ob = oa;
#pragma unroll
            for (int j = 0; j < J; ++j) {
              const float4 va = setp[j * RP4 + 16 + 2 * p], vb = setp[j * RP4 + 17 + 2 * p];
              const float e0 = exp2f(s0[j] - m0), e1 = exp2f(s1[j] - m1);
              sum0 += e0; sum1 += e1;
              oa.x = fmaf(e0, va.x, oa.x); oa.y = fmaf(e1, va.y, oa.y); oa.z = fmaf(e0, va.z, oa.z); oa.w = fmaf(e1, va.w, oa.w);
              ob.x = fmaf(e0, vb.x, ob.x); ob.y = fmaf(e1, vb.y, ob.y); ob.z = fmaf(e0, vb.z, ob.z); ob.w = fmaf(e1, vb.w, ob.w);
            }
            const float i0 = rsc[rr] / sum0, i1 = rsc[rr] / sum1;
            // the q slot of this row / head pair is consumed: it now holds the attention output
            rowps[rr][2 * p] = make_float4(oa.x * i0, oa.y * i1, oa.z * i0, oa.w * i1);
            rowps[rr][2 * p + 1] = make_float4(ob.x * i0, ob.y * i1, ob.z * i0, ob.w * i1);
          }
        }
      } else       {
        const float sa = weighted ? aconf_a : 1.0f, sb = weighted ? aconf_b : 1.0f;
        uint4* rowpa = reinterpret_cast<uint4*>(qkv_w + ra * QPW);
        uint4* rowpb = reinterpret_cast<uint4*>(qkv_w + rb * QPW);
        const uint4* setp = reinterpret_cast<const uint4*>(qkv_w + aset0 * QPW);
        constexpr int RP4 = QPW / 4;  // row pitch in 16-byte units (13)
#pragma unroll 1
        for (int pp = 0; pp < 2; ++pp) {
          const int p = ahh + 2 * pp;
          const uint4 qa = rowpa[p], qb = rowpb[p];
          __half2 sca[J], scb[J];
          __half2 mxa, mxb;
#pragma unroll
          for (int j = 0; j < J; ++j) {
            const uint4 k = setp[j * RP4 + 4 + p];
            __half2 s0 = __hmul2(h2(qa.x), h2(k.x)), s1 = __hmul2(h2(qb.x), h2(k.x));
            s0 = __hfma2(h2(qa.y), h2(k.y), s0); s1 = __hfma2(h2(qb.y), h2(k.y), s1);
            s0 = __hfma2(h2(qa.z), h2(k.z), s0); s1 = __hfma2(h2(qb.z), h2(k.z), s1);
            s0 = __hfma2(h2(qa.w), h2(k.w), s0); s1 = __hfma2(h2(qb.w), h2(k.w), s1);
            sca[j] = s0; scb[j] = s1;
            mxa = (j == 0) ? s0 : __hmax2(mxa, s0);
            mxb = (j == 0) ? s1 : __hmax2(mxb, s1);
          }
          const __half2 z = __float2half2_rn(0.f);
          __half2 suma = z, a0 = z, a1 = z, a2 = z, a3 = z, sumb = z, b0 = z, b1 = z, b2 = z, b3 = z;
#pragma unroll
          for (int j = 0; j < J; ++j) {
            const uint4 v = setp[j * RP4 + 8 + p];
            const __half2 ea = ex2_h2(__hsub2(sca[j], mxa)), eb = ex2_h2(__hsub2(scb[j], mxb));
            suma = __hadd2(suma, ea); sumb = __hadd2(sumb, eb);
            a0 = __hfma2(ea, h2(v.x), a0); b0 = __hfma2(eb, h2(v.x), b0);
            a1 = __hfma2(ea, h2(v.y), a1); b1 = __hfma2(eb, h2(v.y), b1);
            a2 = __hfma2(ea, h2(v.z), a2); b2 = __hfma2(eb, h2(v.z), b2);
            a3 = __hfma2(ea, h2(v.w), a3); b3 = __hfma2(eb, h2(v.w), b3);
          }
          // the q slot of a row / head pair is consumed: it now holds the attention output (A operand of proj)
          {
            const float2 sf = __half22float2(suma);
            const __half2 inv = __floats2half2_rn(__fdividef(sa, sf.x), __fdividef(sa, sf.y));
            uint4 o;
            o.x = u32(__hmul2(a0, inv)); o.y = u32(__hmul2(a1, inv)); o.z = u32(__hmul2(a2, inv)); o.w = u32(__hmul2(a3, inv));
            rowpa[p] = o;
          }
          if (two) {
            const float2 sf = __half22float2(sumb);
            const __half2 inv = __floats2half2_rn(__fdividef(sb, sf.x), __fdividef(sb, sf.y));
            uint4 o;
            o.x = u32(__hmul2(b0, inv)); o.y = u32(__hmul2(b1, inv)); o.z = u32(__hmul2(b2, inv)); o.w = u32(__hmul2(b3, inv));
            rowpb[p] = o;
          }
        }
      }
      __syncthreads();
      // ---- proj + residual ----
      if constexpr (PRECISE) {
        uint32_t a0h[2][4], a0l[2][4], a1h[2][4], a1l[2][4];
#pragma unroll
        for (int kt = 0; kt < 2; ++kt) {
#pragma unroll
          for (int r = 0; r < 4; ++r) {  // fragment register r: row + 8 * (r & 1), columns 16 kt + 8 * (r >> 1) + 2t, +1
            const int off = (r & 1) * 8 * QPF + 16 * kt + (r >> 1) * 8 + 2 * t;
            const float2 v0 = *reinterpret_cast<const float2*>(qkv_f + lr[0] * QPF + off);
            const float2 v1 = *reinterpret_cast<const float2*>(qkv_f + lr[1] * QPF + off);
            split_f16(v0.x, v0.y, a0h[kt][r], a0l[kt][r]);
            split_f16(v1.x, v1.y, a1h[kt][r], a1l[kt][r]);
          }
        }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          float c0[4], c1[4];
          gemm_tile2_split<2>(c0, c1, a0h, a0l, a1h, a1l, w + OFF_PROJ, nt, wv + F_PROJB, lane, t);
#pragma unroll
          for (int i = 0; i < 4; ++i) { x[0][nt][i] += c0[i]; x[1][nt][i] += c1[i]; }
        }
      } else {
        uint32_t a0[2][4], a1[2][4];
#pragma unroll
        for (int kt = 0; kt < 2; ++kt) {
          a0[kt][0] = qkv_w[lr[0] * QPW + 8 * kt + t];
          a0[kt][1] = qkv_w[(lr[0] + 8) * QPW + 8 * kt + t];
          a0[kt][2] = qkv_w[lr[0] * QPW + 8 * kt + 4 + t];
          a0[kt][3] = qkv_w[(lr[0] + 8) * QPW + 8 * kt + 4 + t];
          a1[kt][0] = qkv_w[lr[1] * QPW + 8 * kt + t];
          a1[kt][1] = qkv_w[(lr[1] + 8) * QPW + 8 * kt + t];
          a1[kt][2] = qkv_w[lr[1] * QPW + 8 * kt + 4 + t];
          a1[kt][3] = qkv_w[(lr[1] + 8) * QPW + 8 * kt + 4 + t];
        }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          float c0[4], c1[4];
          gemm_tile2<2>(c0, c1, a0, a1, w + OFF_PROJ, nt, wv + F_PROJB, lane, t);
#pragma unroll
          for (int i = 0; i < 4; ++i) { x[0][nt][i] += c0[i]; x[1][nt][i] += c1[i]; }
        }
      }
      // ---- LN2 + fc1 + GELU + fc2 + residual ----
      if constexpr (PRECISE) {
        uint32_t a0h[2][4], a0l[2][4], a1h[2][4], a1l[2][4];
        ln_to_afrag_split(x[0], a0h, a0l);
        ln_to_afrag_split(x[1], a1h, a1l);
        uint32_t h0h[4][4], h0l[4][4], h1h[4][4], h1l[4][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          float c0[4], c1[4];
          gemm_tile2_split<2>(c0, c1, a0h, a0l, a1h, a1l, w + OFF_FC1, nt, wv + F_FC1B, lane, t);
          const int kt = nt >> 1, r = (nt & 1) * 2;
          split_f16(gelu_erf(c0[0]), gelu_erf(c0[1]), h0h[kt][r], h0l[kt][r]);
          split_f16(gelu_erf(c0[2]), gelu_erf(c0[3]), h0h[kt][r + 1], h0l[kt][r + 1]);
          split_f16(gelu_erf(c1[0]), gelu_erf(c1[1]), h1h[kt][r], h1l[kt][r]);
          split_f16(gelu_erf(c1[2]), gelu_erf(c1[3]), h1h[kt][r + 1], h1l[kt][r + 1]);
        }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          float c0[4], c1[4];
          gemm_tile2_split<4>(c0, c1, h0h, h0l, h1h, h1l, w + OFF_FC2, nt, wv + F_FC2B, lane, t);
#pragma unroll
          for (int i = 0; i < 4; ++i) { x[0][nt][i] += c0[i]; x[1][nt][i] += c1[i]; }
        }
      } else {
        uint32_t a0[2][4], a1[2][4];
        ln_to_afrag(x[0], a0);
        ln_to_afrag(x[1], a1);
        uint32_t h0[4][4], h1[4][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          float c0[4], c1[4];
          gemm_tile2<2>(c0, c1, a0, a1, w + OFF_FC1, nt, wv + F_FC1B, lane, t);
          h0[nt >> 1][(nt & 1) * 2 + 0] = gelu_tanh_fit_h2(pack_f16(c0[0], c0[1]));
          h0[nt >> 1][(nt & 1) * 2 + 1] = gelu_tanh_fit_h2(pack_f16(c0[2], c0[3]));
          h1[nt >> 1][(nt & 1) * 2 + 0] = gelu_tanh_fit_h2(pack_f16(c1[0], c1[1]));
          h1[nt >> 1][(nt & 1) * 2 + 1] = gelu_tanh_fit_h2(pack_f16(c1[2], c1[3]));
        }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          float c0[4], c1[4];
          gemm_tile2<4>(c0, c1, h0, h1, w + OFF_FC2, nt, wv + F_FC2B, lane, t);
#pragma unroll
          for (int i = 0; i < 4; ++i) { x[0][nt][i] += c0[i]; x[1][nt][i] += c1[i]; }
        }
      }
    }
  }

  // planes out (TokenArgs::tok_hi): per-row (sum, sum^2) of everything this CTA writes, reduced per set in a fixed order
  // through the weight buffer no layer is using any more
  const bool planes_out = args.x_out == nullptr && args.io.token.tok_hi != nullptr;
  float2* rowstat = reinterpret_cast<float2*>(wbuf + ((args.depth == 0 ? 1 : args.depth) & 1) * LW);

  // ---- Spatial_norm (multiview_mpl.py:412), fp32 out ----
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) { s0 += x[mt][nt][0] + x[mt][nt][1]; s1 += x[mt][nt][2] + x[mt][nt][3]; }
    const float m0 = quad_sum(s0) * (1.0f / D), m1 = quad_sum(s1) * (1.0f / D);
    float q0 = 0.f, q1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const float d0 = x[mt][nt][0] - m0, d1 = x[mt][nt][1] - m0, d2 = x[mt][nt][2] - m1, d3 = x[mt][nt][3] - m1;
      q0 += d0 * d0 + d1 * d1;
      q1 += d2 * d2 + d3 * d3;
    }
    const float rs0 = rsqrtf(quad_sum(q0) * (1.0f / D) + 1e-6f), rs1 = rsqrtf(quad_sum(q1) * (1.0f / D) + 1e-6f);
    const int64_t gr0 = tile * args.rows_used + lr[mt], gr1 = gr0 + 8;
    float y[4][4];  // Spatial_norm output, same fragment layout as x
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      if (!args.final_norm) {  // GROUPED: there is no norm behind the FPT stack, the residual goes out as is
        y[nt][0] = x[mt][nt][0]; y[nt][1] = x[mt][nt][1]; y[nt][2] = x[mt][nt][2]; y[nt][3] = x[mt][nt][3];
        continue;
      }
      const float2 wg = __ldg(reinterpret_cast<const float2*>(args.sn_w + 8 * nt + 2 * t));
      const float2 bg = __ldg(reinterpret_cast<const float2*>(args.sn_b + 8 * nt + 2 * t));
      y[nt][0] = (x[mt][nt][0] - m0) * rs0 * wg.x + bg.x; y[nt][1] = (x[mt][nt][1] - m0) * rs0 * wg.y + bg.y;
      y[nt][2] = (x[mt][nt][2] - m1) * rs1 * wg.x + bg.x; y[nt][3] = (x[mt][nt][3] - m1) * rs1 * wg.y + bg.y;
    }
    if (args.x_out != nullptr) {
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        if (ok[mt][0]) *reinterpret_cast<float2*>(args.x_out + (view_row0 + gr0) * D + 8 * nt + 2 * t) = make_float2(y[nt][0], y[nt][1]);
        if (ok[mt][1]) *reinterpret_cast<float2*>(args.x_out + (view_row0 + gr1) * D + 8 * nt + 2 * t) = make_float2(y[nt][2], y[nt][3]);
      }
      continue;
    }
    // FPT token build fused behind (multiview_mpl.py:463-499): [+ confidence embedding] [| ray embedding] + 3D position,
    // written straight into tok [B, V, tok_w] (8-byte stores, 32 contiguous bytes per quad)
    const TokenArgs& k = args.io.token;
    const int V = gridDim.y;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float rs = 0.f, rq = 0.f;  // this lane's share of the row's (sum, sum^2)
      auto emit = [&](int64_t off, float v0, float v1) {
        if (planes_out) {
          const __nv_bfloat162 hh = __floats2bfloat162_rn(v0, v1);
          const uint32_t u = *reinterpret_cast<const uint32_t*>(&hh);
          const __nv_bfloat162 ll = __floats2bfloat162_rn(v0 - __uint_as_float(u << 16), v1 - __uint_as_float(u & 0xffff0000u));
          *reinterpret_cast<uint32_t*>(k.tok_hi + off) = u;
          *reinterpret_cast<__nv_bfloat162*>(k.tok_lo + off) = ll;
          rs += v0 + v1;
          rq = fmaf(v0, v0, fmaf(v1, v1, rq));
        } else {
          *reinterpret_cast<float2*>(k.tok + off) = make_float2(v0, v1);
        }
      };
      if (ok[mt][h]) {  // (the quad reduction below is executed by every lane of the warp, valid row or not)
        const int64_t gr = h ? gr1 : gr0;
        const int64_t b = gr / J;
        const int j = (int)(gr - b * J);
        const int64_t trow = (b * V + view) * (int64_t)k.tok_w;
        const bool need_dir = k.ray_layout != 0 || k.pos_table == nullptr;
        float dx = 0.f, dy = 0.f, dz = 0.f, inv = 0.f;
        if (need_dir) {
          const float* r = k.rays[view] + b * k.pose_stride + j * 3;
          const float* ce = k.centers[view] + b * k.center_stride;
          dx = __ldg(r) - __ldg(ce); dy = __ldg(r + 1) - __ldg(ce + 1); dz = __ldg(r + 2) - __ldg(ce + 2);
          inv = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);  // F.normalize eps
        }
        const float pc = (k.Wcf != nullptr) ? __ldg(k.poses[view] + b * k.pose_stride + j * 3 + 2) : 0.f;
        auto pos_at = [&](int pos_c) {  // 3D position code of channel pos_c of this joint
          if (k.pos_table != nullptr) return __ldg(k.pos_table + j * k.pos_w + pos_c);
          const float* wl = k.Wl + pos_c * 3;
          return fmaf(__ldg(wl + 2), dz * inv, fmaf(__ldg(wl + 1), dy * inv, fmaf(__ldg(wl), dx * inv, __ldg(k.bl + pos_c))));
        };
        // channels per joint slot of the pose part; perm_layout: the interleaved row is stored as [J pose parts | J ray parts]
        const int slot = (k.ray_layout == 1 && !k.perm_layout) ? 2 * D : D;
  #pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const int c = 8 * nt + 2 * t;
          float v0 = y[nt][2 * h], v1 = y[nt][2 * h + 1];
          if (k.Wcf != nullptr) {
            v0 += fmaf(__ldg(k.Wcf + c), pc, __ldg(k.bcf + c));
            v1 += fmaf(__ldg(k.Wcf + c + 1), pc, __ldg(k.bcf + c + 1));
          }
          v0 += pos_at(c);
          v1 += pos_at(c + 1);
          emit(trow + j * slot + c, v0, v1);
          if (k.ray_layout != 0) {
            const float* w0 = k.Wr + c * 3;
            float r0 = fmaf(__ldg(w0 + 2), dz, fmaf(__ldg(w0 + 1), dy, fmaf(__ldg(w0), dx, __ldg(k.br + c))));
            float r1 = fmaf(__ldg(w0 + 5), dz, fmaf(__ldg(w0 + 4), dy, fmaf(__ldg(w0 + 3), dx, __ldg(k.br + c + 1))));
            if (k.ray_layout == 1) {  // [x | ray] per joint, the position code spans both halves
              r0 += pos_at(D + c);
              r1 += pos_at(D + c + 1);
              emit(trow + (k.perm_layout ? (J + j) * D : j * slot + D) + c, r0, r1);
            } else {                  // J pose tokens then J ray tokens (no position code on the ray tokens)
              emit(trow + (J + j) * D + c, r0, r1);
            }
          }
        }
      }
      if (planes_out) {
        rs = quad_sum(rs);
        rq = quad_sum(rq);
        if (t == 0) rowstat[lr[mt] + 8 * h] = make_float2(rs, rq);
      }
    }
  }
  if (planes_out) {
    __syncthreads();
    // one thread per set: its J rows in order (bitwise reproducible), then slot 0 of the row's statistics; other slots zero
    const TokenArgs& k = args.io.token;
    const int set = threadIdx.x;
    const int64_t gr = tile * args.rows_used + (int64_t)set * J;
    if (set * J < args.rows_used && gr < rows_in_view) {
      float s1 = 0.f, s2 = 0.f;
      for (int j = 0; j < J; ++j) { const float2 v = rowstat[set * J + j]; s1 += v.x; s2 += v.y; }
      const int64_t row = (gr / J) * gridDim.y + view;
      k.stats[row] = make_float2(s1, s2);
      for (int i = 1; i < k.stat_slots; ++i) k.stats[i * k.stats_ld + row] = make_float2(0.f, 0.f);
    }
  }
}

// fp32 parameters of one Block -> the fragment-packed layer blob (fp16 operands, head-pair interleave, q scale folded)
struct SptPackArgs {
  const float *n1w, *n1b, *qkvw, *qkvb, *projw, *projb, *n2w, *n2b, *fc1w, *fc1b, *fc2w, *fc2b;
  uint32_t* dst;
  float q_scale;  // softmax scale * log2(e), folded into the q rows of the QKV weight and bias
};

__device__ __forceinline__ uint32_t pack_f16_rn(float lo, float hi) {
  __half2 p = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

__global__ void spt_pack_kernel(const SptPackArgs a) {
  const int i_out = blockIdx.x * blockDim.x + threadIdx.x;
  if (i_out >= LAYER_WORDS_FULL) return;
  const bool lo_part = i_out >= LAYER_WORDS;       // the LO fragments: fp16(w - fp16(w)), same order as the hi fragments
  const int i = lo_part ? i_out - LAYER_WORDS : i_out;
  if (i < FRAG_WORDS) {
    const float* W;
    int K, KT, base, kind;  // kind 0 qkv (output rows permuted), 1 proj (input columns permuted), 2 plain
    if (i < OFF_PROJ) { W = a.qkvw; K = 32; KT = 2; base = OFF_QKV; kind = 0; }
    else if (i < OFF_FC1) { W = a.projw; K = 32; KT = 2; base = OFF_PROJ; kind = 1; }
    else if (i < OFF_FC2) { W = a.fc1w; K = 32; KT = 2; base = OFF_FC1; kind = 2; }
    else { W = a.fc2w; K = 64; KT = 4; base = OFF_FC2; kind = 2; }
    const int j = i - base;
    const int reg = j & 1, lane = (j >> 1) & 31, tl = j >> 6;
    const int nt = tl / KT, kt = tl % KT;
    const int g = lane >> 2, t = lane & 3;
    int n = 8 * nt + g;
    const int k = 16 * kt + 2 * t + 8 * reg;
    float sc = 1.0f;
    if (kind == 0) {
      const int third = n / 32;
      n = third * 32 + chan_of_pos(n % 32);
      if (third == 0) sc = a.q_scale;
    }
    const int k0 = (kind == 1) ? chan_of_pos(k) : k, k1 = (kind == 1) ? chan_of_pos(k + 1) : k + 1;
    // the LayerNorm in front of QKV / fc1 leaves its gamma here (W' = W diag(gamma)) and its beta in the bias below
    const float* gam = (i < OFF_PROJ) ? a.n1w : ((i >= OFF_FC1 && i < OFF_FC2) ? a.n2w : nullptr);
    const float g0 = gam ? gam[k0] : 1.0f, g1 = gam ? gam[k1] : 1.0f;
    const float w0 = W[n * K + k0] * sc * g0, w1 = W[n * K + k1] * sc * g1;
    const uint32_t hi = pack_f16_rn(w0, w1);
    if (lo_part) {
      const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
      a.dst[i_out] = pack_f16_rn(w0 - hf.x, w1 - hf.y);
    } else {
      a.dst[i_out] = hi;
    }
  } else {
    const int f = i - FRAG_WORDS;
    // bias quads: word (16 nt + 4 t + comp) of a section = bias of output column 8 nt + 2 t + (comp & 1)
    const int sec = f < F_PROJB ? 0 : (f < F_FC1B ? 1 : (f < F_FC2B ? 2 : 3));
    const int idx = f - (sec == 0 ? F_QKVB : (sec == 1 ? F_PROJB : (sec == 2 ? F_FC1B : F_FC2B)));
    const int col = 8 * (idx / 16) + 2 * ((idx % 16) / 4) + (idx & 1);
    float v;
    if (sec == 0) {
      const int third = col / 32, n = third * 32 + chan_of_pos(col % 32);
      v = a.qkvb ? a.qkvb[n] : 0.f;
      for (int k = 0; k < 32; ++k) v = fmaf(a.qkvw[n * 32 + k], a.n1b[k], v);  // b' = b + W beta
      v *= (third == 0 ? a.q_scale : 1.0f);
    } else if (sec == 1) {
      v = a.projb[col];
    } else if (sec == 2) {
      v = a.fc1b[col];
      for (int k = 0; k < 32; ++k) v = fmaf(a.fc1w[col * 32 + k], a.n2b[k], v);
    } else {
      v = a.fc2b[col];
    }
    a.dst[i] = __float_as_uint(v);
  }
}

}  // namespace

#ifndef MPL_SPT_ALT
bool spt_fused_supports(int J_, int d, int H, int hidden) { return J_ == J && d == D && H == HEADS && hidden == HID; }
size_t spt_fused_layer_bytes() { return (size_t)LAYER_WORDS_FULL * 4; }

int launch_spt_pack_layer(const float* n1w, const float* n1b, const float* qkvw, const float* qkvb, const float* projw,
                          const float* projb, const float* n2w, const float* n2b, const float* fc1w, const float* fc1b,
                          const float* fc2w, const float* fc2b, float scale, void* dst, cudaStream_t s) {
  SptPackArgs a{n1w, n1b, qkvw, qkvb, projw, projb, n2w, n2b, fc1w, fc1b, fc2w, fc2b, reinterpret_cast<uint32_t*>(dst),
                scale * 1.4426950408889634f};
  spt_pack_kernel<<<(LAYER_WORDS_FULL + 255) / 256, 256, 0, s>>>(a);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

int launch_spt_fused(const float* x_in, float* x_out, const void* const* wpack_per_view, int V, int64_t B, int depth,
                     const float* sn_w, const float* sn_b, const float* conf, int conf_weighted, const SptIo* io,
                     int precise, cudaStream_t s) {
  if (B == 0 || V == 0) return MPL_OK;
  if ((x_in == nullptr || x_out == nullptr) && io == nullptr) {
    set_error("launch_spt_fused: fused embedding / token build need their argument blocks");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  SptArgs a{};
  a.x_in = x_in;
  a.x_out = x_out;
  a.conf_weighted = conf_weighted;
  a.group = 1;
  a.rows_used = ROWS;
  a.final_norm = 1;
  if (io != nullptr) a.io = *io;
  for (int v = 0; v < V; ++v) a.wpack[v] = reinterpret_cast<const uint32_t*>(wpack_per_view[v]);
  a.sn_w = sn_w;
  a.sn_b = sn_b;
  a.conf = conf;
  a.B = B;
  a.depth = depth;
  // per device: function attributes live in the device's context (DataParallel replicas); setting one twice is harmless
  static std::atomic<unsigned char> attr_set[64][2];
  int dev = 0;
  MPL_CUDA(cudaGetDevice(&dev));
  auto kern = precise ? spt_fused_kernel_precise : spt_fused_kernel_fast<false>;
  const int smem_bytes = precise ? Smem<true>::TOTAL : Smem<false>::TOTAL;
  if (dev < 0 || dev >= 64 || !attr_set[dev][precise ? 1 : 0].load(std::memory_order_acquire)) {
    MPL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    if (dev >= 0 && dev < 64) attr_set[dev][precise ? 1 : 0].store(1, std::memory_order_release);
  }
  dim3 grid((unsigned)ceil_div(B, SETS), (unsigned)V);
  kern<<<grid, THREADS, smem_bytes, s>>>(a);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

int launch_fpt_kp_fused_alt(float* tok, const void* wpack, int V, int64_t B, int depth, cudaStream_t s);  // the 16-set object
#endif  // !MPL_SPT_ALT

// The keypoint-token FPT stack (bf16 mode) in one launch: tok [B, V * 17, 32] fp32 updated in place by depth + 1 block
// applications (last block twice, multiview_mpl.py:420-423), attention over the V * 17 tokens of each pose.
#ifdef MPL_SPT_ALT
int launch_fpt_kp_fused_alt(float* tok, const void* wpack, int V, int64_t B, int depth, cudaStream_t s) {
#else
int launch_fpt_kp_fused(float* tok, const void* wpack, int V, int64_t B, int depth, cudaStream_t s) {
  // whole poses per CTA tile: 14 sets hold (14 / V) * V of them, the 16-set object (16 / V) * V -- taken where that is >= 25 %
  // more of the tile (V = 5: 15 vs 10 sets, V = 8: 16 vs 8)
  if (4 * ((16 / std::max(V, 1)) * V) * SETS >= 5 * ((SETS / std::max(V, 1)) * V) * 16 && V <= 16)
    return launch_fpt_kp_fused_alt(tok, wpack, V, B, depth, s);
#endif
  if (B == 0 || depth == 0) return MPL_OK;
  if (V < 1 || V > SETS) {
    set_error("launch_fpt_kp_fused: %d views do not fit one CTA tile of %d sets", V, SETS);
    return MPL_ERR_UNSUPPORTED;
  }
  SptArgs a{};
  a.x_in = tok;
  a.x_out = tok;
  a.wpack[0] = reinterpret_cast<const uint32_t*>(wpack);
  a.B = B * V;                       // "poses" of the kernel = 17-row sets
  a.depth = depth;
  a.group = V;
  const int sets_used = (SETS / V) * V;
  a.rows_used = sets_used * J;
  a.final_norm = 0;
  static std::atomic<unsigned char> attr_set[64];
  int dev = 0;
  MPL_CUDA(cudaGetDevice(&dev));
  auto kern = spt_fused_kernel_fast<true>;
  if (dev < 0 || dev >= 64 || !attr_set[dev].load(std::memory_order_acquire)) {
    MPL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Smem<false>::TOTAL));
    if (dev >= 0 && dev < 64) attr_set[dev].store(1, std::memory_order_release);
  }
  dim3 grid((unsigned)ceil_div(B * V, sets_used), 1);
  kern<<<grid, THREADS, Smem<false>::TOTAL, s>>>(a);
  MPL_LAUNCH_CHECK();
  return MPL_OK;
}

}  // namespace mpl
