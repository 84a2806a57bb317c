// Launchers of the CUDA kernels behind mpl_forward.  Shapes use the reference's names:
// B poses, V views, J joints, d = embed_dim_ratio, H heads, D = FPT width (SURVEY.md §2.2).
#pragma once
#include "common.cuh"

namespace mpl {

constexpr int kMaxViews = 16;

// ---- K1: joint embedding (multiview_mpl.py:349-398) -------------------------------------------------------------
struct EmbedArgs {
  const float* poses[kMaxViews];
  const float* rays[kMaxViews];
  const float* centers[kMaxViews];
  const float* We[kMaxViews];  // Spatial_patch_to_embedding[.v].weight [d, in_ch]
  const float* be[kMaxViews];  //                                 .bias [d]
  const float* Wc[kMaxViews];  // confidence_to_embedding[.v].weight [d, 1] (or null)
  const float* bc[kMaxViews];
  const float* Ps[kMaxViews];  // Spatial_pos_embed[.v] [J, d]
  const float* pos3d;          // add_3D_pos_encoding_in_Spatial: learnable table [J, pos3d_ld] ...
  const float* Wl;             // ... or pos_3d_linear.weight [d, 3] / .bias
  const float* bl;
  int64_t pose_stride, center_stride, B;
  int pos3d_ld, in_ch, add_conf, mult_conf, spatial_pos_mode;  // 0 none, 1 learnable, 2 linear(normalize(ray-center))
  int V, J, d;
  float* x;     // [V, B, J, d]
  float* conf;  // [V, B, J] or null (confidence_as_attention_uncertainty_weight)
};
int launch_embed(const EmbedArgs& a, cudaStream_t s);
int try_launch_embed_vec(const EmbedArgs& a, cudaStream_t s);  // io_kernels.cu: MPL_OK if launched, 1 if the generic kernel is needed

// ---- FPT token build (multiview_mpl.py:463-499) ------------------------------------------------------------------
struct TokenArgs {
  const float* xn;  // Spatial_norm output [V, B, J, d]
  const float* poses[kMaxViews];
  const float* rays[kMaxViews];
  const float* centers[kMaxViews];
  int64_t pose_stride, center_stride, B;
  const float* Wcf;  // confidence_to_embedding_FPT weight [d,1] / bias (or null)
  const float* bcf;
  const float* Wr;  // ray_to_embedding [d,3] / bias (or null)
  const float* br;
  const float* pos_table;  // learnable pos_3d_embed / pos_3d_view_coding [J, pos_w] (or null)
  const float* Wl;         // pos_3d_linear [pos_w, 3] / bias (used when pos_table == null)
  const float* bl;
  int pos_w;
  int ray_layout;  // 0 none, 1 interleave (cat dim=2), 2 append (cat dim=1)
  int V, J, d, tok_w;
  float* tok;           // [B, V, tok_w] fp32
  int perm_layout;      // ray_layout 1 written as [J pose parts | J ray parts] (channel-permuted residual stream, model.cu)
  // LayerNorm-fused bf16 mode behind the single-kernel SPT: the token rows leave as the two bf16 planes of the FPT residual
  // stream (hi, lo) together with their per-row (sum, sum^2) in statistics slot 0 -- what launch_ln_prep would make of `tok`
  __nv_bfloat16* tok_hi;
  __nv_bfloat16* tok_lo;
  float2* stats;        // [slots][stats_ld]
  int stat_slots;
  int64_t stats_ld;
};
int launch_token_build(const TokenArgs& a, cudaStream_t s);
int try_launch_token_build_vec(const TokenArgs& a, cudaStream_t s);

// ---- LayerNorm over the last dim; column e of the output reads input column (e / seg_len) * seg_stride + e % seg_len
int launch_layernorm(const float* x, int64_t ldx, int seg_len, int seg_stride, const float* w, const float* b, float eps,
                     float* y, int64_t ldy, int64_t rows, int C, cudaStream_t s);
// same, bf16 output (A operand of the tcgen05 projections)
int launch_layernorm_bf16(const float* x, int64_t ldx, const float* w, const float* b, float eps, __nv_bfloat16* y,
                          int64_t ldy, int64_t rows, int C, cudaStream_t s);
// same, split bf16 planes out (A operand of the fp32-grade split-mode projections): hi at y, lo at y + plane
int launch_layernorm_split(const float* x, int64_t ldx, const float* w, const float* b, float eps, __nv_bfloat16* y,
                           int64_t ldy, int64_t plane, int64_t rows, int C, cudaStream_t s);

// entry of the LayerNorm-fused FPT: the fp32 token rows as two bf16 planes (hi = bf16(x), lo = bf16(x - hi), row pitch ldb)
// + their (sum, sum^2) in statistics slot 0 of `slots`
int launch_ln_prep(const float* x, int64_t ldx, __nv_bfloat16* x_hi, __nv_bfloat16* x_lo, int64_t ldb, void* stats, int slots,
                   int64_t rows, int C, cudaStream_t s);
// hi + lo planes -> fp32 (the heads that are not served by the plane-reading head kernel)
int launch_join_planes(const __nv_bfloat16* hi, const __nv_bfloat16* lo, float* out, int64_t n, cudaStream_t s);
// pack time: W' = bf16(W diag(gamma)), colsum = row sums of W', bias' = b + W beta
int launch_ln_fold(const float* W, const float* b, const float* gamma, const float* beta, __nv_bfloat16* Wf, float* colsum,
                   float* bias_f, int N, int K, cudaStream_t s, const int* kperm = nullptr);

// ---- fp32 CUDA-core Linear: Y = act(X W^T + bias) (+ R) ------------------------------------------------------------
int launch_linear_f32(const float* X, int64_t lda, const float* W, const float* bias, const float* R, int64_t ldr,
                      float* Y, int64_t ldc, int64_t M, int N, int K, int act, cudaStream_t s);

// ---- generic attention core over sets of N tokens (multiview_mpl.py:53-64): qkv [sets*N, 3C] -> out [sets*N, C] ---
// conf (or null): [sets*N] post-softmax query-row scale (multiview_mpl.py:61-62)
int launch_attention_f32(const float* qkv, float* out, int64_t sets, int N, int H, int hd, float scale, const float* conf,
                         cudaStream_t s);
// bf16 in / bf16 out variant used behind the tensor-core QKV projection
int launch_attention_bf16(const __nv_bfloat16* qkv, __nv_bfloat16* out, int64_t sets, int N, int H, int hd, float scale,
                          cudaStream_t s);
// fp32 in / split bf16 planes out (hi at out, lo at out + plane); scratch: [sets * N, H * hd] fp32 for the shapes the
// view-token kernel does not serve
int launch_attention_split(const float* qkv, __nv_bfloat16* out, int64_t plane, float* scratch, int64_t sets, int N, int H,
                           int hd, float scale, cudaStream_t s);

// ---- Conv1d(V -> 1, k = 1) over the view axis (multiview_mpl.py:281,445): y[b,e] = sum_v w[v] x[b,v,e] + bias -------
int launch_view_mean(const float* x, const float* w, const float* bias, float* y, int64_t B, int V, int E, cudaStream_t s);

// ---- K5: fused head for the default head (multiview_mpl.py:425-446,517-523):
//      strip ray channels -> View_norm -> view-weighted mean -> LayerNorm(1e-5) -> Linear(E -> 3J) ------------------
struct HeadArgs {
  const float* tok;  // [B, V, tok_w] fp32 residual stream after the FPT ...
  const __nv_bfloat16* tok_hi;  // ... or (LayerNorm-fused bf16 mode) its two bf16 planes, same shape; tok is ignored when set
  const __nv_bfloat16* tok_lo;
  int64_t B;
  int V, tok_w, E, seg_len, seg_stride, out_dim;
  const float* vn_w; const float* vn_b;  // View_norm
  const float* wm_w; const float* wm_b;  // weighted_mean (Conv1d) [V], [1]
  const float* hn_w; const float* hn_b;  // head.0 LayerNorm
  const float* hw;   const float* hb;    // head.1 Linear [out_dim, E]
  const float* hwT;                      // the same weight x 2^10, split into fp16 hi / lo parts in mma B-fragment order
                                         // (launch_head_transpose; E * 64 floats reserved), or null: generic kernel
  float* out;                            // [B, out_dim]
};
int launch_head_fused(const HeadArgs& a, cudaStream_t s);
int try_launch_head_warp(const HeadArgs& a, cudaStream_t s);
bool head_warp_supports(const HeadArgs& a);  // shape test of the K5 kernel (E, out_dim, seg_len, seg_stride, tok_w)
int launch_head_transpose(const float* W, float* WT, int out_dim, int E, cudaStream_t s);

// ---- pack helpers ---------------------------------------------------------------------------------------------------
// Linear followed by eval-mode BatchNorm1d folded into one Linear: W' = W * g / sqrt(var + eps), b' = (b - mean) * g / sqrt(var+eps) + beta
int launch_fold_bn(const float* W, const float* b, const float* g, const float* beta, const float* mean, const float* var,
                   float eps, float* Wf, float* bf, int N, int K, cudaStream_t s);
int launch_to_bf16(const float* src, __nv_bfloat16* dst, int64_t n, cudaStream_t s);
int launch_to_f16(const float* src, void* dst, int64_t n, cudaStream_t s);
// Channel-permuted residual stream (model.cu, MplModel::perm): dst row n = src row perm[n] of a [N, K] matrix, as bf16 or
// fp16; dst[i] = src[perm[i]] for a vector
int launch_to_half_rows(const float* src, void* dst, int N, int K, const int* perm, int fp16, cudaStream_t s);
int launch_gather_f32(const float* src, float* dst, int n, const int* perm, cudaStream_t s);
int launch_to_split(const float* src, __nv_bfloat16* dst, int64_t n, int64_t plane, cudaStream_t s);  // hi at dst, lo at dst + plane

// ---- tcgen05 projection GEMM (gemm_tcgen05.cu) ----------------------------------------------------------------------
enum GemmEpilogue { EPI_BIAS = 0, EPI_BIAS_GELU = 1, EPI_BIAS_RESIDUAL = 2, EPI_LN_BIAS = 4, EPI_LN_BIAS_GELU = 5, EPI_RESIDUAL_EMIT = 6 };
// LayerNorm fused around the bf16 projections (see gemm_tcgen05.cu):
//   EPI_RESIDUAL_EMIT  the residual stream x [M, N] is two bf16 planes, hi = Y and lo = x_lo (x ~ hi + lo): x += A W^T + bias in
//                      place on both planes (TMA in, TMA out), plus per-row partial (sum, sum^2) of the new x into stats_out
//                      [gemm_ln_slots(N)][M rounded up to 256] float2 (slot-major; rows past M are scratch).  N % 16 == 0;
//   EPI_LN_BIAS(_GELU) Y = act(rstd * (A W'^T - mu * colsum) + bias) with A = the hi plane (raw residual rows), W' = W diag(gamma),
//                      bias = b + W beta, (mu, rstd) from stats_in [slots_in][M rounded up to 256].
struct GemmLnArgs {
  const float* colsum;
  const void* stats_in;
  void* stats_out;
  void* x_lo;
  int slots_in;
  float eps;
  int ab_fp16;   // A and W hold fp16 (not bf16) values
  int out_fp16;  // EPI_LN_BIAS(_GELU): write fp16 (not bf16); the GELU then runs in packed half2 arithmetic
  int ldy;       // residual-emit: row pitch (elements) of the two residual planes when only their first N columns are
                 // updated (0 = N)
};
int gemm_ln_slots(int N);
// A [M,K] row-major (lda = K), W [N,K] row-major.  dtype MPL_PREC_BF16: bf16 matrices.  dtype MPL_PREC_TF32 (the fp32-grade
// "split" mode): every matrix is TWO bf16 planes, [2][rows][K] = hi = bf16(x) then lo = bf16(x - hi), and the kernel
// accumulates hi.hi + hi.lo + lo.hi.  EPI_BIAS / EPI_BIAS_GELU write Y [M,N] in the operand format (bf16, or two planes
// [2][M][N]) or fp32 if out_fp32; EPI_BIAS_RESIDUAL does Y(fp32) += A W^T + bias in place.
int launch_gemm_tcgen05(const void* A, const void* W, const float* bias, void* Y, int64_t M, int N, int K, int dtype,
                        int epilogue, int out_fp32, cudaStream_t s, const GemmLnArgs* ln = nullptr);
bool gemm_tcgen05_supports(int N, int K, int dtype);

// QKV projection + cross-view attention fused (bf16 mode, LayerNorm folded; D = H * 136 or H * 68 with H even, 2 <= V <= 8): att [M, D] bf16 straight
// from the raw residual rows xb [M, D] bf16 + their statistics -- no q|k|v tensor.  Wp / colsum / bias_f come from
// launch_qkv_attn_pack (W [3D, D], b [3D] or null, LayerNorm gamma / beta, softmax scale).
bool qkv_attn_supports(int D, int H, int tokens);
size_t qkv_attn_weight_elems(int D, int H);  // bf16 elements of Wp
int qkv_attn_vec_len(int D, int H);          // floats of colsum / bias_f
// kperm (or null): input channel k of the packed matrix is channel kperm[k] of W / gamma / beta
int launch_qkv_attn_pack(const float* W, const float* b, const float* gamma, const float* beta, void* Wp, float* colsum,
                         float* bias_f, int H, int D, float scale, cudaStream_t s, const int* kperm = nullptr);
int launch_qkv_attn(const void* xb, const void* Wp, const float* bias_f, const float* colsum, const void* stats, int slots,
                    float eps, void* att, int64_t M, int D, int H, int V, cudaStream_t s);

// ---- K2: fused Spatial Pose Transformer stack (spt_fused.cu) ---------------------------------------------------------
bool spt_fused_supports(int J, int d, int H, int hidden);
size_t spt_fused_layer_bytes();
int launch_spt_pack_layer(const float* n1w, const float* n1b, const float* qkvw, const float* qkvb, const float* projw,
                          const float* projb, const float* n2w, const float* n2b, const float* fc1w, const float* fc1b,
                          const float* fc2w, const float* fc2b, float scale, void* dst, cudaStream_t s);
// x_in / x_out [V, B, 17, 32] fp32; wpack_per_view[v] -> [depth] fragment-packed layers (the softmax scale is folded
// into them by launch_spt_pack_layer); applies every block application of the stack (confidence-weighted pass when
// conf_weighted, last block twice) and Spatial_norm.  x_in == null: the K1 joint embedding is computed in the kernel's
// prologue from io->embed (spatial_pos_mode 0 / 1 only); x_out == null: the FPT tokens are written by its epilogue from
// io->token (tok, layouts, ray / confidence / position embeddings) -- no embed / token-build launch, no xs / xn round trip.
struct SptIo {
  EmbedArgs embed;
  TokenArgs token;
};
int launch_spt_fused(const float* x_in, float* x_out, const void* const* wpack_per_view, int V, int64_t B, int depth,
                     const float* sn_w, const float* sn_b, const float* conf, int conf_weighted, const SptIo* io,
                     int precise, cudaStream_t s);  // precise: fp32 softmax arithmetic + exact erf GELU (tf32 mode)

// the keypoint-token FPT stack (FPT_blocks_view_keypoint_tokens, width 32, 8 heads, bf16 mode) as one launch of the
// same kernel: tok [B, V * 17, 32] fp32 in place, wpack = [depth] layers packed by launch_spt_pack_layer from blocks.{l}.*
int launch_fpt_kp_fused(float* tok, const void* wpack, int V, int64_t B, int depth, cudaStream_t s);

// ---- metric + input builder -----------------------------------------------------------------------------------------
// room_affine: host pointer to 6 floats (scale xyz, offset xyz) or null -- the room un-scaling of function_mpl.py:476-488
// G = 0: mpl_mpjpe_accumulate (group ignored); G >= 1: mpl_mpjpe_accumulate_grouped, acc [G][11 J + 1]
int launch_mpjpe_accumulate(const float* pred, const float* gt, const float* conf3d, const int32_t* group, int G, int64_t B,
                            int J, float unit_scale, const float* room_affine, double* acc, cudaStream_t s);
// G = 0: mpl_pmpjpe_accumulate (mask, group ignored); G >= 1: mpl_pmpjpe_accumulate_masked, acc [G][2 J + 4]
int launch_pmpjpe_accumulate(const float* pred, const float* gt, const float* mask, const int32_t* group, int G, int64_t B,
                             int J, float unit_scale, int scaling, int reflection, double* acc, cudaStream_t s);
// calib_stride: 0 = one calib [V, 18] for every pose; else pose b reads calib + b * calib_stride (>= 18 V, checked by the caller)
int launch_build_inputs(const float* pix, const double* calib, int64_t calib_stride, int64_t B, int V, int J, float* poses,
                        float* rays, float* centers, cudaStream_t s);
int launch_synth_project(uint64_t seed, int64_t start, int64_t B, int V, int J, const double* calib, int64_t calib_stride,
                         const double* room, int conf_ones, float* pix, float* target, cudaStream_t s);
int launch_triangulate(const float* pix, const double* calib, int64_t calib_stride, int64_t B, int V, int J, float min_conf,
                       float* points, int32_t* views_used, cudaStream_t s);
int launch_triangulate_robust(const float* pix, const double* calib, int64_t calib_stride, int64_t B, int V, int J,
                              float min_conf, float inlier_px, float* points, int32_t* inliers, cudaStream_t s);
int launch_triangulate_refine(const float* pix, const double* calib, int64_t calib_stride, int64_t B, int V, int J,
                              float min_conf, const int32_t* view_mask, const float* init, int max_iters, float* points,
                              float* reproj_px, cudaStream_t s);
int launch_detector_noise(uint64_t seed, int64_t start, int64_t B, int V, int J, const double* calib, int64_t calib_stride,
                          float sigma_px, float p_outlier, float p_miss, float* pix, cudaStream_t s);
int launch_synth_cameras(uint64_t seed, int64_t start, int64_t B, int V, double f0, double w, double h, const double* room,
                         double* calib, cudaStream_t s);
// mpl_undistort_pixels (undistort) or mpl_distort_pixels (margins ignored); strides checked by the caller
int launch_synth_calib_noise(uint64_t seed, int64_t start, int64_t B, int V, const double* calib, int64_t calib_stride,
                             double sigma_rot, double sigma_pos, double* calib_out, cudaStream_t s);
size_t rig_workspace_bytes(int64_t B, int V, int J);
int launch_calibrate_rig(const float* pix, const double* calib, int64_t B, int V, int J, float min_conf,
                         const int32_t* view_mask, const float* init, double sigma_px, double sigma_rot, double sigma_pos,
                         int max_iters, double* calib_out, float* points, double* report, void* workspace, cudaStream_t s);
int launch_lens_pixels(bool undistort, const float* pin, float* pout, const double* calib, int64_t calib_stride,
                       const double* dist, int64_t dist_stride, double margin_x, double margin_y, int64_t B, int V, int J,
                       cudaStream_t s);
// associate.cu: multi-person scenes, association, gathering and scoring (argument checks in model.cu)
int launch_synth_people(uint64_t seed, int64_t start, int64_t F, int P, int V, int J, const float* pix, float* scene,
                        int32_t* perm, cudaStream_t s);
int launch_associate_people(const float* scene, const double* calib, int64_t calib_stride, int64_t F, int P, int V, int J,
                            float min_conf, int min_joints, double max_dist, int K, int32_t* members, int32_t* labels,
                            int32_t* people, cudaStream_t s);
int launch_gather_people(const float* scene, const int32_t* members, int64_t F, int P, int K, int V, int J, float* out,
                         cudaStream_t s);
int launch_association_score(const int32_t* members, const int32_t* labels, const int32_t* perm, int64_t F, int P, int K,
                             int V, int32_t* owner, double* acc, cudaStream_t s);
// track.cu: people that move, tracking of person rows across frames and its score (argument checks in model.cu)
int launch_synth_motion(uint64_t seed, int64_t start, int64_t S, int T, int P, int V, int J, const double* calib,
                        int64_t calib_stride, const double* room, double fps, int conf_ones, float* pix, float* target,
                        cudaStream_t s);
size_t track_state_bytes(int max_tracks, int J);
int launch_track_people(const float* points, const float* joint_mask, int64_t S, int64_t T, int K, int J, int min_joints,
                        double max_dist, int max_age, int max_tracks, void* state, int32_t* track_id, cudaStream_t s);
int launch_tracking_score(const int32_t* track_id, const int32_t* owner, int64_t S, int64_t T, int K, int P, double* acc,
                          cudaStream_t s);

}  // namespace mpl
