/*
 * mpl_b200.h — C ABI of the B200-native MPL lifter forward.
 *
 * One shared library (libmpl_b200.so, hand-written CUDA for sm_100a) replaces the PyTorch-eager forward of the
 * reference's lifting network.  Every entry point cites the reference interface it stands in for
 * (paths relative to the reference checkout, aghasemzadeh/OpenMPL):
 *
 *   MPL/lib/models/multiview_mpl.py:95-317   MultiView_MPL.__init__  (constructor kwargs  -> MplDesc / mpl_create)
 *   MPL/lib/models/multiview_mpl.py:450-525  MultiView_MPL.forward   (poses, rays, centers -> mpl_forward)
 *   MPL/lib/utils/utils.py:148-153           load_state_dict of checkpoints (-> mpl_param_* / mpl_pack_weights)
 *   MPL/lib/core/evaluate.py:91-125          calc_mpjpe / calc_distance_per_dim (-> mpl_mpjpe_accumulate)
 *   MPL/lib/utils/pose_utils.py:61-143       PoseUtils.procrustes (-> mpl_pmpjpe_accumulate)
 *   MPL/lib/dataset/joints_dataset_mpl.py:615-648,701-715,762-772,817-820,872-904
 *                                            per-sample input construction (-> mpl_build_inputs)
 *   MPL/lib/multiviews/triangulate.py:59-115 linear triangulation baseline (-> mpl_triangulate)
 * Defined here, with no counterpart in the reference: robust (RANSAC) triangulation (mpl_triangulate_robust), nonlinear
 * refinement of triangulated points (mpl_triangulate_refine), a detector-error model for the synthetic data
 * (mpl_synth_detector_noise), a generator of random camera setups (mpl_synth_cameras), lens distortion of pixels
 * (mpl_distort_pixels / mpl_undistort_pixels), a calibration-error model (mpl_synth_calib_noise) and bundle adjustment of a
 * rig's extrinsics from its detections (mpl_calibrate_rig), and multi-person scenes with the association of detections
 * across views (mpl_synth_people, mpl_associate_people, mpl_gather_people, mpl_association_score), and people that move
 * with the tracking of person rows across frames (mpl_synth_motion, mpl_track_people, mpl_tracking_score).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - the library never allocates user-visible device memory: inputs, outputs, the packed weight blob and the
 *     workspace are caller-owned device buffers, borrowed for the duration of the call;
 *   - all work is enqueued on the caller's stream on the caller's current device; no hidden synchronisation;
 *   - every function returns MPL_OK (0) or a negative MplStatus; mpl_last_error() gives the thread-local message;
 *   - entry points are re-entrant; a handle may be used from one thread at a time (one handle per device replica,
 *     like one nn.Module replica per GPU in the reference's DataParallel, MPL/run/valid_mpl.py:177-178);
 *   - calibrations: every entry point that reads `calib` has a *_strided variant with an int64_t calib_stride, the number
 *     of doubles between the [V, 18] calibration blocks of consecutive poses (like the pose_stride / center_stride of
 *     mpl_forward).  0 = one block for the whole batch (the plain entry point, which forwards with 0); >= 18 V = pose b
 *     uses calib + b * calib_stride (a packed [B, V, 18] tensor: 18 V).  Any other value is MPL_ERR_INVALID_ARGUMENT,
 *     before any CUDA call.  With the same block in every pose the results are bitwise those of stride 0.  A real
 *     validation batch mixes calibrations (the reference reads each sample's camera from its own db record,
 *     joints_dataset_mpl.py:499-512), so it needs no splitting by camera.
 */
#ifndef MPL_B200_H_
#define MPL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPL_ABI_VERSION 11

typedef enum MplStatus {
  MPL_OK = 0,
  MPL_ERR_INVALID_ARGUMENT = -1, /* bad pointer / size / struct_size                                             */
  MPL_ERR_CONFIG_RUNTIME = -2,   /* flag combination whose first forward raises RuntimeError in the reference    */
  MPL_ERR_CONFIG_INDEX = -3,     /* flag combination whose first forward raises IndexError in the reference      */
  MPL_ERR_CUDA = -4,             /* a CUDA runtime / driver call failed                                           */
  MPL_ERR_WORKSPACE = -5,        /* workspace or packed buffer too small                                          */
  MPL_ERR_UNSUPPORTED = -6       /* requested precision mode cannot serve this shape (no silent fallback)         */
} MplStatus;

/* Arithmetic of the Linear layers.  LayerNorm, softmax, residual stream and all accumulators are fp32 in every mode. */
typedef enum MplPrecision {
  MPL_PREC_FP32 = 0, /* fp32 operands, fp32 FMA (CUDA cores)                                        */
  MPL_PREC_TF32 = 1, /* the fp32-grade tensor-core mode (the "fp32/TF32 path" of the parity contract): FPT projections
                        on tcgen05 with every operand split into two bf16 planes (hi + lo, 16 significand bits) and
                        hi.hi + hi.lo + lo.hi accumulated in fp32 -- single-pass kind::tf32 (11 bits) cannot hold the
                        1e-3 bound on every shipped configuration; LayerNorm / attention / head fp32               */
  MPL_PREC_BF16 = 2  /* FPT projections: tcgen05 kind::f16 bf16 operands; SPT: bf16 mma; fp32 accum */
} MplPrecision;

/* POD mirror of the keyword arguments of MultiView_MPL.__init__ (multiview_mpl.py:95-117).
 * Dropout / drop-path rates are omitted: the path is inference only (identity in eval, multiview_mpl.py:79). */
typedef struct MplDesc {
  int32_t struct_size; /* = sizeof(MplDesc); ABI guard */
  int32_t num_joints;
  int32_t in_chans;
  int32_t embed_dim_ratio;
  int32_t depth;
  int32_t num_heads;
  int32_t num_views;
  int32_t hidden_dim;
  float mlp_ratio;
  float qk_scale; /* 0 = None -> head_dim^-0.5 (multiview_mpl.py:46) */
  int32_t qkv_bias;
  int32_t add_confidence_input;
  int32_t mult_confidence_emb;
  int32_t concat_confidence_emb;
  int32_t confidence_input_as_third;
  int32_t pose_3d_emb_learnable;
  int32_t linear_weighted_mean;
  int32_t add_3D_pos_encoding_in_Spatial;
  int32_t input_rays_as_token;
  int32_t add_3D_pos_encoding_to_rays;
  int32_t confidence_as_attention_uncertainty_weight;
  int32_t multiple_spatial_blocks;
  int32_t no_transformer_spt;
  int32_t no_transformer_fpt;
  int32_t confidence_in_FPT;
  int32_t deep_head;
  int32_t head_kadkhod;
  int32_t FPT_blocks_view_keypoint_tokens;
  int32_t precision; /* MplPrecision */
  /* implementation switches (not reference keywords); 0-initialised fields select the defaults */
  int32_t ln_fusion;      /* bf16 mode: fold the FPT LayerNorms into the projection GEMMs.  0 = separate LayerNorm kernels,
                             non-zero (make_desc default: 1) = fused: the GEMM that updates the residual stream also emits
                             the next GEMM's operand and per-row (sum, sum^2); the next GEMM multiplies the raw rows by
                             W diag(gamma) and applies (mean, rstd) in its epilogue */
  int32_t gemm_cta_group; /* must be 0 or 2: every projection GEMM tile is 256x256 on a CTA pair (cta_group::2, cluster
                             2x1x1).  Kept so that the struct layout stays; any other value is MPL_ERR_INVALID_ARGUMENT */
  int32_t spt_hidden, fpt_hidden; /* int(width * mlp_ratio) of the SPT / FPT Mlp as the reference's float64 arithmetic gives it
                                     (0 = derive from the float mlp_ratio above) */
  int32_t qkv_attn_fusion; /* bf16 LayerNorm-fused mode, view tokens, 136-wide heads (or an even number of 68-wide ones), 2 to 8 views: QKV projection and
                              cross-view attention run as ONE kernel (no q|k|v tensor).  0 = two kernels, non-zero (make_desc
                              default: 1) = fused where the shape allows */
  int32_t chunk_streams;  /* must be 0 or 1: the pose chunks of a forward run one at a time on the caller's stream.  Kept
                             so that the struct layout stays; any other value is MPL_ERR_INVALID_ARGUMENT */
} MplDesc;

typedef struct MplModel MplModel;          /* opaque host-side handle */
typedef struct CUstream_st* mpl_stream_t;  /* == cudaStream_t */

/* Thread-local message of the last failing call on this thread ("" if none). */
const char* mpl_last_error(void);
int mpl_abi_version(void);

/* MultiView_MPL.__init__ (multiview_mpl.py:95-317).  Host only.  Invalid flag combinations fail here with the
 * status class of the exception the reference raises at its first forward (SURVEY.md §3.2-Q6). */
int mpl_create(const MplDesc* desc, MplModel** out);
void mpl_destroy(MplModel* m);

/* state_dict contract (utils.py:148-153): entry i has the reference's key (without the `features.` prefix of
 * MultiView_MPL_G) and element count; order = registration order of the reference module. */
int mpl_num_params(const MplModel* m);
int mpl_param_info(const MplModel* m, int index, const char** name, int64_t* numel, int32_t* is_int64);

/* Derived dims (multiview_mpl.py:140-142,272-274): which = 0 tok_w, 1 fpt_dim, 2 fpt_tokens, 3 E, 4 spt_hidden,
 * 5 fpt_hidden, 6 outputs (1, or 3 for head_kadkhod), 7 output columns the LAST fc2 of the FPT stack computes (E where the
 * residual stream is kept channel-permuted and the head reads its pose half only, else fpt_dim). */
int64_t mpl_dim(const MplModel* m, int which);

/* Weight repack: fp32 state_dict tensors (device pointers, in mpl_param_info order) -> one caller-owned blob
 * holding what the kernels read (fp32 copies, BatchNorm folded into the preceding Linear, bf16 / tf32 operand
 * copies of the FPT projection matrices).  Call again after the parameters change. */
size_t mpl_packed_bytes(const MplModel* m);
int mpl_pack_weights(MplModel* m, const void* const* params, int num_params, void* packed, size_t packed_bytes,
                     mpl_stream_t stream);

/* Workspace for batches of up to `max_batch` poses (the forward processes larger batches in chunks of
 * mpl_chunk_poses(), so the workspace stops growing there). */
size_t mpl_workspace_bytes(const MplModel* m, int64_t max_batch);
int64_t mpl_chunk_poses(const MplModel* m);
int mpl_set_chunk_poses(MplModel* m, int64_t chunk);

/* MultiView_MPL.forward (multiview_mpl.py:450-525), eval mode.
 *   poses[v]   -> view v 2D joints (x, y, conf)  [B, J, 3] fp32, consecutive poses `pose_stride` floats apart
 *   rays[v]    -> view v ray points              [B, J, 3] fp32, same stride
 *   centers[v] -> view v camera centre           [B, 1, 3] fp32, consecutive poses `center_stride` floats apart
 *                 (the reference's list-of-views convention, core/function_mpl.py:344-350, is V separate
 *                  tensors: stride J*3 and 3; one packed [B,V,J,3] tensor is the same call with stride V*J*3)
 *   out        -> [B, J, 3] fp32;  aux1/aux2 -> the two intermediate predictions of head_kadkhod (else NULL)
 * The pointer arrays are host arrays of V device pointers. */
int mpl_forward(MplModel* m, const void* packed, const float* const* poses, const float* const* rays,
                const float* const* centers, int64_t pose_stride, int64_t center_stride, float* out, float* aux1,
                float* aux2, int64_t batch, void* workspace, size_t workspace_bytes, mpl_stream_t stream);

/* Small-batch path (the reference's runner calls the model at TEST.BATCH_SIZE = 256, configs/h36m/mpl_amass/hm_0_*.yaml:144,
 * MPL/run/valid_mpl.py:205-210, where ~130 launches per forward are latency-bound): with max_batch > 0, an mpl_forward of at most
 * max_batch poses is captured ONCE per (batch, packed, input / output / workspace pointers) as a CUDA graph and later calls
 * with the same arguments replay it with a single graph launch on the caller's stream.  The caller keeps those buffers
 * alive and at the same addresses (the nn.Module stages inputs in persistent buffers for this).  Up to 16 graphs are kept
 * per handle (least recently used evicted); 0 switches the path off and frees them.  A stream that is itself being
 * captured, and profiling mode, take the plain path. */
int mpl_set_graph_batch(MplModel* m, int64_t max_batch);
int mpl_graph_stats(const MplModel* m, int64_t* captures, int64_t* replays);

/* Number of kernel launches the last mpl_forward on this handle enqueued (bench.py's gpu_launches). */
int64_t mpl_last_launch_count(const MplModel* m);

/* Optional per-launch timing with CUDA events on the caller's stream (the reference's only profiling hook is an
 * unsynchronised time.time() around the model call, core/function_mpl.py:346-351).  While enabled, every kernel
 * launch of mpl_forward is bracketed by two events; mpl_profile_collect waits for the last forward's events and
 * returns milliseconds and launch counts per kernel category (mpl_profile_category_name).  Any non-zero `enabled`
 * profiles; the launches run one after the other on the caller's stream, so the per-category times add up to the step. */
int mpl_set_profile(MplModel* m, int enabled);
int mpl_profile_categories(void);
const char* mpl_profile_category_name(int category);
int mpl_profile_collect(MplModel* m, double* ms_per_category, int64_t* launches_per_category, int n);

/* calc_mpjpe / calc_distance_per_dim (evaluate.py:91-125) + the unit / root-centring / confidence-mask rules of
 * core/function_mpl.py:674-687, as running fp64 sums so ranks can be combined with one all-reduce.
 *   acc layout (doubles): [0,J) sum_b ||pred-gt|| per joint (absolute); [J,2J) same, root-relative;
 *   [2J,5J) sum_b |pred-gt| per joint-dim over unmasked entries (absolute); [5J,8J) same, root-relative;
 *   [8J,11J) unmasked count per joint-dim; [11J] pose count.
 *   conf3d may be NULL (no masking); unit_scale = 100 if OUTPUT_IN_METER else 1.
 *   room_affine: NULL, or a HOST array of 6 floats (scale x, y, z, offset x, y, z): the un-scaling validate() applies to the
 *   predictions and targets of room-normalised datasets before it stores them (function_mpl.py:476-488), v * scale + offset in
 *   fp32: (s, s, s, centre) for 'room_scaled_equal', (sx, sy, 1, 0, 0, 0) otherwise. */
#define MPL_METRIC_ACC_LEN(J) (11 * (J) + 1)
int mpl_mpjpe_accumulate(const float* pred, const float* gt, const float* conf3d, int64_t batch, int num_joints,
                         float unit_scale, const float* room_affine, double* acc, mpl_stream_t stream);

/* Procrustes-aligned error (P-MPJPE) as running fp64 sums: per pose, PoseUtils.procrustes(A = gt, B = pred)
 * (MPL/lib/utils/pose_utils.py:61-143) after the unit rule above, then the per-joint distances of calc_mpjpe between the
 * aligned prediction Z and gt.  scaling: 1 = similarity (the reference default), 0 = rigid.  reflection: -1 = 'best'
 * (the reference default: whatever the SVD gives), 0 = forbid, 1 = force (pose_utils.py:112-120).
 *   acc layout (doubles): [0,J) sum_b ||Z_j - gt_j||; [J] sum_b d (normalised residual); [J+1] sum_b scale;
 *   [J+2] pose count. */
#define MPL_PMETRIC_ACC_LEN(J) ((J) + 3)
int mpl_pmpjpe_accumulate(const float* pred, const float* gt, int64_t batch, int num_joints, float unit_scale,
                          int scaling, int reflection, double* acc, mpl_stream_t stream);

/* Grouped metrics (ABI 7): per-group running sums in one call, e.g. the per-action table of H36M, where a batch mixes
 * actions.  Rules shared by the two entry points below:
 *   - acc is [num_groups][L] doubles; pose b adds into block group[b] (a device array of batch int32).  A pose whose group
 *     is outside [0, num_groups) adds nothing and is counted nowhere, so -1 can mark an unlabelled pose.
 *   - group == NULL is allowed only with num_groups == 1: every pose then goes to block 0.
 *   - MPL_ERR_INVALID_ARGUMENT, before any CUDA call: num_groups outside [1, 65536], group == NULL with num_groups > 1, a null
 *     pred, gt or acc, batch < 0, num_joints < 1, and (P-MPJPE) reflection outside {-1, 0, 1}.  After these checks batch == 0
 *     returns MPL_OK without touching the pointers.
 *
 * mpl_mpjpe_accumulate_grouped: each block has the MPL_METRIC_ACC_LEN(J) layout and the masking, root-relative and room rules
 * of mpl_mpjpe_accumulate over the poses of its group, its [11 J] entry counting them.  With num_groups == 1 and every
 * group 0, block 0 is mpl_mpjpe_accumulate's result up to the order of the fp64 sums, bitwise for one pose. */
int mpl_mpjpe_accumulate_grouped(const float* pred, const float* gt, const float* conf3d, const int32_t* group,
                                 int num_groups, int64_t batch, int num_joints, float unit_scale,
                                 const float* room_affine, double* acc, mpl_stream_t stream);

/* mpl_pmpjpe_accumulate_masked: P-MPJPE over the joints each pose marks, in groups.  mask: NULL or a device [batch, J] fp32.
 *   - Joint j of pose b is used iff (mask == NULL or mask[b J + j] > 0) and its six coordinates (pred and gt) are finite, so
 *     non-finite points under a zero mask, or left unmasked, cannot poison a pose.
 *   - A pose is aligned iff it has at least 3 used joints and both centred sums of squares over them (after the unit rule)
 *     are > 0; otherwise it is skipped.  An aligned pose runs the Procrustes of mpl_pmpjpe_accumulate (unit rule, scaling,
 *     reflection rule, completion of a vanishing singular value) on its used joints only: the means (divided by the number
 *     n of used joints), the norms and the cross-covariance are taken over them, in joint order.
 *   - Per-block layout, L = MPL_PMETRIC_MASKED_ACC_LEN(J): [0, J) sum ||Z_j - gt_j|| over the aligned poses where j is used;
 *     [J, 2J) the number of those instances; [2J] sum d; [2J+1] sum scale (1 when scaling == 0); [2J+2] aligned poses;
 *     [2J+3] skipped poses.
 *   - With every joint used the per-pose arithmetic is mpl_pmpjpe_accumulate's in the same order (n = J), so a one-pose call
 *     gives bitwise its [0, J), d and scale. */
#define MPL_PMETRIC_MASKED_ACC_LEN(J) (2 * (J) + 4)
int mpl_pmpjpe_accumulate_masked(const float* pred, const float* gt, const float* mask, const int32_t* group,
                                 int num_groups, int64_t batch, int num_joints, float unit_scale, int scaling,
                                 int reflection, double* acc, mpl_stream_t stream);

/* Per-sample input construction of the dataset (joints_dataset_mpl.py:615-648,701-715,762-772,817-820,872-904),
 * batched: raw detector output (u, v, conf) in pixels + per-view calibration -> the model's poses / rays / centers.
 *   pix   [B, V, J, 3] fp32 (u, v, conf);  calib [V, 18] fp64 = R (9, row-major world->cam), t (3), fx, fy, cx, cy, w, h
 *   poses / rays [B, V, J, 3], centers [B, V, 1, 3] fp32 (packed layout accepted by mpl_forward). */
int mpl_build_inputs(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints, float* poses,
                     float* rays, float* centers, mpl_stream_t stream);
/* mpl_build_inputs with a calibration per pose: pose b reads calib + b * calib_stride (see Conventions). */
int mpl_build_inputs_strided(const float* pix, const double* calib, int64_t calib_stride, int64_t batch, int num_views,
                             int num_joints, float* poses, float* rays, float* centers, mpl_stream_t stream);

/* MHP-style synthetic data on the device (what MHP/utils.py:261-318 + MPL/lib/utils/calib.py:42-77 do to AMASS poses:
 * place a 3D pose in the room, project it through every calibration).  Pose i of `seed` depends only on (seed, start + i)
 * (numpy Philox4x64-10 stream, identical to openmpl_b200/synth.py), so any sharding of the global index range gives the
 * same data.  room [4] fp64 = (min_x, max_x, min_y, max_y); calib as in mpl_build_inputs.
 *   pix    [B, V, J, 3] fp32 raw pixels (u, v, conf) -- feed to mpl_build_inputs;  target [B, J, 3] fp32, metres. */
int mpl_synth_project(uint64_t seed, int64_t start, int64_t batch, int num_views, int num_joints, const double* calib,
                      const double* room, int conf_ones, float* pix, float* target, mpl_stream_t stream);
/* mpl_synth_project through a calibration per pose (calib + b * calib_stride for pose start + b; see Conventions).  The 3D
 * poses and confidences do not depend on the calibrations. */
int mpl_synth_project_strided(uint64_t seed, int64_t start, int64_t batch, int num_views, int num_joints, const double* calib,
                              int64_t calib_stride, const double* room, int conf_ones, float* pix, float* target,
                              mpl_stream_t stream);

/* Random camera setups for the synthetic data (defined by this library; no reference counterpart): calib_out [B, V, 18] fp64
 * in the row layout of mpl_build_inputs for poses [start, start + B), to be used with calib_stride 18 V.  Per (pose i,
 * view v), U0..U5 come from the Philox4x64-10 stream of mpl_synth_project under key (seed, 2) (pose i owns counter blocks
 * [i nb, (i + 1) nb), nb = ceil(6 V / 4); slot 6 v + m is U_m), so the result depends only on (seed, global pose index):
 *   azimuth                 a = 2 pi (v + 0.8 (U0 - 0.5)) / V + 0.3   (each camera stays in its own sector)
 *   horizontal distance     4.5 (0.75 + 0.5 U1) m from the look-at point;  height 0.9 + 1.2 U2 m
 *   look-at point           room centre ((min_x + max_x) / 2, (min_y + max_y) / 2, 0.9) + (0.5 (U3 - 0.5), 0.5 (U4 - 0.5), 0)
 *   intrinsics              fx = fy = f0 (0.8 + 0.4 U5), principal point (w / 2, h / 2), image w x h
 *   R                       rows x, y, z: z the unit optical axis towards the look-at point, x = z x (0, 0, 1) normalised,
 *                           y = z x x (image y down);  t = the camera position
 * Every U = 0.5 gives the ring camera of openmpl_b200/synth.py make_rig.  fp64; room [4] fp64 on the device as in
 * mpl_synth_project.  1 <= V <= 16, start >= 0, f0, w, h finite, f0 > 0, w > 1, h > 1.  Allocates nothing and never
 * synchronises.  batch == 0 returns MPL_OK without touching the pointers. */
int mpl_synth_cameras(uint64_t seed, int64_t start, int64_t batch, int num_views, double f0, double w, double h,
                      const double* room, double* calib_out, mpl_stream_t stream);

/* Linear multi-view triangulation of the same raw detections, the baseline a multi-view lifter is measured against
 * (MPL/lib/multiviews/triangulate.py:59-115, which calls pymvg's find3d once per joint): per (pose, joint), view v takes
 * part iff conf > min_conf and 0 < u < w - 1 and 0 < v < h - 1 (the comparisons of mpl_build_inputs, so with min_conf = 0
 * the used views are those whose confidence the lifter sees as > 0).  Each used view contributes the unweighted pixel-space
 * rows u P3 - P1 and v P3 - P2 with P = K [R | -R t] (no distortion); X~ is the right singular vector of the smallest
 * singular value of the stacked 2n x 4 matrix (Hartley & Zisserman section 12.2), X = X~[:3] / X~[3].  fp64 throughout.
 *   pix [B, V, J, 3] fp32 (u, v, conf), calib [V, 18] fp64 as in mpl_build_inputs, 1 <= V <= 16;
 *   points [B, J, 3] fp32 in world units (NaN where fewer than 2 views are used), views_used [B, J] int32.
 * Allocates nothing and never synchronises (graph-capturable).  batch == 0 returns MPL_OK without touching the pointers. */
int mpl_triangulate(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints, float min_conf,
                    float* points, int32_t* views_used, mpl_stream_t stream);
/* mpl_triangulate with a calibration per pose (see Conventions); same argument checks plus calib_stride. */
int mpl_triangulate_strided(const float* pix, const double* calib, int64_t calib_stride, int64_t batch, int num_views,
                            int num_joints, float min_conf, float* points, int32_t* views_used, mpl_stream_t stream);

/* Outlier-robust triangulation of the same detections: exhaustive-pair RANSAC with the MSAC cost, then a
 * confidence-weighted DLT refit (defined by this library; the reference has no robust triangulation).  Candidate views are
 * those of mpl_triangulate.  Per (pose, joint), in fp64:
 *   - every candidate pair (a, b), a < b in lexicographic order, gives the hypothesis X~_ab, the unweighted DLT of exactly
 *     those two views (mpl_triangulate's solve);
 *   - its cost is sum over all candidates c of min(e_c^2, inlier_px^2), e_c the pixel reprojection error through
 *     P_c = K [R | -R t], infinite where the depth (P_c3 . X~) / X~_4 is not > 0 or not finite; the lowest cost wins, an
 *     exact tie the earlier pair (no random sampling: deterministic for any batch split, graph-capturable);
 *   - the inliers are the candidates with e_c < inlier_px; with at least two of them the point is the DLT over the inliers
 *     with each view's two rows multiplied by its conf (the maximum-likelihood weighting when the pixel noise is
 *     proportional to 1 / conf).  When every candidate is an inlier and every conf is 1 the point is bitwise mpl_triangulate's.
 *   pix [B, V, J, 3] fp32 (u, v, conf), calib [V, 18] fp64 as in mpl_build_inputs, 1 <= V <= 16, inlier_px finite and > 0;
 *   points [B, J, 3] fp32 (NaN where there are fewer than 2 candidates or fewer than 2 inliers), inliers [B, J] int32
 *   bitmask of the inlier views (bit v; 0 where the point is NaN).
 * Allocates nothing and never synchronises.  batch == 0 returns MPL_OK without touching the pointers. */
int mpl_triangulate_robust(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints,
                           float min_conf, float inlier_px, float* points, int32_t* inliers, mpl_stream_t stream);
/* mpl_triangulate_robust with a calibration per pose (see Conventions); same argument checks plus calib_stride. */
int mpl_triangulate_robust_strided(const float* pix, const double* calib, int64_t calib_stride, int64_t batch, int num_views,
                                   int num_joints, float min_conf, float inlier_px, float* points, int32_t* inliers,
                                   mpl_stream_t stream);

/* Levenberg-Marquardt refinement of given 3D points on the confidence-weighted reprojection error (defined by this library;
 * the reference has no refinement).  With pixel noise of std sigma / conf the maximum-likelihood point minimises the cost C
 * below (Hartley & Zisserman section 12.3), which neither DLT above does.  Per (pose, joint) item b, j, in fp64 throughout:
 *   - views used: view v takes part iff it is a candidate of mpl_triangulate (conf > min_conf and strictly inside the image)
 *     and, when view_mask is not NULL, bit v of view_mask[b, j] is set (bits >= V are ignored).  Pass mpl_triangulate_robust's
 *     inliers to refine over them, NULL for every candidate; a views_used count is not a mask;
 *   - cost: C(X) = sum_v w_v ((p_0 / p_2 - u_v)^2 + (p_1 / p_2 - v_v)^2), w_v = conf_v^2, p = P_v [X; 1] with
 *     P_v = K [R | -R t].  C = +inf if any used view has p_2 <= 0 or a non-finite p_2;
 *   - X_0 = init converted to fp64.  The item is not refined when init is not finite, fewer than 2 views are used or C(X_0)
 *     is not finite: it gets points = init bit for bit and reproj_px = NaN;
 *   - iteration k = 1 .. max_iters: at the current X (relinearised only after an accepted step), D_v is the 2 x 3 Jacobian
 *     of pi(P_v [X; 1]) and r_v its residual; A = sum w_v D_v^T D_v, g = sum w_v D_v^T r_v.  Before the first iteration only,
 *     mu = 1e-3 max_i A_ii.  (A + mu I) delta = -g is solved by a 3 x 3 Cholesky; a pivot that is not finite and > 0
 *     rejects the step (mu *= 10; there is no delta, so the stopping test below is skipped).  If C(X + delta) < C(X) the
 *     step is accepted, X += delta and mu /= 10, otherwise rejected, mu *= 10.  The iteration stops after iteration k if
 *     |delta|_2 <= 1e-10 (|X|_2 + 1e-10), X taken at the start of the iteration, or when k = max_iters;
 *   - outputs: points = X rounded to fp32, reproj_px = sqrt(C(X) / sum_v w_v), the conf-weighted RMS pixel error at the
 *     returned fp64 X.  C(X) <= C(X_0) by construction.
 *   pix [B, V, J, 3] fp32 and calib as in mpl_triangulate, view_mask NULL or [B, J] int32, init [B, J, 3] fp32,
 *   points [B, J, 3] fp32, reproj_px [B, J] fp32.  init may equal points (in-place refinement); no other aliasing.
 *   1 <= V <= 16, J >= 1, 1 <= max_iters <= 100.  Deterministic and independent of how the batch is split; allocates
 *   nothing and never synchronises (graph-capturable).  batch == 0 returns MPL_OK without touching the pointers. */
int mpl_triangulate_refine(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints,
                           float min_conf, const int32_t* view_mask, const float* init, int max_iters, float* points,
                           float* reproj_px, mpl_stream_t stream);
/* mpl_triangulate_refine with a calibration per pose (see Conventions); same argument checks plus calib_stride. */
int mpl_triangulate_refine_strided(const float* pix, const double* calib, int64_t calib_stride, int64_t batch,
                                   int num_views, int num_joints, float min_conf, const int32_t* view_mask,
                                   const float* init, int max_iters, float* points, float* reproj_px,
                                   mpl_stream_t stream);

/* Detector-error model for the synthetic pixels of mpl_synth_project, applied in place (defined by this library; the
 * reference's data carries the errors of a real detector).  pix [B, V, J, 3] (u, v, conf) of poses [start, start + B);
 * only w and h of calib [V, 18] are read.  Entries with conf == 0 are left alone.  Each other entry draws U0..U5 from the
 * Philox4x64-10 stream of mpl_synth_project under key (seed, 1) (pose i owns counter blocks [i nb, (i + 1) nb),
 * nb = ceil(6 V J / 4); uniform slot (v J + j) 6 + m is U_m), so the result depends only on (seed, global pose index):
 *   U0 < p_miss:              a miss, conf = 0 and the pixel is kept;
 *   U0 < p_miss + p_outlier:  a confident false detection, u = U3 (w - 1), v = U4 (h - 1), conf = 0.3 + 0.7 U5;
 *   otherwise:                Gaussian noise of std sigma_px / conf: (u, v) += sigma_px / conf * r (cos t, sin t),
 *                             r = sqrt(-2 ln max(U1, 1e-12)), t = 2 pi U2; conf unchanged.
 * fp64, rounded once to fp32; all parameters 0 leave pix bitwise unchanged.  sigma_px finite and >= 0, p_outlier and
 * p_miss in [0, 1] with a sum <= 1, 1 <= V <= 16, start >= 0.  batch == 0 returns MPL_OK without touching the pointers. */
int mpl_synth_detector_noise(uint64_t seed, int64_t start, int64_t batch, int num_views, int num_joints, const double* calib,
                             float sigma_px, float p_outlier, float p_miss, float* pix, mpl_stream_t stream);
/* mpl_synth_detector_noise with a calibration per pose (only its w, h are read; see Conventions). */
int mpl_synth_detector_noise_strided(uint64_t seed, int64_t start, int64_t batch, int num_views, int num_joints,
                                     const double* calib, int64_t calib_stride, float sigma_px, float p_outlier, float p_miss,
                                     float* pix, mpl_stream_t stream);

/* Lens distortion (ABI 8; defined by this library, the reference's cameras are pinholes).  OpenCV's 5-coefficient
 * Brown-Conrady model on normalised camera coordinates x = ((u - cx) / fx, (v - cy) / fy) of a pixel (u, v):
 *   r2 = x^2 + y^2,  rho = 1 + k1 r2 + k2 r2^2 + k3 r2^3,
 *   D(x) = (x rho + 2 p1 x y + p2 (r2 + 2 x^2),  y rho + p1 (r2 + 2 y^2) + 2 p2 x y).
 * dist holds (k1, k2, p1, p2, k3) per view (the order of CMU Panoptic's distCoef and of OpenCV's distCoeffs), fp64:
 * [V, 5] for the whole batch (dist_stride 0) or pose b at dist + b * dist_stride (>= 5 V; a packed [B, V, 5] tensor: 5 V).
 * dist_stride is independent of calib_stride (the calibration convention above), so per-pose cameras can share one lens.
 * Validity: an undistorted normalised point x is valid iff both
 *   (a) the radial map r -> r rho(r) is increasing on [0, |x|]: g(s) = 1 + 3 k1 s + 5 k2 s^2 + 7 k3 s^3 > 0 at s = r2 and at
 *       every root of g'(s) = 3 k1 + 10 k2 s + 21 k3 s^2 strictly inside (0, r2) (k3 != 0: the real roots
 *       (-10 k2 -/+ sqrt(100 k2^2 - 252 k1 k3)) / (42 k3); k3 == 0, k2 != 0: -3 k1 / (10 k2)), and
 *   (b) det J(x) > 0, J the 2 x 2 Jacobian of D.
 * Past a fold the polynomial maps points far outside the field of view back into the image; a real camera images none.
 * Shared rules of the two entry points below:
 *   - pix_in / pix_out [B, V, J, 3] fp32 (u, v, conf); pix_in == pix_out (in place) is allowed, no other overlap;
 *   - calib as in mpl_build_inputs (fx, fy, cx, cy and, for the undistortion, w and h are read); fp64 throughout, each
 *     output pixel rounded once to fp32; entries with conf == 0 are copied unchanged;
 *   - MPL_ERR_INVALID_ARGUMENT, before any CUDA call: batch < 0, V outside [1, 16], J < 1, a calib_stride or dist_stride
 *     that is not 0 or >= 18 V / 5 V, a margin that is not finite or is negative; then batch == 0 returns MPL_OK without
 *     touching the pointers (an empty tensor has no storage); then a null pointer is MPL_ERR_INVALID_ARGUMENT;
 *   - one thread per entry; allocates nothing and never synchronises (graph-capturable); results do not depend on how the
 *     batch is split.
 *
 * mpl_distort_pixels: ideal pinhole pixels (mpl_synth_project's, which are not clipped) -> the pixels a camera with this lens
 * records: u_d = u + fx (x_d - x), v_d = v + fy (y_d - y) with (x_d, y_d) = D(x) (= fx x_d + cx up to rounding).  An entry
 * whose x is not valid gets conf = 0 and keeps its pixel.  An entry whose five coefficients are all 0 is copied unchanged, so
 * with a zero lens the output is the input bit for bit (non-finite pixels and -0 included).
 * The synthetic step between mpl_synth_project and mpl_synth_detector_noise. */
int mpl_distort_pixels(const float* pix_in, float* pix_out, const double* calib, const double* dist, int64_t batch,
                       int num_views, int num_joints, mpl_stream_t stream);
int mpl_distort_pixels_strided(const float* pix_in, float* pix_out, const double* calib, int64_t calib_stride,
                               const double* dist, int64_t dist_stride, int64_t batch, int num_views, int num_joints,
                               mpl_stream_t stream);

/* mpl_undistort_pixels: detected (distorted) pixels -> the pinhole pixels of the same rays, for the triangulations, in a frame
 * grown by margin_x / margin_y pixels on each side: pass them the calibration with cx + margin_x, cy + margin_y,
 * w + 2 margin_x, h + 2 margin_y (DLT, reprojection errors and refinement are invariant under that shift), so undistorted
 * pixels beyond the original frame stay candidates.  Per entry with conf != 0:
 *   - the raw pixel not strictly inside the original frame (0 < u < w - 1 and 0 < v < h - 1, the candidate test of the
 *     triangulations): conf = 0, pixel kept.  So the candidate sets are those of the raw pixels;
 *   - otherwise Newton's method solves D(x) = x_d, x_d = ((u - cx) / fx, (v - cy) / fy), from x = x_d: at most 20 steps
 *     x -= J(x)^-1 (D(x) - x_d) (Cramer's rule), stopping after a step with |dx| + |dy| not > 1e-14 (NaN included).  The
 *     inversion succeeds iff the final x satisfies |D(x)_0 - x_d| + |D(x)_1 - y_d| <= 1e-12 and the validity rule; then
 *     u' = u + fx (x - x_d) + margin_x, v' = v + fy (y - y_d) + margin_y (= fx x + cx + margin_x up to rounding), conf kept;
 *     a failed inversion gives u' = v' = NaN, conf = 0.
 * With zero coefficients and zero margins u and v are copied bit for bit (so is conf, except where the raw pixel is outside
 * the frame, where no triangulation uses it). */
int mpl_undistort_pixels(const float* pix_in, float* pix_out, const double* calib, const double* dist, double margin_x,
                         double margin_y, int64_t batch, int num_views, int num_joints, mpl_stream_t stream);
int mpl_undistort_pixels_strided(const float* pix_in, float* pix_out, const double* calib, int64_t calib_stride,
                                 const double* dist, int64_t dist_stride, double margin_x, double margin_y, int64_t batch,
                                 int num_views, int num_joints, mpl_stream_t stream);

/* Calibration errors and rig calibration (ABI 9; defined by this library).  Rotation vectors: Exp(w) is Rodrigues' formula
 * I + sin t / t [w]x + (1 - cos t) / t^2 [w]x^2, t = |w|, and J_l(w) = I + (1 - cos t) / t^2 [w]x + (t - sin t) / t^3 [w]x^2
 * its left Jacobian; below t^2 = 1e-2 the three coefficients come from their Taylor series through t^8.
 *
 * mpl_synth_calib_noise: calib_out [B, V, 18] packed = the calibrations of poses [start, start + B), read from calib with the
 * calib_stride convention (0: one [V, 18] block; >= 18 V), perturbed.  Per (pose i, view v), U0..U5 come from the
 * Philox4x64-10 stream of mpl_synth_project under key (seed, 3), in the slot layout of mpl_synth_cameras (nb = ceil(6 V / 4),
 * slot 6 v + m is U_m), so the result depends only on (seed, global pose index).  Six standard normals by Box-Muller:
 * n_2k = r cos(2 pi U_2k+1), n_2k+1 = r sin(2 pi U_2k+1), r = sqrt(-2 ln max(U_2k, 1e-12)), k = 0, 1, 2.  Then
 *   R' = Exp(sigma_rot (n0, n1, n2)) R   (radians; a rotation in the camera frame, R maps world -> camera)
 *   t' = t + sigma_pos (n3, n4, n5)       (the camera centre, world units)
 * fx, fy, cx, cy, w, h are copied bit for bit; sigma_rot == 0 keeps R and sigma_pos == 0 keeps t bit for bit.  A fixed rig is
 * perturbed as pose 0: batch 1, start 0, stride 0.  fp64, one thread per (pose, view); allocates nothing and never
 * synchronises.  MPL_ERR_INVALID_ARGUMENT, before any CUDA call: V outside [1, 16], start < 0, a sigma that is not finite or
 * is negative, a bad calib_stride, batch < 0; then batch == 0 returns MPL_OK; then a null pointer, or calib_out == calib
 * with a stride other than 18 V, is MPL_ERR_INVALID_ARGUMENT. */
int mpl_synth_calib_noise(uint64_t seed, int64_t start, int64_t batch, int num_views, const double* calib,
                          int64_t calib_stride, double sigma_rot, double sigma_pos, double* calib_out, mpl_stream_t stream);

/* mpl_calibrate_rig: bundle adjustment of the extrinsics of one rig calib [V, 18] (no strided variant: a rig is calibrated
 * from many poses) from the detections pix [B, V, J, 3] of B poses, starting from the points init [B, J, 3] (e.g.
 * mpl_triangulate's under the same calib).  fp64 throughout.
 *   - used views of (b, j): the candidates of mpl_triangulate (conf > min_conf, strictly inside the image) whose bit is set
 *     in view_mask[b, j] when view_mask [B, J] int32 is not NULL (the rule of mpl_triangulate_refine);
 *   - items: the pairs (b, j) whose init is finite, with at least 2 used views, every one of which sees init at a finite
 *     depth > 0 under calib.  The set is fixed at the start;
 *   - parameters: per camera omega_v (R_v = Exp(omega_v) R0_v, omega_v = 0 at the start) and the centre c_v (c0_v at the
 *     start), R0 / c0 from calib; per item X_i (init at the start).  Intrinsics are fixed;
 *   - cost, y = R_v (X - c_v), pi(y) = (fx y0 / y2 + cx, fy y1 / y2 + cy):
 *       C = sum_items sum_used v (conf^2 / sigma_px^2) |pi(y) - (u, v)|^2 + sum_v (|omega_v|^2 / sigma_rot^2
 *           + |c_v - c0_v|^2 / sigma_pos^2),
 *     +inf if a used observation has y2 <= 0 or a non-finite y2.  The prior is the distribution mpl_synth_calib_noise draws
 *     from (so with the same sigmas this is the MAP rig) and it fixes the 7-DoF similarity gauge, hence every sigma > 0;
 *   - Jacobians, exact: dy/domega = -[y]x J_l(omega), dy/dc = -R, dy/dX = R;
 *   - LM: A = J^T W J and g = J^T W r over every residual, data and prior; the step solves (A + mu I) delta = -g, mu on every
 *     camera and point parameter; mu0 = 1e-3 max diag(A) at the start.  Schur solve: per item the Cholesky factor of
 *     M_i = A_ii + mu I, S = A_cc + mu I - sum_i A_ci M_i^-1 A_ic with the matching right-hand side, a dense Cholesky of S,
 *     delta X_i = -M_i^-1 (g_i + A_ic delta c).  A Cholesky pivot that is not finite and > 0, in any M_i or in S, rejects the
 *     step (mu *= 10) and skips the stop test.  If C(new) < C the step is accepted, mu /= 10; otherwise rejected, mu *= 10.
 *     Iteration k stops the solve if the 6 V camera step satisfies |delta_cam|_2 <= 1e-10 (|c|_2 + 1e-10), c the 3 V centres
 *     before the iteration, or when k = max_iters;
 *   - outputs: calib_out [V, 18] = Exp(omega_v) R0_v and c_v with the other six fields copied bit for bit (R0 bit for bit
 *     while omega_v is exactly 0); points [B, J, 3] fp32 (may be NULL, may alias init) = the refined X for items, init bit for
 *     bit otherwise; report [8] fp64 on the device = items, observations, C at the start, C at the end, the conf-weighted
 *     RMS pixel error sqrt(sum conf^2 e^2 / sum conf^2) at the start and at the end, iterations run, accepted steps.  With
 *     no item calib_out is calib bit for bit, points is init and the report is all 0;
 *   - MPL_ERR_INVALID_ARGUMENT, before any CUDA call: V outside [2, 16], J < 1, batch < 1, a sigma that is not finite or
 *     <= 0, max_iters outside [1, 100], a null pix / calib / init / calib_out / report / workspace.  A workspace shorter
 *     than mpl_calibrate_rig_workspace_bytes(batch, V, J) is MPL_ERR_WORKSPACE (the query returns 0 for a shape the call
 *     rejects);
 *   - allocates nothing and never synchronises: the LM control lives in the workspace, a fixed sequence of 4 max_iters + 3
 *     launches is enqueued and the iterations after the stop return at once (graph-capturable).  Bitwise deterministic: no
 *     floating-point atomics, partial sums reduced in a fixed order, their number a function of (batch, V, J) only. */
size_t mpl_calibrate_rig_workspace_bytes(int64_t batch, int num_views, int num_joints);
int mpl_calibrate_rig(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints, float min_conf,
                      const int32_t* view_mask, const float* init, double sigma_px, double sigma_rot, double sigma_pos,
                      int max_iters, double* calib_out, float* points, double* report, void* workspace,
                      size_t workspace_bytes, mpl_stream_t stream);

/* Multi-person association across views (ABI 11; defined by this library: the reference's datasets give which detection of
 * each view belongs to which person).  Every other entry point takes pix [B, V, J, 3] with row b of every view one person;
 * the calls below get that grouping from the detections.
 *
 * Scene layout: a frame holds P detection slots per view.  scene [F, P, V, J, 3] fp32 (u, v, conf): entry (f, s, v) is slot s
 * of view v; slots of different views are unrelated.  Detection (s, v) has the flat index m = s V + v.  Viewed as
 * [F P, V, J, 3] a scene has the [B, V, J, 3] shape, so the lens and input-builder entry points apply to it unchanged.
 *
 * mpl_synth_people: scenes out of person-ordered pixels.  pix [F P, V, J, 3] holds person p of frame f in row f P + p (e.g.
 * mpl_synth_project of poses [start P, (start + F) P) with lens and detector noise); perm [F, V, P] int32 gets, for frame f
 * and view v, the person in each slot, and scene[f, s, v] = pix[f P + perm[f, v, s], v], copied bit for bit.  The draw:
 * global frame i = start + f owns the counter blocks [i nb, (i + 1) nb), nb = ceil(V P / 4), of the Philox4x64-10 stream of
 * mpl_synth_project under key (seed, 4); slot v P + s of those is U_s of view v, and perm[f, v] is the stable ascending
 * argsort of U_0 .. U_{P-1} (openmpl_b200/synth.py synth_people is the twin).  MPL_ERR_INVALID_ARGUMENT, before any CUDA
 * call: frames < 0, start < 0, V outside [1, 16], P < 1, P V > 128, J < 1; then frames == 0 returns MPL_OK; then a null
 * pointer or scene == pix is MPL_ERR_INVALID_ARGUMENT.
 *
 * mpl_associate_people(_strided): groups the detections of each frame into people, fp64 throughout.  Frame f reads the
 * calibration calib + f calib_stride (the calib_stride convention with frames in place of poses).
 *   - candidate joint: conf > min_conf and strictly inside the w x h image (the rule of mpl_triangulate);
 *   - active detection: at least min_joints candidate joints;
 *   - ray of a candidate joint of view v: origin c_v (calib t), direction d = R^T ((u - cx) / fx, (v - cy) / fy, 1).  The
 *     model is a pinhole: undistort first (mpl_undistort_pixels), as for the triangulations;
 *   - joint distance of two rays: the distance of the two lines, |(c2 - c1) . n| / |n| with n = d1 x d2; where
 *     |n|^2 <= 1e-24 |d1|^2 |d2|^2, |(c2 - c1) x d1| / |d1|;
 *   - pair cost of active (s, v) and (t, w), v < w (member 1 in the lower view): the median of the joint distances over the
 *     joints that are candidates in both (the mean of the two middle values for an even count); +inf when fewer than
 *     min_joints joints are shared.  The median keeps a few confident false detections from hiding a true pair;
 *   - greedy complete linkage: every active detection starts as its own cluster.  The pairs with cost <= max_dist, sorted by
 *     (cost, key) ascending with key = m1 P V + m2 (m1 the member in the lower view), are taken in order; each merges its
 *     two clusters unless they are already one, they share a view, or some cross pair of their members has a cost that is
 *     not <= max_dist;
 *   - people: the clusters with >= 2 members, ranked by member count descending, then smallest member m ascending;
 *   - outputs: members [F, K, V] int32, the slot of view v in the person of rank k, or -1 (rows past the last person all
 *     -1); labels [F, P, V] int32, the rank of the detection's person if that rank is < K, -1 for an active detection in no
 *     output person, -2 for an inactive one; people [F] int32, the number of people (may exceed K);
 *   - MPL_ERR_INVALID_ARGUMENT, before any CUDA call: frames < 0, V outside [2, 16], P < 1, P V > 128 (at most 8128 pairs
 *     per frame), J outside [1, 32], min_joints outside [1, J], max_dist not finite or not > 0, K < 1, a bad calib_stride;
 *     then frames == 0 returns MPL_OK; then a null pointer is MPL_ERR_INVALID_ARGUMENT;
 *   - one CTA per frame; no floating-point atomics; results independent of how the frames are split; allocates nothing and
 *     never synchronises (graph-capturable).
 *
 * mpl_gather_people: out [F, K, V, J, 3] fp32, out[f, k, v] = scene[f, members[f, k, v], v] bit for bit, zeros (u = v =
 * conf = 0) where the member is -1 (or any value outside [0, P)).  Viewed as [F K, V, J, 3] it is a batch of people for the
 * input builder, the forward, the triangulations and the refinement; with a lens, gather from the raw scene for the lifter
 * and from the undistorted scene for the triangulations.  MPL_ERR_INVALID_ARGUMENT, before any CUDA call: frames < 0, P < 1,
 * K < 1, V outside [1, 16], J < 1; then frames == 0 returns MPL_OK; then a null pointer.
 *
 * mpl_association_score: scores members / labels (of mpl_associate_people) against the true slots perm (of
 * mpl_synth_people).  The true person of detection (s, v) is perm[f, v, s]; a detection is active iff its label is not -2.
 *   owner [F, K] int32: the true person with the most members in row k, ties to the smaller person index; -1 for an empty row;
 *   acc [MPL_ASSOC_ACC_LEN] fp64 running sums (added to, so ranks combine with one all-reduce):
 *     [0] frames; [1] associable people (true persons with >= 2 active detections); [2] non-empty rows; [3] pure rows (every
 *     member belongs to one person); [4] complete rows (pure, and holding every active detection of that person);
 *     [5] predicted linked pairs (member pairs within rows); [6] correct linked pairs (of the same person); [7] true pairs
 *     (pairs of active detections of one person, in different views).
 *   Integer counts reduced in a fixed order, added once per call.  MPL_ERR_INVALID_ARGUMENT, before any CUDA call: frames < 0,
 *   V outside [1, 16], P < 1, P V > 128, K < 1; then frames == 0 returns MPL_OK (acc untouched); then a null pointer. */
#define MPL_ASSOC_ACC_LEN 8
int mpl_synth_people(uint64_t seed, int64_t start, int64_t frames, int people, int num_views, int num_joints, const float* pix,
                     float* scene, int32_t* perm, mpl_stream_t stream);
int mpl_associate_people(const float* scene, const double* calib, int64_t frames, int people, int num_views, int num_joints,
                         float min_conf, int min_joints, double max_dist, int max_people, int32_t* members, int32_t* labels,
                         int32_t* num_people, mpl_stream_t stream);
int mpl_associate_people_strided(const float* scene, const double* calib, int64_t calib_stride, int64_t frames, int people,
                                 int num_views, int num_joints, float min_conf, int min_joints, double max_dist,
                                 int max_people, int32_t* members, int32_t* labels, int32_t* num_people,
                                 mpl_stream_t stream);
int mpl_gather_people(const float* scene, const int32_t* members, int64_t frames, int people, int max_people, int num_views,
                      int num_joints, float* out, mpl_stream_t stream);
int mpl_association_score(const int32_t* members, const int32_t* labels, const int32_t* perm, int64_t frames, int people,
                          int max_people, int num_views, int32_t* owner, double* acc, mpl_stream_t stream);

/* Multi-person tracking across frames (additions to ABI 11: new entry points only, so a caller built against ABI 11 is
 * unaffected; defined by this library).  A sequence is T consecutive frames of one scene; the calls below give each person
 * row of a frame a track id that persists from frame to frame.
 *
 * mpl_synth_motion: S sequences of T frames of P people that move, for sequences [start, start + S).  Row
 * r = ((start + s) T + t) P + p (local row b = (s T + t) P + p) holds person p in frame t of global sequence i = start + s:
 * target [S T P, J, 3] fp32 (metres) and pix [S T P, V, J, 3] fp32 (u, v, conf), the formats of mpl_synth_project.  Viewed as
 * [F P, ...] with F = S T frames the rows feed mpl_distort_pixels, mpl_synth_detector_noise (start index r) and
 * mpl_synth_people (frame index (start + s) T + t) unchanged.  The motion of (i, p) is drawn from the Philox4x64-10 stream of
 * mpl_synth_project under key (seed, 5): g = i P + p owns the counter blocks [g nb, (g + 1) nb), nb = ceil((9 + 6 (J - 1)) /
 * 4), with uniform slots U0 .. U8 and the body pairs (u1_m, u2_m) in slots 9 + m and 9 + 3 (J - 1) + m, m = 3 (j - 1) + k.
 * With tau = t / fps seconds, room (x0, x1, y0, y1), w_x = x1 - x0 and w_y = y1 - y0:
 *   - root x = (x0 + x1) / 2 + a_x sin(2 pi f_x tau + 2 pi U4), a_x = (0.25 + 0.25 U0) w_x, f_x = 0.03 + 0.07 U2 Hz; y likewise
 *     with U1, U3, U5 and w_y (so the root stays in the room and moves at most 2 pi 0.1 0.5 |(w_x, w_y)| m/s);
 *     z = 0.8 + 0.2 U6, constant;
 *   - heading theta = 2 pi U7 + (U8 - 0.5) tau rad (at most 0.5 rad/s);
 *   - body o_0 = 0, o_j[k] = 0.25 sqrt(-2 ln max(u1_m, 1e-12)) cos(2 pi u2_m) (mpl_synth_project's Box-Muller), fixed in time;
 *   - joints X_j = root + Rz(theta) o_j, fp64, so the motion of (i, p, t) depends only on (seed, i, p, t, J, fps, room);
 *   - pixels: mpl_synth_project's camera model (x_cam = R (X - t), u = f x_cam / z + c, no clipping, conf 0 behind the
 *     camera) through calib + b calib_stride (the calib_stride convention with rows in place of poses), and conf = 1 with
 *     conf_ones, otherwise 0.3 + 0.7 U from mpl_synth_project's confidence slots of pose index r (key (seed, 0)): a row's
 *     confidences are those mpl_synth_project gives pose r.
 * openmpl_b200/synth.py synth_motion is the numpy twin.  MPL_ERR_INVALID_ARGUMENT, before any CUDA call: sequences < 0,
 * start < 0, frames < 1, people < 1, V outside [1, 16], J < 1, fps not finite or not > 0, a bad calib_stride; then
 * sequences == 0 returns MPL_OK; then a null pointer.
 *
 * mpl_track_people: online tracking of person rows, sequence by sequence; the state carries the tracks across calls.
 *   points [S, T, K, J, 3] fp32: per frame, K rows of 3D joints (e.g. mpl_triangulate_robust of mpl_gather_people rows, or
 *     the lifter's output); NaN joints are allowed.  joint_mask NULL or [S, T, K, J] fp32.
 *   state: per sequence mpl_track_state_bytes(max_tracks, J) bytes, opaque, 4-byte aligned, sequence s at s times that size;
 *     all-zero bytes are a fresh sequence.  mpl_track_state_bytes returns 0 for a shape the call rejects (max_tracks
 *     outside [1, 128], J outside [1, 32]).
 *   track_id [S, T, K] int32 output.  The rules, frame by frame in order:
 *   - used joint: its three coordinates are finite and joint_mask is NULL or > 0; a row with >= min_joints used joints is a
 *     detection;
 *   - a track remembers, per joint, the last observed position (fp32, bit for bit) and whether it has one, its id and its
 *     count of consecutive missed frames.  No prediction (zero velocity);
 *   - cost of (track, row), fp64: the median over the joints used in the row and remembered by the track of the joint
 *     distance sqrt((dx dx + dy dy) + dz dz), each product and sum rounded (no fused multiply-add); the mean of the two
 *     middle values for an even count; +inf with fewer than min_joints such joints;
 *   - matching: the pairs with cost <= max_dist, sorted by (cost, key) ascending with key = id K + k, are taken in order; a
 *     pair matches unless its track or its row is already matched.  A matched track overwrites the joints the row uses,
 *     keeps the others and resets its misses to 0;
 *   - ageing: every unmatched live track increments its misses and is freed when they exceed max_age;
 *   - births: every unmatched detection, in row order, starts a track with the sequence's next id (0, 1, 2, ...) while
 *     fewer than max_tracks tracks are live; otherwise its id is -1;
 *   - track_id: the id the row was matched to or born as; -1 for a row that is not a detection or found no free track.
 *   Sequences are independent; frames [0, T1) then [T1, T) on the same state give bitwise the ids of one call on [0, T).
 *   MPL_ERR_INVALID_ARGUMENT, before any CUDA call: sequences < 0, frames < 0 or > INT32_MAX, K outside [1, 64], J outside
 *   [1, 32], min_joints outside [1, J], max_dist not finite or not > 0, max_age < 0, max_tracks outside [1, 128]; then
 *   sequences == 0 or frames == 0 returns MPL_OK; then a null points / state / track_id or a misaligned state.  One CTA per
 *   sequence with its state in shared memory; no floating-point atomics; allocates nothing and never synchronises
 *   (graph-capturable).
 *
 * mpl_tracking_score: CLEAR-MOT style counts of track_id [S, T, K] (of mpl_track_people from a zeroed state, whole
 * sequences) against the rows' true persons owner [S, T, K] (e.g. mpl_association_score's owner; -1 for none) of P persons,
 * each present in every frame (T P objects per sequence).  The match of person q in frame t is the smallest row k with
 * owner == q and track_id >= 0, its id the hypothesis.  acc [MPL_TRACK_ACC_LEN] fp64 running sums (added to):
 *   [0] sequences; [1] frames; [2] objects; [3] matches; [4] misses (objects - matches); [5] false positives (rows with
 *   track_id >= 0 that are no match); [6] ID switches (a match whose hypothesis differs from q's previous match in the
 *   sequence); [7] fragmentations (a match after a frame without one, following an earlier match); [8] mostly tracked
 *   (persons matched in >= 80 % of the frames); [9] mostly lost (< 20 %); [10] tracks (1 + the largest id per sequence).
 *   Integer counts reduced in a fixed order, added once per call.  MPL_ERR_INVALID_ARGUMENT, before any CUDA call:
 *   sequences < 0, frames < 0 or > INT32_MAX, K < 1, P < 1; then sequences == 0 or frames == 0 returns MPL_OK (acc untouched);
 *   then a null pointer. */
#define MPL_TRACK_ACC_LEN 11
int mpl_synth_motion(uint64_t seed, int64_t start, int64_t sequences, int frames, int people, int num_views, int num_joints,
                     const double* calib, int64_t calib_stride, const double* room, double fps, int conf_ones, float* pix,
                     float* target, mpl_stream_t stream);
size_t mpl_track_state_bytes(int max_tracks, int num_joints);
int mpl_track_people(const float* points, const float* joint_mask, int64_t sequences, int64_t frames, int max_rows,
                     int num_joints, int min_joints, double max_dist, int max_age, int max_tracks, void* state,
                     int32_t* track_id, mpl_stream_t stream);
int mpl_tracking_score(const int32_t* track_id, const int32_t* owner, int64_t sequences, int64_t frames, int max_rows,
                       int people, double* acc, mpl_stream_t stream);

/* ---- unit-test hooks for the building blocks (used by tests/ only) ------------------------------------------- */
/* Y[M,N] = epilogue(A[M,K] . W[N,K]^T): the tcgen05 projection kernel in isolation.
 *   dtype: MPL_PREC_BF16 (A, W bf16) or MPL_PREC_TF32 (split mode: A = [2][M][K], W = [2][N][K] bf16 planes hi, lo)
 *   epilogue: 0 bias -> operand format (bf16, or two planes [2][M][N]) / fp32 per `out_fp32`; 1 bias+GELU;
 *             2 bias + residual(fp32, in place in Y) */
int mpl_test_gemm(const void* A, const void* W, const float* bias, void* Y, int64_t M, int N, int K, int dtype,
                  int epilogue, int out_fp32, mpl_stream_t stream);

/* The LayerNorm-fused epilogues of the bf16 mode in isolation (DESIGN.md section 4).
 *   epilogue 4 / 5 (LayerNorm-apply, QKV / fc1): Y[M,N] (bf16, or fp16 when out_fp16) = act(rstd * (A W'^T - mu * colsum) + bias),
 *       A = raw residual rows rounded to bf16, W' = bf16(W diag(gamma)), colsum[n] = sum_k W'[n,k], bias = b + W beta,
 *       (mu, rstd) from stats_in = [slots_in][M rounded up to 256] float2 partial (sum x, sum x^2) per row, eps = LayerNorm eps;
 *   epilogue 6 (residual-emit, proj / fc2): the residual stream x [M,N] as two bf16 planes (Y = hi, x_lo = lo), updated in place:
 *       x += A W^T + bias; stats_out = [mpl_test_gemm_ln_slots(N)][M rounded up to 256] float2 partial (sum, sum^2) of the new x;
 *       ab_fp16: A and W hold fp16 instead of bf16. */
int mpl_test_gemm_ln(const void* A, const void* W, const float* bias, void* Y, int64_t M, int N, int K, int epilogue,
                     const float* colsum, const void* stats_in, int slots_in, void* stats_out, void* x_lo, float eps,
                     int ab_fp16, int out_fp16, mpl_stream_t stream);
int mpl_test_gemm_ln_slots(int N);
/* Epilogue 6 on the first N columns of residual planes whose rows are `ldy` >= N elements apart (the last fc2 of the stack
 * updates the pose half of the channel-permuted residual stream only, DESIGN.md section 3); the other columns stay. */
int mpl_test_gemm_emit_pitch(const void* A, const void* W, const float* bias, void* Y, int64_t M, int N, int K, void* stats_out,
                             void* x_lo, int ab_fp16, int ldy, mpl_stream_t stream);
/* The fused QKV projection + cross-view attention kernel (multiview_mpl.py:48-64 behind the folded norm1) in isolation:
 *   xb [M, D] bf16 raw residual rows, W [3D, D] / bias [3D] (or NULL) / gamma, beta [D] fp32 on the device, stats as above,
 *   att [M, D] bf16 out; M = poses * V rows, D = H * 136 (or H * 68, H even), 2 <= V <= 8.
 *   scratch: device buffer of at least align256(H*416*D*2) + 2 * align256(H*416*4) bytes for the packed operands. */
int mpl_test_qkv_attn(const void* xb, const float* W, const float* bias, const float* gamma, const float* beta,
                      const void* stats, int slots, float eps, float scale, void* att, int64_t M, int D, int H, int V,
                      void* scratch, size_t scratch_bytes, mpl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MPL_B200_H_ */
