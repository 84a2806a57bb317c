// Host side of libmpl_b200: the constructor contract (parameter table, derived dims, validity), weight packing,
// workspace layout and the forward orchestration (multiview_mpl.py:95-317, 349-525), plus the extern "C" boundary.
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "kernels.cuh"

namespace mpl {

static thread_local std::string g_last_error;

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
}

struct ParamInfo {
  std::string name;
  int64_t numel;
  bool is_int64;
  size_t offset;  // byte offset of the fp32 copy inside the packed blob
};

struct Derived {  // extra packed tensors computed from the parameters
  std::string name;
  int64_t numel;
  int esz;
  size_t offset;
};

struct BnFold {
  std::string lin, bn;
  int N, K;
};

struct BlockW {
  const float *n1w, *n1b, *qkvw, *qkvb, *projw, *projb, *n2w, *n2b, *fc1w, *fc1b, *fc2w, *fc2b;
  const void *qkvw_tc, *projw_tc, *fc1w_tc, *fc2w_tc;  // tensor-core operand copies (FPT, bf16 / tf32 modes)
  const float *qkv_cs, *qkv_bf, *fc1_cs, *fc1_bf;      // LayerNorm-fused mode: column sums of W' and folded biases
  const void* qa_w;                                    // fused QKV + attention: head-tiled W'' and its column sums / biases
  const float *qa_cs, *qa_b;
};

}  // namespace mpl

using namespace mpl;

struct MplModel {
  MplDesc d;
  // derived dims (spec.make_config)
  int J, V, dim, H, depth, in_ch, tok_w, fpt_dim, fpt_tokens, E, pos3d_lin_out, pos3d_w, spt_hidden, fpt_hidden;
  bool add_conf, mult_conf, conf_emb, multi;
  int ray_layout;  // 0 none, 1 interleave, 2 append
  int n_out;
  bool fpt_tc;     // FPT projections run on tcgen05 (precision != fp32 and shapes fit)
  bool spt_fused;  // the SPT stack runs as the single fused fp16-mma kernel (bf16 / tf32 modes, d=32, H=8, J=17)
  bool ln_fused;   // bf16 mode: the FPT LayerNorms are folded into the projection GEMMs (no LayerNorm kernel)
  // LN-fused planes behind the single-kernel SPT with interleaved ray tokens ([x_j | ray_j] per joint, ray_layout 1) and the K5
  // head: the residual stream is kept CHANNEL-PERMUTED as [all pose parts | all ray parts].  Every consumer is permutation
  // equivariant once its weights are permuted at pack time (LayerNorm gamma / beta and W columns of QKV / fc1, W rows and
  // biases of proj / fc2), so nothing changes at run time except that (1) the head reads one contiguous half row instead of
  // the pose half of every 128-byte line and (2) the LAST fc2 of the stack computes the pose half only: the head never
  // reads the ray channels of the final residual (multiview_mpl.py:425-433 strips them).
  bool perm;
  std::vector<int> perm_host;  // packed channel c holds reference channel perm_host[c]
  bool qkv_attn;      // bf16 LN-fused mode, view tokens, D = H * 136 (or H * 68), 2 <= V <= 8: QKV GEMM + cross-view attention are one kernel
  bool fpt_kp_fused;  // bf16 mode, keypoint-token FPT (width 32, 8 heads, J = 17): the whole FPT stack is one kernel launch
  int ln_slots;    // statistics slots per row written by the residual-emit GEMMs
  std::vector<ParamInfo> params;
  std::unordered_map<std::string, int> index;
  std::vector<Derived> derived;
  std::unordered_map<std::string, int> dindex;
  std::vector<BnFold> folds;
  size_t packed_bytes = 0;
  int64_t chunk = 32768;
  int64_t launches = 0;
  // small-batch path: the whole forward of a (batch, pointer set) captured once as a CUDA graph and replayed with one launch
  struct GraphKey {
    int64_t batch, pose_stride, center_stride;
    const void* packed;
    const void* in[3][kMaxViews];
    void *out, *aux1, *aux2, *workspace;
  };
  struct GraphEntry {
    GraphKey key;
    cudaGraphExec_t exec;
    int64_t launches;
    uint64_t last_used;
  };
  std::vector<GraphEntry> graphs;
  int64_t graph_max_batch = 0;   // 0: off (mpl_set_graph_batch)
  cudaStream_t cap_stream = nullptr;
  uint64_t graph_clock = 0;
  int64_t graph_hits = 0, graph_captures = 0;
  // weight pointers of every block, resolved once per packed blob (no string lookups on the launch path)
  const void* resolved_for = nullptr;
  std::vector<mpl::BlockW> fpt_blocks;
  // optional per-launch CUDA-event profiling (bench.py's roofline numbers come from here)
  bool profile = false;
  struct ProfRec { int cat; cudaEvent_t e0, e1; };
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
};

namespace mpl {

static void add_param(MplModel* m, const std::string& name, int64_t numel, bool is_int64 = false) {
  m->index[name] = (int)m->params.size();
  m->params.push_back({name, numel, is_int64, 0});
}
static void add_linear(MplModel* m, const std::string& p, int out_f, int in_f) {
  add_param(m, p + "weight", (int64_t)out_f * in_f);
  add_param(m, p + "bias", out_f);
}
static void add_bn(MplModel* m, const std::string& p, int n) {
  add_param(m, p + "weight", n);
  add_param(m, p + "bias", n);
  add_param(m, p + "running_mean", n);
  add_param(m, p + "running_var", n);
  add_param(m, p + "num_batches_tracked", 1, true);
}
static void add_block(MplModel* m, const std::string& p, int dim, int hidden, bool qkv_bias) {
  add_param(m, p + "norm1.weight", dim);
  add_param(m, p + "norm1.bias", dim);
  add_param(m, p + "attn.qkv.weight", (int64_t)3 * dim * dim);
  if (qkv_bias) add_param(m, p + "attn.qkv.bias", 3 * dim);
  add_linear(m, p + "attn.proj.", dim, dim);
  add_param(m, p + "norm2.weight", dim);
  add_param(m, p + "norm2.bias", dim);
  add_linear(m, p + "mlp.fc1.", hidden, dim);
  add_linear(m, p + "mlp.fc2.", dim, hidden);
}
static void add_derived(MplModel* m, const std::string& name, int64_t numel, int esz) {
  m->dindex[name] = (int)m->derived.size();
  m->derived.push_back({name, numel, esz, 0});
}

// Flag combinations whose first forward raises in the reference (SURVEY.md §3.2-Q6); same order as spec._first_forward_error.
static int validate(const MplModel* m) {
  const MplDesc& d = m->d;
  if (d.num_joints < 1 || d.embed_dim_ratio < 1 || d.num_heads < 1 || d.num_views < 1 || d.depth < 0) {
    set_error("num_joints, embed_dim_ratio, num_heads, num_views must be positive and depth non-negative");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (d.num_views > kMaxViews) {
    set_error("num_views = %d exceeds the supported maximum of %d", d.num_views, kMaxViews);
    return MPL_ERR_UNSUPPORTED;
  }
  if (d.in_chans != 2) {
    set_error("in_chans must be 2: the forward slices pose[:, :, 0:2|0:3] (multiview_mpl.py:359-364)");
    return MPL_ERR_CONFIG_RUNTIME;
  }
  if (m->dim % m->H != 0 && !d.no_transformer_spt && d.depth > 0) {
    set_error("embed_dim_ratio must be divisible by num_heads (reshape at multiview_mpl.py:55)");
    return MPL_ERR_CONFIG_RUNTIME;
  }
  if (d.no_transformer_spt && d.multiple_spatial_blocks) {
    set_error("index 0 is out of range (Spatial_blocks is empty, multiview_mpl.py:401)");
    return MPL_ERR_CONFIG_INDEX;
  }
  if (d.add_3D_pos_encoding_to_rays && !d.input_rays_as_token) {
    set_error("The size of tensor a (%d) must match the size of tensor b (%d) at non-singleton dimension 2 "
              "(multiview_mpl.py:483)", m->dim, 2 * m->dim);
    return MPL_ERR_CONFIG_RUNTIME;
  }
  if (d.input_rays_as_token && d.add_3D_pos_encoding_to_rays && d.add_3D_pos_encoding_in_Spatial && d.pose_3d_emb_learnable) {
    set_error("The size of tensor a (%d) must match the size of tensor b (%d) at non-singleton dimension 2 "
              "(multiview_mpl.py:396)", m->dim, 2 * m->dim);
    return MPL_ERR_CONFIG_RUNTIME;
  }
  if (d.input_rays_as_token && d.FPT_blocks_view_keypoint_tokens && !d.no_transformer_fpt) {
    set_error("Given normalized_shape=[%d], expected input with shape [*, %d], but got input of width %d "
              "(multiview_mpl.py:75,497)", m->dim, m->dim, 2 * m->dim);
    return MPL_ERR_CONFIG_RUNTIME;
  }
  if (!d.no_transformer_fpt && m->fpt_dim % m->H != 0 && d.depth > 0) {
    set_error("FPT width must be divisible by num_heads (reshape at multiview_mpl.py:55)");
    return MPL_ERR_CONFIG_RUNTIME;
  }
  return MPL_OK;
}

static void build_tables(MplModel* m) {
  const MplDesc& d = m->d;
  const int J = m->J, V = m->V, dim = m->dim, E = m->E;
  std::vector<std::string> views;
  if (m->multi) for (int v = 0; v < V; ++v) views.push_back(std::to_string(v) + ".");
  else views.push_back("");
  if (!m->multi) add_param(m, "Spatial_pos_embed", (int64_t)J * dim);
  add_param(m, "pos_3d_embed", (int64_t)J * m->pos3d_w);
  add_param(m, "pos_3d_view_coding", (int64_t)J * m->pos3d_w);
  for (auto& v : views) add_linear(m, "Spatial_patch_to_embedding." + v, dim, m->in_ch);
  if (m->conf_emb) for (auto& v : views) add_linear(m, "confidence_to_embedding." + v, dim, 1);
  if (m->multi) for (int v = 0; v < V; ++v) add_param(m, "Spatial_pos_embed." + std::to_string(v), (int64_t)J * dim);
  add_linear(m, "pos_3d_linear.", m->pos3d_lin_out, 3);
  if (d.input_rays_as_token) add_linear(m, "ray_to_embedding.", dim, 3);
  if (d.confidence_in_FPT) add_linear(m, "confidence_to_embedding_FPT.", dim, 1);
  if (!d.no_transformer_spt)
    for (auto& v : views)
      for (int l = 0; l < m->depth; ++l) add_block(m, "Spatial_blocks." + v + std::to_string(l) + ".", dim, m->spt_hidden, d.qkv_bias);
  if (!d.no_transformer_fpt)
    for (int l = 0; l < m->depth; ++l) add_block(m, "blocks." + std::to_string(l) + ".", m->fpt_dim, m->fpt_hidden, d.qkv_bias);
  add_param(m, "Spatial_norm.weight", dim);
  add_param(m, "Spatial_norm.bias", dim);
  add_param(m, "View_norm.weight", E);
  add_param(m, "View_norm.bias", E);
  if (d.linear_weighted_mean) add_linear(m, "weighted_mean.", E, V * E);
  else { add_param(m, "weighted_mean.weight", V); add_param(m, "weighted_mean.bias", 1); }
  const int out_dim = 3 * J, Hd = d.hidden_dim;
  if (d.head_kadkhod) {
    for (int s = 0; s < 3; ++s) {
      const int first_in = (s == 0) ? E : out_dim + E;
      const std::string p = "head." + std::to_string(s) + ".";
      if (s == 0) {
        add_param(m, p + "0.0.weight", E);
        add_param(m, p + "0.0.bias", E);
        add_linear(m, p + "0.1.", Hd, first_in);
        add_bn(m, p + "0.2.", Hd);
        m->folds.push_back({p + "0.1.", p + "0.2.", Hd, first_in});
      } else {
        add_linear(m, p + "0.0.", Hd, first_in);
        add_bn(m, p + "0.1.", Hd);
        m->folds.push_back({p + "0.0.", p + "0.1.", Hd, first_in});
      }
      for (int k = 1; k <= 2; ++k) {
        add_linear(m, p + std::to_string(k) + ".0.", Hd, Hd);
        add_bn(m, p + std::to_string(k) + ".1.", Hd);
        m->folds.push_back({p + std::to_string(k) + ".0.", p + std::to_string(k) + ".1.", Hd, Hd});
      }
      add_linear(m, p + "3.", out_dim, Hd);
    }
  } else if (d.deep_head) {
    add_param(m, "head.0.weight", E);
    add_param(m, "head.0.bias", E);
    add_linear(m, "head.1.", Hd, E);
    add_bn(m, "head.2.", Hd);
    add_linear(m, "head.4.", Hd, Hd);
    add_bn(m, "head.5.", Hd);
    add_linear(m, "head.7.", Hd, Hd);
    add_bn(m, "head.8.", Hd);
    add_linear(m, "head.10.", out_dim, Hd);
    m->folds.push_back({"head.1.", "head.2.", Hd, E});
    m->folds.push_back({"head.4.", "head.5.", Hd, Hd});
    m->folds.push_back({"head.7.", "head.8.", Hd, Hd});
  } else {
    add_param(m, "head.0.weight", E);
    add_param(m, "head.0.bias", E);
    add_linear(m, "head.1.", out_dim, E);
  }
  // derived tensors
  for (auto& f : m->folds) {
    add_derived(m, "fold:" + f.lin + "weight", (int64_t)f.N * f.K, 4);
    add_derived(m, "fold:" + f.lin + "bias", f.N, 4);
  }
  const int maxdim = std::max(m->dim, m->fpt_dim);
  add_derived(m, "zeros", 3 * (int64_t)maxdim, 4);
  if (!d.linear_weighted_mean && !d.deep_head && !d.head_kadkhod && out_dim <= 64) add_derived(m, "headT", (int64_t)E * 64, 4);
  if (m->spt_fused) {
    const int stacks = m->multi ? V : 1;
    for (int st = 0; st < stacks; ++st) add_derived(m, "sptpack:" + std::to_string(st), (int64_t)m->depth * spt_fused_layer_bytes(), 1);
  }
  if (m->fpt_kp_fused) add_derived(m, "fptpack", (int64_t)m->depth * spt_fused_layer_bytes(), 1);
  if (m->perm) add_derived(m, "perm", m->fpt_dim, 4);
  if (m->fpt_tc) {
    // bf16 mode: one bf16 (fp16 for fc2 under LayerNorm fusion) copy; split mode: two bf16 planes (hi, lo) per matrix
    const int esz = (d.precision == MPL_PREC_BF16) ? 2 : 4;
    const char* tag = (d.precision == MPL_PREC_BF16) ? "bf16:" : "split:";
    for (int l = 0; l < m->depth; ++l) {
      const std::string p = "blocks." + std::to_string(l) + ".";
      const int64_t D = m->fpt_dim, Hf = m->fpt_hidden;
      if (m->ln_fused) {
        if (m->qkv_attn) {
          add_derived(m, "qaw:" + p + "attn.qkv", (int64_t)qkv_attn_weight_elems((int)D, m->H), 2);
          add_derived(m, "qacs:" + p + "attn.qkv", qkv_attn_vec_len((int)D, m->H), 4);
          add_derived(m, "qab:" + p + "attn.qkv", qkv_attn_vec_len((int)D, m->H), 4);
        } else {
          add_derived(m, "lnw:" + p + "attn.qkv", 3 * D * D, 2);
          add_derived(m, "lncs:" + p + "attn.qkv", 3 * D, 4);
          add_derived(m, "lnb:" + p + "attn.qkv", 3 * D, 4);
        }
        add_derived(m, "lnw:" + p + "mlp.fc1", Hf * D, 2);
        add_derived(m, "lncs:" + p + "mlp.fc1", Hf, 4);
        add_derived(m, "lnb:" + p + "mlp.fc1", Hf, 4);
        if (m->perm) {  // biases of the two residual-emit GEMMs in the permuted channel order
          add_derived(m, "pb:" + p + "attn.proj.bias", D, 4);
          add_derived(m, "pb:" + p + "mlp.fc2.bias", D, 4);
        }
      } else {
        add_derived(m, tag + p + "attn.qkv.weight", 3 * D * D, esz);
        add_derived(m, tag + p + "mlp.fc1.weight", Hf * D, esz);
      }
      add_derived(m, tag + p + "attn.proj.weight", D * D, esz);
      add_derived(m, tag + p + "mlp.fc2.weight", D * Hf, esz);
    }
  }
  size_t off = 0;
  for (auto& p : m->params) {
    p.offset = off;
    if (!p.is_int64) off = align_up(off + (size_t)p.numel * 4, 256);
  }
  for (auto& t : m->derived) {
    t.offset = off;
    off = align_up(off + (size_t)t.numel * t.esz, 256);
  }
  m->packed_bytes = off;
}

struct Packed {
  const MplModel* m;
  const uint8_t* base;
  const float* f(const std::string& name) const {
    auto it = m->index.find(name);
    if (it == m->index.end()) throw std::runtime_error("internal: unknown parameter " + name);
    return reinterpret_cast<const float*>(base + m->params[it->second].offset);
  }
  const void* dv(const std::string& name) const {
    auto it = m->dindex.find(name);
    if (it == m->dindex.end()) throw std::runtime_error("internal: unknown derived tensor " + name);
    return base + m->derived[it->second].offset;
  }
  const float* df(const std::string& name) const { return reinterpret_cast<const float*>(dv(name)); }
};

// ---- workspace -------------------------------------------------------------------------------------------------------
struct Workspace {
  float *xs, *xn, *qkv, *att, *hid, *conf;       // SPT, [V*Bc*J, .]
  float* tok;                                    // [Bc, V*tok_w] fp32 residual stream of the FPT
  void *fxn, *fqkv, *fatt, *fhid;                // FPT activations (fp32 / bf16 per precision)
  void* fxl;                                     // LayerNorm-fused bf16 mode: lo plane of the residual stream (fxn = hi plane)
  void* fstats;                                  // [Bc*N, ln_slots] float2 row statistics (LayerNorm-fused bf16 mode)
  float *vn, *pooled, *hn, *h1, *h2, *cat;       // head
  size_t bytes;
};

static Workspace layout_workspace(const MplModel* m, int64_t Bc, uint8_t* base) {
  Workspace w{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    uint8_t* p = base ? base + off : nullptr;
    off = align_up(off + bytes, 256);
    return p;
  };
  const int64_t Rs = (int64_t)m->V * Bc * m->J;
  const int d = m->dim;
  w.xs = (float*)take(Rs * d * 4);
  w.xn = (float*)take(Rs * d * 4);
  if (!m->d.no_transformer_spt && !m->spt_fused) {
    w.qkv = (float*)take(Rs * 3 * d * 4);
    w.att = (float*)take(Rs * d * 4);
    w.hid = (float*)take(Rs * m->spt_hidden * 4);
  }
  if (m->d.confidence_as_attention_uncertainty_weight) w.conf = (float*)take(Rs * 4);
  w.tok = (float*)take(Bc * (int64_t)m->V * m->tok_w * 4);
  if (!m->d.no_transformer_fpt && !m->fpt_kp_fused) {
    const int64_t Rf = m->ln_fused ? (int64_t)align_up((size_t)(Bc * m->fpt_tokens), 256) : Bc * m->fpt_tokens;
    const int64_t D = m->fpt_dim, Hf = m->fpt_hidden;
    const int esz = (m->fpt_tc && m->d.precision == MPL_PREC_BF16) ? 2 : 4;
    w.fxn = take(Rf * D * esz);
    if (m->ln_fused) w.fxl = take(Rf * D * 2);
    if (!m->qkv_attn) w.fqkv = take(Rf * 3 * D * esz);
    w.fatt = take(Rf * D * esz);
    w.fhid = take(Rf * Hf * esz);
    if (m->ln_fused) w.fstats = take(Rf * (size_t)m->ln_slots * 8);
  }
  const int E = m->E, Hd = m->d.hidden_dim, out_dim = 3 * m->J;
  const bool fused_head = !m->d.linear_weighted_mean && !m->d.deep_head && !m->d.head_kadkhod;
  if (!fused_head) {
    w.vn = (float*)take(Bc * (int64_t)m->V * E * 4);
    w.pooled = (float*)take(Bc * (int64_t)E * 4);
    w.hn = (float*)take(Bc * (int64_t)E * 4);
    if (m->d.deep_head || m->d.head_kadkhod) {
      w.h1 = (float*)take(Bc * (int64_t)Hd * 4);
      w.h2 = (float*)take(Bc * (int64_t)Hd * 4);
    }
    if (m->d.head_kadkhod) w.cat = (float*)take(Bc * (int64_t)(out_dim + E) * 4);
  }
  w.bytes = off;
  return w;
}

// ---- forward ---------------------------------------------------------------------------------------------------------
enum ProfCat {
  CAT_EMBED = 0, CAT_SPT_LN, CAT_SPT_LINEAR, CAT_SPT_ATTN, CAT_TOKEN, CAT_FPT_LN, CAT_FPT_QKV, CAT_FPT_ATTN, CAT_FPT_PROJ,
  CAT_FPT_FC1, CAT_FPT_FC2, CAT_HEAD, CAT_SPT_FUSED, CAT_FPT_FUSED, CAT_COUNT
};

static cudaEvent_t prof_event(MplModel* m) {
  if (m->ev_used == m->ev_pool.size()) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    m->ev_pool.push_back(e);
  }
  return m->ev_pool[m->ev_used++];
}

// launch + count (+ bracket with events when profiling)
#define LC(cat, expr)                                        \
  do {                                                       \
    cudaEvent_t e0__ = nullptr, e1__ = nullptr;              \
    if (m->profile) {                                        \
      e0__ = prof_event(m);                                  \
      e1__ = prof_event(m);                                  \
      if (e0__) cudaEventRecord(e0__, s);                    \
    }                                                        \
    MPL_TRY(expr);                                           \
    ++m->launches;                                           \
    if (m->profile && e0__ && e1__) {                        \
      cudaEventRecord(e1__, s);                              \
      m->prof.push_back({(cat), e0__, e1__});                \
    }                                                        \
  } while (0)

static BlockW block_weights(const MplModel* m, const Packed& P, const std::string& p, bool tc) {
  BlockW b{};
  b.n1w = P.f(p + "norm1.weight");
  b.n1b = P.f(p + "norm1.bias");
  b.qkvw = P.f(p + "attn.qkv.weight");
  b.qkvb = m->d.qkv_bias ? P.f(p + "attn.qkv.bias") : P.df("zeros");
  b.projw = P.f(p + "attn.proj.weight");
  b.projb = P.f(p + "attn.proj.bias");
  b.n2w = P.f(p + "norm2.weight");
  b.n2b = P.f(p + "norm2.bias");
  b.fc1w = P.f(p + "mlp.fc1.weight");
  b.fc1b = P.f(p + "mlp.fc1.bias");
  b.fc2w = P.f(p + "mlp.fc2.weight");
  b.fc2b = P.f(p + "mlp.fc2.bias");
  if (tc) {
    const std::string tag = (m->d.precision == MPL_PREC_BF16) ? "bf16:" : "split:";
    if (m->ln_fused) {
      if (m->qkv_attn) {
        b.qa_w = P.dv("qaw:" + p + "attn.qkv");
        b.qa_cs = P.df("qacs:" + p + "attn.qkv");
        b.qa_b = P.df("qab:" + p + "attn.qkv");
      } else {
        b.qkvw_tc = P.dv("lnw:" + p + "attn.qkv");
        b.qkv_cs = P.df("lncs:" + p + "attn.qkv");
        b.qkv_bf = P.df("lnb:" + p + "attn.qkv");
      }
      b.fc1w_tc = P.dv("lnw:" + p + "mlp.fc1");
      b.fc1_cs = P.df("lncs:" + p + "mlp.fc1");
      b.fc1_bf = P.df("lnb:" + p + "mlp.fc1");
    } else {
      b.qkvw_tc = P.dv(tag + p + "attn.qkv.weight");
      b.fc1w_tc = P.dv(tag + p + "mlp.fc1.weight");
    }
    b.projw_tc = P.dv(tag + p + "attn.proj.weight");
    b.fc2w_tc = P.dv(tag + p + "mlp.fc2.weight");
    if (m->perm) {
      b.projb = P.df("pb:" + p + "attn.proj.bias");
      b.fc2b = P.df("pb:" + p + "mlp.fc2.bias");
    }
  }
  return b;
}

// Block.forward (multiview_mpl.py:84-92), fp32 CUDA-core arithmetic; x [rows, C] is updated in place.
static int block_f32(MplModel* m, bool fpt, const BlockW& w, float* x, int64_t rows, int64_t sets, int N, int C, int hidden,
                     float scale, const float* conf, float* xn, float* qkv, float* att, float* hid, cudaStream_t s) {
  const int c_ln = fpt ? CAT_FPT_LN : CAT_SPT_LN, c_at = fpt ? CAT_FPT_ATTN : CAT_SPT_ATTN;
  const int c_qkv = fpt ? CAT_FPT_QKV : CAT_SPT_LINEAR, c_proj = fpt ? CAT_FPT_PROJ : CAT_SPT_LINEAR;
  const int c_fc1 = fpt ? CAT_FPT_FC1 : CAT_SPT_LINEAR, c_fc2 = fpt ? CAT_FPT_FC2 : CAT_SPT_LINEAR;
  LC(c_ln, launch_layernorm(x, C, C, C, w.n1w, w.n1b, 1e-6f, xn, C, rows, C, s));
  LC(c_qkv, launch_linear_f32(xn, C, w.qkvw, w.qkvb, nullptr, 0, qkv, 3 * C, rows, 3 * C, C, ACT_NONE, s));
  LC(c_at, launch_attention_f32(qkv, att, sets, N, m->H, C / m->H, scale, conf, s));
  LC(c_proj, launch_linear_f32(att, C, w.projw, w.projb, x, C, x, C, rows, C, C, ACT_NONE, s));
  LC(c_ln, launch_layernorm(x, C, C, C, w.n2w, w.n2b, 1e-6f, xn, C, rows, C, s));
  LC(c_fc1, launch_linear_f32(xn, C, w.fc1w, w.fc1b, nullptr, 0, hid, hidden, rows, hidden, C, ACT_GELU, s));
  LC(c_fc2, launch_linear_f32(hid, hidden, w.fc2w, w.fc2b, x, C, x, C, rows, C, hidden, ACT_NONE, s));
  return MPL_OK;
}

// Same block with the four projections on tcgen05; LayerNorm / softmax / residual stay fp32.  bf16 mode: bf16 operands (one
// MMA per k-step).  tf32-named mode = fp32-grade "split" arithmetic: every GEMM operand is a pair of bf16 planes (hi, lo) and
// the tensor cores accumulate hi.hi + hi.lo + lo.hi (the producers -- LayerNorm, attention, the fc1 epilogue -- write planes).
static int block_tc(MplModel* m, const BlockW& w, float* x, int64_t rows, int64_t sets, int N, int C, int hidden, float scale,
                    void* xn, void* xl, void* qkv, void* att, void* hid, void* stats, bool last, cudaStream_t s) {
  const int prec = m->d.precision;
  const int hd = C / m->H;
  if (m->ln_fused) {
    // The residual stream lives in two bf16 planes: xn = hi (also the A operand of QKV / fc1), xl = lo; `stats` holds its
    // per-row (sum, sum^2) partials.  All three are rewritten by every residual-emit epilogue (launch_ln_prep makes them from
    // the fp32 tokens before the first block): 5 launches per block, no LayerNorm kernel, x (fp32) is not touched.
    GemmLnArgs app{};  // LayerNorm-apply side (QKV, fc1)
    app.stats_in = stats;
    app.slots_in = m->ln_slots;
    app.eps = 1e-6f;
    GemmLnArgs emit{};  // residual-emit side (proj, fc2)
    emit.stats_out = stats;
    emit.x_lo = xl;
    if (m->qkv_attn) {
      // QKV projection and cross-view attention in one kernel: the q|k|v tensor never exists
      LC(CAT_FPT_QKV, launch_qkv_attn(xn, w.qa_w, w.qa_b, w.qa_cs, stats, m->ln_slots, 1e-6f, att, rows, C, m->H, N, s));
    } else {
      app.colsum = w.qkv_cs;
      LC(CAT_FPT_QKV, launch_gemm_tcgen05(xn, w.qkvw_tc, w.qkv_bf, qkv, rows, 3 * C, C, prec, EPI_LN_BIAS, 0, s, &app));
      LC(CAT_FPT_ATTN, launch_attention_bf16((const __nv_bfloat16*)qkv, (__nv_bfloat16*)att, sets, N, m->H, hd, scale, s));
    }
    LC(CAT_FPT_PROJ, launch_gemm_tcgen05(att, w.projw_tc, w.projb, xn, rows, C, C, prec, EPI_RESIDUAL_EMIT, 0, s, &emit));
    app.colsum = w.fc1_cs;
    app.out_fp16 = 1;   // hidden activations in fp16 (GELU in packed half2), fc2 runs kind::f16 on fp16 operands
    LC(CAT_FPT_FC1, launch_gemm_tcgen05(xn, w.fc1w_tc, w.fc1_bf, hid, rows, hidden, C, prec, EPI_LN_BIAS_GELU, 0, s, &app));
    emit.ab_fp16 = 1;
    // channel-permuted stream: the head reads the first E = J * d channels only, so the last fc2 of the stack leaves the ray
    // half of the residual as it is (half the MMAs, half the residual traffic of that launch)
    const int n_fc2 = (last && m->perm) ? m->E : C;
    emit.ldy = C;
    LC(CAT_FPT_FC2, launch_gemm_tcgen05(hid, w.fc2w_tc, w.fc2b, xn, rows, n_fc2, hidden, prec, EPI_RESIDUAL_EMIT, 0, s, &emit));
    return MPL_OK;
  }
  if (prec == MPL_PREC_BF16) {
    LC(CAT_FPT_LN, launch_layernorm_bf16(x, C, w.n1w, w.n1b, 1e-6f, (__nv_bfloat16*)xn, C, rows, C, s));
    LC(CAT_FPT_QKV, launch_gemm_tcgen05(xn, w.qkvw_tc, w.qkvb, qkv, rows, 3 * C, C, prec, EPI_BIAS, 0, s, nullptr));
    LC(CAT_FPT_ATTN, launch_attention_bf16((const __nv_bfloat16*)qkv, (__nv_bfloat16*)att, sets, N, m->H, hd, scale, s));
    LC(CAT_FPT_PROJ, launch_gemm_tcgen05(att, w.projw_tc, w.projb, x, rows, C, C, prec, EPI_BIAS_RESIDUAL, 1, s, nullptr));
    LC(CAT_FPT_LN, launch_layernorm_bf16(x, C, w.n2w, w.n2b, 1e-6f, (__nv_bfloat16*)xn, C, rows, C, s));
    LC(CAT_FPT_FC1, launch_gemm_tcgen05(xn, w.fc1w_tc, w.fc1b, hid, rows, hidden, C, prec, EPI_BIAS_GELU, 0, s, nullptr));
    LC(CAT_FPT_FC2, launch_gemm_tcgen05(hid, w.fc2w_tc, w.fc2b, x, rows, C, hidden, prec, EPI_BIAS_RESIDUAL, 1, s, nullptr));
  } else {
    // split planes: xn / att [2][rows][C], hid [2][rows][hidden] bf16; qkv [rows][3C] fp32 (the attention arithmetic is fp32).
    // xn is free between the QKV GEMM and the second LayerNorm: it doubles as the fp32 scratch of the attention fallback.
    __nv_bfloat16* xnp = (__nv_bfloat16*)xn;
    __nv_bfloat16* attp = (__nv_bfloat16*)att;
    LC(CAT_FPT_LN, launch_layernorm_split(x, C, w.n1w, w.n1b, 1e-6f, xnp, C, rows * C, rows, C, s));
    LC(CAT_FPT_QKV, launch_gemm_tcgen05(xn, w.qkvw_tc, w.qkvb, qkv, rows, 3 * C, C, prec, EPI_BIAS, 1, s, nullptr));
    LC(CAT_FPT_ATTN, launch_attention_split((const float*)qkv, attp, rows * C, (float*)xn, sets, N, m->H, hd, scale, s));
    LC(CAT_FPT_PROJ, launch_gemm_tcgen05(att, w.projw_tc, w.projb, x, rows, C, C, prec, EPI_BIAS_RESIDUAL, 1, s, nullptr));
    LC(CAT_FPT_LN, launch_layernorm_split(x, C, w.n2w, w.n2b, 1e-6f, xnp, C, rows * C, rows, C, s));
    LC(CAT_FPT_FC1, launch_gemm_tcgen05(xn, w.fc1w_tc, w.fc1b, hid, rows, hidden, C, prec, EPI_BIAS_GELU, 0, s, nullptr));
    LC(CAT_FPT_FC2, launch_gemm_tcgen05(hid, w.fc2w_tc, w.fc2b, x, rows, C, hidden, prec, EPI_BIAS_RESIDUAL, 1, s, nullptr));
  }
  return MPL_OK;
}

static int forward_chunk(MplModel* m, const Packed& P, const float* const* poses, const float* const* rays,
                         const float* const* centers, int64_t pose_stride, int64_t center_stride, float* out, float* aux1,
                         float* aux2, int64_t Bc, const Workspace& w, cudaStream_t s) {
  const MplDesc& d = m->d;
  const int J = m->J, V = m->V, dim = m->dim, E = m->E;
  auto vs = [&](int v) { return m->multi ? std::to_string(v) + "." : std::string(""); };
  // ---- K1 embed (multiview_mpl.py:349-398) ----
  EmbedArgs ea{};
  for (int v = 0; v < V; ++v) {
    ea.poses[v] = poses[v];
    ea.rays[v] = rays ? rays[v] : nullptr;
    ea.centers[v] = centers ? centers[v] : nullptr;
    ea.We[v] = P.f("Spatial_patch_to_embedding." + vs(v) + "weight");
    ea.be[v] = P.f("Spatial_patch_to_embedding." + vs(v) + "bias");
    if (m->conf_emb) {
      ea.Wc[v] = P.f("confidence_to_embedding." + vs(v) + "weight");
      ea.bc[v] = P.f("confidence_to_embedding." + vs(v) + "bias");
    }
    ea.Ps[v] = m->multi ? P.f("Spatial_pos_embed." + std::to_string(v)) : P.f("Spatial_pos_embed");
  }
  ea.pose_stride = pose_stride;
  ea.center_stride = center_stride;
  ea.B = Bc;
  ea.in_ch = m->in_ch;
  ea.add_conf = m->add_conf;
  ea.mult_conf = m->mult_conf;
  ea.spatial_pos_mode = 0;
  if (d.add_3D_pos_encoding_in_Spatial && rays != nullptr && centers != nullptr) {
    if (d.pose_3d_emb_learnable) {
      ea.spatial_pos_mode = 1;
      ea.pos3d = P.f("pos_3d_embed");
      ea.pos3d_ld = m->pos3d_w;
    } else {
      ea.spatial_pos_mode = 2;
      ea.Wl = P.f("pos_3d_linear.weight");
      ea.bl = P.f("pos_3d_linear.bias");
    }
  }
  ea.V = V; ea.J = J; ea.d = dim;
  ea.x = w.xs;
  ea.conf = w.conf;
  // ---- token build arguments (:463-499); the launch itself follows the SPT unless the SPT kernel fuses it ----
  TokenArgs ta{};
  ta.xn = w.xn;
  for (int v = 0; v < V; ++v) {
    ta.poses[v] = poses[v];
    ta.rays[v] = rays ? rays[v] : nullptr;
    ta.centers[v] = centers ? centers[v] : nullptr;
  }
  ta.pose_stride = pose_stride;
  ta.center_stride = center_stride;
  ta.B = Bc;
  if (d.confidence_in_FPT) {
    ta.Wcf = P.f("confidence_to_embedding_FPT.weight");
    ta.bcf = P.f("confidence_to_embedding_FPT.bias");
  }
  if (d.input_rays_as_token) {
    ta.Wr = P.f("ray_to_embedding.weight");
    ta.br = P.f("ray_to_embedding.bias");
  }
  if (!d.add_3D_pos_encoding_in_Spatial) {
    if (d.pose_3d_emb_learnable) {
      ta.pos_table = P.f("pos_3d_embed");
      ta.pos_w = m->pos3d_w;
    } else {
      ta.Wl = P.f("pos_3d_linear.weight");
      ta.bl = P.f("pos_3d_linear.bias");
      ta.pos_w = m->pos3d_lin_out;
    }
  } else {
    ta.pos_table = P.f("pos_3d_view_coding");
    ta.pos_w = m->pos3d_w;
  }
  ta.ray_layout = m->ray_layout;
  ta.V = V; ta.J = J; ta.d = dim; ta.tok_w = m->tok_w;
  ta.tok = w.tok;
  // the single-kernel SPT computes the embedding in its prologue and writes the FPT tokens from its epilogue
  const bool fuse_embed = m->spt_fused && ea.spatial_pos_mode != 2;
  const bool fuse_token = m->spt_fused;
  // LayerNorm-fused mode: the FPT residual stream lives in two bf16 planes (+ per-row statistics).  The single-kernel SPT
  // writes them from its epilogue; any other producer leaves fp32 tokens and launch_ln_prep converts them.
  const bool planes = m->ln_fused && !d.no_transformer_fpt && m->depth > 0 && !m->fpt_kp_fused;
  const bool spt_planes = planes && fuse_token;
  if (spt_planes) {
    ta.tok_hi = (__nv_bfloat16*)w.fxn;
    ta.tok_lo = (__nv_bfloat16*)w.fxl;
    ta.stats = reinterpret_cast<float2*>(w.fstats);
    ta.stat_slots = m->ln_slots;
    ta.stats_ld = (int64_t)align_up((size_t)(Bc * m->fpt_tokens), 256);
    ta.perm_layout = m->perm ? 1 : 0;
  }
  if (!fuse_embed) LC(CAT_EMBED, launch_embed(ea, s));
  // ---- SPT blocks (multiview_mpl.py:400-410): conf-weighted pass, last block twice; then Spatial_norm (:412) ----
  const int64_t Rs = (int64_t)V * Bc * J;
  if (m->spt_fused) {
    const void* wp[kMaxViews];
    for (int v = 0; v < V; ++v) wp[v] = P.dv("sptpack:" + std::to_string(m->multi ? v : 0));
    SptIo io{ea, ta};
    LC(CAT_SPT_FUSED, launch_spt_fused(fuse_embed ? nullptr : w.xs, fuse_token ? nullptr : w.xn, wp, V, Bc, m->depth,
                                       P.f("Spatial_norm.weight"), P.f("Spatial_norm.bias"), fuse_embed ? nullptr : w.conf,
                                       d.confidence_as_attention_uncertainty_weight ? 1 : 0, &io,
                                       d.precision == MPL_PREC_TF32 ? 1 : 0, s));
  } else {
    if (!d.no_transformer_spt && m->depth > 0) {
      const int hd = dim / m->H;
      const float scale = d.qk_scale != 0.f ? d.qk_scale : 1.0f / sqrtf((float)hd);
      const int stacks = m->multi ? V : 1;
      const int64_t rows_per_stack = (m->multi ? 1 : V) * Bc * J;
      for (int st = 0; st < stacks; ++st) {
        float* x = w.xs + (int64_t)st * rows_per_stack * dim;
        const float* cf = w.conf ? w.conf + (int64_t)st * rows_per_stack : nullptr;
        const std::string vp = m->multi ? std::to_string(st) + "." : std::string("");
        for (int ix = 0; ix < m->depth; ++ix) {
          const BlockW bw = block_weights(m, P, "Spatial_blocks." + vp + std::to_string(ix) + ".", false);
          const int reps = 1 + (ix == m->depth - 1 ? 1 : 0);
          if (cf != nullptr)
            MPL_TRY(block_f32(m, false, bw, x, rows_per_stack, rows_per_stack / J, J, dim, m->spt_hidden, scale, cf, w.xn, w.qkv, w.att, w.hid, s));
          for (int r = 0; r < reps; ++r)
            MPL_TRY(block_f32(m, false, bw, x, rows_per_stack, rows_per_stack / J, J, dim, m->spt_hidden, scale, nullptr, w.xn, w.qkv, w.att, w.hid, s));
        }
      }
    }
    LC(CAT_TOKEN, launch_layernorm(w.xs, dim, dim, dim, P.f("Spatial_norm.weight"), P.f("Spatial_norm.bias"), 1e-6f, w.xn, dim, Rs, dim, s));
  }
  if (!fuse_token) LC(CAT_TOKEN, launch_token_build(ta, s));
  // ---- FPT blocks (multiview_mpl.py:416-423) ----
  if (m->fpt_kp_fused) {
    LC(CAT_FPT_FUSED, launch_fpt_kp_fused(w.tok, P.dv("fptpack"), V, Bc, m->depth, s));
  } else if (!d.no_transformer_fpt && m->depth > 0) {
    const int D = m->fpt_dim, N = m->fpt_tokens;
    const int hd = D / m->H;
    const float scale = d.qk_scale != 0.f ? d.qk_scale : 1.0f / sqrtf((float)hd);
    const int64_t rows = Bc * N;
    if (m->ln_fused && !spt_planes)
      LC(CAT_FPT_LN, launch_ln_prep(w.tok, D, (__nv_bfloat16*)w.fxn, (__nv_bfloat16*)w.fxl, D, w.fstats, m->ln_slots, rows, D, s));
    if (m->resolved_for != P.base) {  // once per packed blob: no string lookups on the launch path afterwards
      m->fpt_blocks.clear();
      for (int ix = 0; ix < m->depth; ++ix) m->fpt_blocks.push_back(block_weights(m, P, "blocks." + std::to_string(ix) + ".", m->fpt_tc));
      m->resolved_for = P.base;
    }
    for (int ix = 0; ix < m->depth; ++ix) {
      const BlockW& bw = m->fpt_blocks[ix];
      const int reps = 1 + (ix == m->depth - 1 ? 1 : 0);
      for (int r = 0; r < reps; ++r) {
        if (m->fpt_tc)
          MPL_TRY(block_tc(m, bw, w.tok, rows, Bc, N, D, m->fpt_hidden, scale, w.fxn, w.fxl, w.fqkv, w.fatt, w.fhid, w.fstats,
                           ix == m->depth - 1 && r == reps - 1, s));
        else
          MPL_TRY(block_f32(m, true, bw, w.tok, rows, Bc, N, D, m->fpt_hidden, scale, nullptr, (float*)w.fxn, (float*)w.fqkv, (float*)w.fatt, (float*)w.fhid, s));
      }
    }
  }
  // ---- ray strip + View_norm + weighted mean + head (multiview_mpl.py:425-446, 506-523) ----
  int seg_len = E, seg_stride = E;
  if (m->ray_layout == 1 && !m->perm) { seg_len = dim; seg_stride = 2 * dim; }  // [J, 2d] -> first d of every joint slot
  const int out_dim = 3 * J;
  const bool fused_head = !d.linear_weighted_mean && !d.deep_head && !d.head_kadkhod;
  // LayerNorm-fused mode: the FPT left the residual stream in two bf16 planes.  The K5 head kernel reads them directly; every
  // other head takes the fp32 token buffer, refilled from the planes first.
  bool head_planes = false;
  if (planes) {
    HeadArgs probe{};
    probe.E = E; probe.out_dim = out_dim; probe.seg_len = seg_len; probe.seg_stride = seg_stride; probe.tok_w = m->tok_w;
    head_planes = fused_head && m->dindex.count("headT") && head_warp_supports(probe);
    if (!head_planes)
      LC(CAT_HEAD, launch_join_planes((const __nv_bfloat16*)w.fxn, (const __nv_bfloat16*)w.fxl, w.tok, Bc * (int64_t)V * m->tok_w, s));
  }
  if (fused_head) {
    HeadArgs ha{};
    ha.tok = w.tok;
    if (head_planes) { ha.tok_hi = (const __nv_bfloat16*)w.fxn; ha.tok_lo = (const __nv_bfloat16*)w.fxl; } ha.B = Bc; ha.V = V; ha.tok_w = m->tok_w; ha.E = E; ha.seg_len = seg_len; ha.seg_stride = seg_stride;
    ha.out_dim = out_dim;
    ha.vn_w = P.f("View_norm.weight"); ha.vn_b = P.f("View_norm.bias");
    ha.wm_w = P.f("weighted_mean.weight"); ha.wm_b = P.f("weighted_mean.bias");
    ha.hn_w = P.f("head.0.weight"); ha.hn_b = P.f("head.0.bias");
    ha.hw = P.f("head.1.weight"); ha.hb = P.f("head.1.bias");
    ha.hwT = m->dindex.count("headT") ? P.df("headT") : nullptr;
    ha.out = out;
    LC(CAT_HEAD, launch_head_fused(ha, s));
    return MPL_OK;
  }
  LC(CAT_HEAD, launch_layernorm(w.tok, m->tok_w, seg_len, seg_stride, P.f("View_norm.weight"), P.f("View_norm.bias"), 1e-6f, w.vn, E,
                     Bc * V, E, s));
  if (d.linear_weighted_mean)
    LC(CAT_HEAD, launch_linear_f32(w.vn, (int64_t)V * E, P.f("weighted_mean.weight"), P.f("weighted_mean.bias"), nullptr, 0, w.pooled, E, Bc, E, V * E, ACT_NONE, s));
  else
    LC(CAT_HEAD, launch_view_mean(w.vn, P.f("weighted_mean.weight"), P.f("weighted_mean.bias"), w.pooled, Bc, V, E, s));
  const int Hd = d.hidden_dim;
  if (d.head_kadkhod) {
    // three residual stages; stage s > 0 consumes cat([previous prediction, pooled]) (multiview_mpl.py:506-516)
    float* stage_out[3] = {aux1, aux2, out};
    for (int st = 0; st < 3; ++st) {
      const std::string p = "head." + std::to_string(st) + ".";
      const float* in;
      int in_w;
      if (st == 0) {
        LC(CAT_HEAD, launch_layernorm(w.pooled, E, E, E, P.f(p + "0.0.weight"), P.f(p + "0.0.bias"), 1e-5f, w.hn, E, Bc, E, s));
        in = w.hn;
        in_w = E;
        LC(CAT_HEAD, launch_linear_f32(in, in_w, P.df("fold:" + p + "0.1.weight"), P.df("fold:" + p + "0.1.bias"), nullptr, 0, w.h1, Hd, Bc, Hd, in_w, ACT_RELU, s));
      } else {
        // cat = [prev (3J) | pooled (E)]
        MPL_CUDA(cudaMemcpy2DAsync(w.cat, (size_t)(out_dim + E) * 4, stage_out[st - 1], (size_t)out_dim * 4, (size_t)out_dim * 4, Bc, cudaMemcpyDeviceToDevice, s));
        MPL_CUDA(cudaMemcpy2DAsync(w.cat + out_dim, (size_t)(out_dim + E) * 4, w.pooled, (size_t)E * 4, (size_t)E * 4, Bc, cudaMemcpyDeviceToDevice, s));
        in = w.cat;
        in_w = out_dim + E;
        LC(CAT_HEAD, launch_linear_f32(in, in_w, P.df("fold:" + p + "0.0.weight"), P.df("fold:" + p + "0.0.bias"), nullptr, 0, w.h1, Hd, Bc, Hd, in_w, ACT_RELU, s));
      }
      LC(CAT_HEAD, launch_linear_f32(w.h1, Hd, P.df("fold:" + p + "1.0.weight"), P.df("fold:" + p + "1.0.bias"), nullptr, 0, w.h2, Hd, Bc, Hd, Hd, ACT_RELU, s));
      LC(CAT_HEAD, launch_linear_f32(w.h2, Hd, P.df("fold:" + p + "2.0.weight"), P.df("fold:" + p + "2.0.bias"), nullptr, 0, w.h1, Hd, Bc, Hd, Hd, ACT_RELU, s));
      LC(CAT_HEAD, launch_linear_f32(w.h1, Hd, P.f(p + "3.weight"), P.f(p + "3.bias"), nullptr, 0, stage_out[st], out_dim, Bc, out_dim, Hd, ACT_NONE, s));
    }
    return MPL_OK;
  }
  LC(CAT_HEAD, launch_layernorm(w.pooled, E, E, E, P.f("head.0.weight"), P.f("head.0.bias"), 1e-5f, w.hn, E, Bc, E, s));
  if (d.deep_head) {
    LC(CAT_HEAD, launch_linear_f32(w.hn, E, P.df("fold:head.1.weight"), P.df("fold:head.1.bias"), nullptr, 0, w.h1, Hd, Bc, Hd, E, ACT_RELU, s));
    LC(CAT_HEAD, launch_linear_f32(w.h1, Hd, P.df("fold:head.4.weight"), P.df("fold:head.4.bias"), nullptr, 0, w.h2, Hd, Bc, Hd, Hd, ACT_RELU, s));
    LC(CAT_HEAD, launch_linear_f32(w.h2, Hd, P.df("fold:head.7.weight"), P.df("fold:head.7.bias"), nullptr, 0, w.h1, Hd, Bc, Hd, Hd, ACT_RELU, s));
    LC(CAT_HEAD, launch_linear_f32(w.h1, Hd, P.f("head.10.weight"), P.f("head.10.bias"), nullptr, 0, out, out_dim, Bc, out_dim, Hd, ACT_NONE, s));
  } else {
    LC(CAT_HEAD, launch_linear_f32(w.hn, E, P.f("head.1.weight"), P.f("head.1.bias"), nullptr, 0, out, out_dim, Bc, out_dim, E, ACT_NONE, s));
  }
  return MPL_OK;
}

}  // namespace mpl

// =====================================================================================================================
// extern "C" boundary
// =====================================================================================================================
#define MPL_API_BEGIN try {
#define MPL_API_END                                  \
  }                                                  \
  catch (const std::exception& e) {                  \
    mpl::set_error("%s", e.what());                  \
    return MPL_ERR_INVALID_ARGUMENT;                 \
  }

extern "C" {

const char* mpl_last_error(void) { return g_last_error.c_str(); }
int mpl_abi_version(void) { return MPL_ABI_VERSION; }

int mpl_create(const MplDesc* desc, MplModel** out) {
  MPL_API_BEGIN
  if (desc == nullptr || out == nullptr) {
    set_error("mpl_create: null argument");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (desc->struct_size != (int32_t)sizeof(MplDesc)) {
    set_error("mpl_create: MplDesc.struct_size = %d, library expects %d", desc->struct_size, (int)sizeof(MplDesc));
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (desc->precision < MPL_PREC_FP32 || desc->precision > MPL_PREC_BF16) {
    set_error("mpl_create: unknown precision %d", desc->precision);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (desc->gemm_cta_group != 0 && desc->gemm_cta_group != 2) {
    set_error("mpl_create: gemm_cta_group must be 0 or 2 (CTA pairs), got %d", desc->gemm_cta_group);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (desc->chunk_streams != 0 && desc->chunk_streams != 1) {
    set_error("mpl_create: chunk_streams must be 0 or 1 (the caller's stream), got %d", desc->chunk_streams);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  *out = nullptr;
  MplModel* m = new MplModel();
  m->d = *desc;
  const MplDesc& d = m->d;
  m->J = d.num_joints; m->V = d.num_views; m->dim = d.embed_dim_ratio; m->H = d.num_heads; m->depth = d.depth;
  m->in_ch = d.confidence_input_as_third ? d.in_chans + 1 : d.in_chans;
  m->add_conf = d.add_confidence_input && !d.concat_confidence_emb;  // Q3 (multiview_mpl.py:173-176)
  m->mult_conf = d.mult_confidence_emb && !d.concat_confidence_emb;
  m->conf_emb = m->add_conf || m->mult_conf;
  m->multi = d.multiple_spatial_blocks != 0;
  m->E = m->dim * m->J;
  m->tok_w = m->E * (d.input_rays_as_token ? 2 : 1);
  m->ray_layout = !d.input_rays_as_token ? 0 : (d.add_3D_pos_encoding_to_rays ? 1 : 2);
  if (d.FPT_blocks_view_keypoint_tokens) { m->fpt_dim = m->dim; m->fpt_tokens = m->V * m->J; }
  else { m->fpt_dim = m->tok_w; m->fpt_tokens = m->V; }
  m->pos3d_lin_out = (d.add_3D_pos_encoding_to_rays && !d.add_3D_pos_encoding_in_Spatial) ? 2 * m->dim : m->dim;
  m->pos3d_w = d.add_3D_pos_encoding_to_rays ? 2 * m->dim : m->dim;
  // int(dim * mlp_ratio) as the reference computes it in float64 (multiview_mpl.py:25-26,78): the host passes the two integers,
  // because the ratio itself crosses the ABI as a float (0.7 * 10 = 7 in float64, 6 in float32)
  m->spt_hidden = d.spt_hidden > 0 ? d.spt_hidden : (int)((double)m->dim * (double)d.mlp_ratio);
  m->fpt_hidden = d.fpt_hidden > 0 ? d.fpt_hidden : (int)((double)m->fpt_dim * (double)d.mlp_ratio);
  m->n_out = d.head_kadkhod ? 3 : 1;
  const int st = validate(m);
  if (st != MPL_OK) {
    delete m;
    return st;
  }
  m->spt_fused = d.precision != MPL_PREC_FP32 && !d.no_transformer_spt && m->depth > 0 &&
                 spt_fused_supports(m->J, m->dim, m->H, m->spt_hidden);
  // keypoint-token FPT: same block shape as the SPT (width 32, 8 heads, hidden 64, sets of 17 rows) -> same kernel, grouped
  m->fpt_kp_fused = d.precision == MPL_PREC_BF16 && d.FPT_blocks_view_keypoint_tokens && !d.no_transformer_fpt && m->depth > 0 &&
                    m->V <= 16 && spt_fused_supports(m->J, m->fpt_dim, m->H, m->fpt_hidden);
  m->fpt_tc = false;
  if (d.precision != MPL_PREC_FP32 && !d.no_transformer_fpt && m->depth > 0 && !m->fpt_kp_fused) {
    const bool ok = gemm_tcgen05_supports(3 * m->fpt_dim, m->fpt_dim, d.precision) &&
                    gemm_tcgen05_supports(m->fpt_dim, m->fpt_dim, d.precision) &&
                    gemm_tcgen05_supports(m->fpt_hidden, m->fpt_dim, d.precision) &&
                    gemm_tcgen05_supports(m->fpt_dim, m->fpt_hidden, d.precision);
    if (!ok) {
      delete m;
      set_error("precision mode %d needs FPT widths that are multiples of 16 (fpt_dim=%d, hidden=%d); use MPL_PREC_FP32",
                d.precision, m->fpt_dim, m->fpt_hidden);
      return MPL_ERR_UNSUPPORTED;
    }
    m->fpt_tc = true;
  }
  // LayerNorm fusion: the residual-emit epilogue works on whole 32-column chunks, launch_ln_prep on float4 rows
  m->ln_fused = m->fpt_tc && d.precision == MPL_PREC_BF16 && d.ln_fusion != 0 && m->fpt_dim % 32 == 0 && m->fpt_dim <= 32 * 4 * 17;
  m->ln_slots = m->ln_fused ? gemm_ln_slots(m->fpt_dim) : 0;
  m->qkv_attn = m->ln_fused && d.qkv_attn_fusion != 0 && qkv_attn_supports(m->fpt_dim, m->H, m->fpt_tokens);
  {
    // channel-permuted residual stream (see MplModel::perm): every producer and consumer of the planes must be one that
    // knows the permutation -- the SPT epilogue, the LN-fused GEMMs and the K5 head reading the planes
    HeadArgs probe{};
    probe.E = m->E; probe.out_dim = 3 * m->J; probe.seg_len = m->E; probe.seg_stride = m->E; probe.tok_w = m->tok_w;
    const bool k5 = !d.linear_weighted_mean && !d.deep_head && !d.head_kadkhod && 3 * m->J <= 64 && head_warp_supports(probe);
    m->perm = m->ln_fused && m->ray_layout == 1 && m->spt_fused && !m->fpt_kp_fused && !d.no_transformer_fpt && m->depth > 0 &&
              k5 && m->fpt_dim == 2 * m->E && gemm_tcgen05_supports(m->E, m->fpt_hidden, d.precision);
    if (m->perm) {
      m->perm_host.resize(m->fpt_dim);
      for (int c = 0; c < m->fpt_dim; ++c) {
        const int half = c / m->E, e = c % m->E;  // packed: [pose parts | ray parts]; reference: [x_j | ray_j] per joint
        m->perm_host[c] = (e / m->dim) * 2 * m->dim + half * m->dim + e % m->dim;
      }
    }
  }
  build_tables(m);
  *out = m;
  return MPL_OK;
  MPL_API_END
}

void mpl_destroy(MplModel* m) {
  if (m == nullptr) return;
  for (auto& e : m->graphs) cudaGraphExecDestroy(e.exec);
  if (m->cap_stream) cudaStreamDestroy(m->cap_stream);
  for (cudaEvent_t e : m->ev_pool) cudaEventDestroy(e);
  delete m;
}

int mpl_set_profile(MplModel* m, int enabled) {
  if (m == nullptr) {
    set_error("mpl_set_profile: null handle");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  m->profile = enabled != 0;
  m->prof.clear();
  m->ev_used = 0;
  return MPL_OK;
}

int mpl_profile_categories(void) { return CAT_COUNT; }

const char* mpl_profile_category_name(int cat) {
  static const char* names[CAT_COUNT] = {"embed", "spt_layernorm", "spt_linear", "spt_attention", "token_build", "fpt_layernorm",
                                         "fpt_gemm_qkv", "fpt_attention", "fpt_gemm_proj", "fpt_gemm_fc1", "fpt_gemm_fc2", "head",
                                         "spt_fused", "fpt_kp_fused"};
  return (cat >= 0 && cat < CAT_COUNT) ? names[cat] : "";
}

int mpl_profile_collect(MplModel* m, double* ms_per_category, int64_t* launches_per_category, int n) {
  if (m == nullptr || ms_per_category == nullptr || launches_per_category == nullptr || n < CAT_COUNT) {
    set_error("mpl_profile_collect: bad argument (need arrays of mpl_profile_categories() entries)");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  for (int i = 0; i < n; ++i) { ms_per_category[i] = 0.0; launches_per_category[i] = 0; }
  for (auto& r : m->prof) {
    MPL_CUDA(cudaEventSynchronize(r.e1));
    float ms = 0.f;
    MPL_CUDA(cudaEventElapsedTime(&ms, r.e0, r.e1));
    ms_per_category[r.cat] += ms;
    launches_per_category[r.cat] += 1;
  }
  m->prof.clear();
  m->ev_used = 0;
  return MPL_OK;
}

int mpl_num_params(const MplModel* m) { return m ? (int)m->params.size() : 0; }

int mpl_param_info(const MplModel* m, int index, const char** name, int64_t* numel, int32_t* is_int64) {
  if (m == nullptr || index < 0 || index >= (int)m->params.size()) {
    set_error("mpl_param_info: index out of range");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (name) *name = m->params[index].name.c_str();
  if (numel) *numel = m->params[index].numel;
  if (is_int64) *is_int64 = m->params[index].is_int64 ? 1 : 0;
  return MPL_OK;
}

int64_t mpl_dim(const MplModel* m, int which) {
  if (m == nullptr) return -1;
  switch (which) {
    case 0: return m->tok_w;
    case 1: return m->fpt_dim;
    case 2: return m->fpt_tokens;
    case 3: return m->E;
    case 4: return m->spt_hidden;
    case 5: return m->fpt_hidden;
    case 6: return m->n_out;
    case 7: return m->perm ? m->E : m->fpt_dim;
    default: return -1;
  }
}

size_t mpl_packed_bytes(const MplModel* m) { return m ? m->packed_bytes : 0; }

int mpl_pack_weights(MplModel* m, const void* const* params, int num_params, void* packed, size_t packed_bytes,
                     mpl_stream_t stream) {
  MPL_API_BEGIN
  if (m == nullptr || params == nullptr || packed == nullptr) {
    set_error("mpl_pack_weights: null argument");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (num_params != (int)m->params.size()) {
    set_error("mpl_pack_weights: got %d parameter pointers, the model has %d", num_params, (int)m->params.size());
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (packed_bytes < m->packed_bytes) {
    set_error("mpl_pack_weights: packed buffer has %zu bytes, %zu needed", packed_bytes, m->packed_bytes);
    return MPL_ERR_WORKSPACE;
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* base = reinterpret_cast<uint8_t*>(packed);
  for (size_t i = 0; i < m->params.size(); ++i) {
    const ParamInfo& p = m->params[i];
    if (p.is_int64) continue;
    if (params[i] == nullptr) {
      set_error("mpl_pack_weights: parameter %s is null", p.name.c_str());
      return MPL_ERR_INVALID_ARGUMENT;
    }
    MPL_CUDA(cudaMemcpyAsync(base + p.offset, params[i], (size_t)p.numel * 4, cudaMemcpyDeviceToDevice, s));
  }
  Packed P{m, base};
  for (auto& f : m->folds) {
    float* Wf = const_cast<float*>(P.df("fold:" + f.lin + "weight"));
    float* bf = const_cast<float*>(P.df("fold:" + f.lin + "bias"));
    MPL_TRY(launch_fold_bn(P.f(f.lin + "weight"), P.f(f.lin + "bias"), P.f(f.bn + "weight"), P.f(f.bn + "bias"),
                           P.f(f.bn + "running_mean"), P.f(f.bn + "running_var"), 1e-5f, Wf, bf, f.N, f.K, s));
  }
  {
    const Derived& z = m->derived[m->dindex.at("zeros")];
    MPL_CUDA(cudaMemsetAsync(base + z.offset, 0, (size_t)z.numel * 4, s));
  }
  if (m->dindex.count("headT")) {
    const Derived& ht = m->derived[m->dindex.at("headT")];
    MPL_TRY(launch_head_transpose(P.f("head.1.weight"), reinterpret_cast<float*>(base + ht.offset), 3 * m->J, m->E, s));
  }
  if (m->spt_fused) {
    const int stacks = m->multi ? m->V : 1;
    const float spt_scale = m->d.qk_scale != 0.f ? m->d.qk_scale : 1.0f / sqrtf((float)(m->dim / m->H));
    for (int st = 0; st < stacks; ++st) {
      const Derived& dd = m->derived[m->dindex.at("sptpack:" + std::to_string(st))];
      for (int l = 0; l < m->depth; ++l) {
        const std::string p = "Spatial_blocks." + (m->multi ? std::to_string(st) + "." : std::string("")) + std::to_string(l) + ".";
        MPL_TRY(launch_spt_pack_layer(P.f(p + "norm1.weight"), P.f(p + "norm1.bias"), P.f(p + "attn.qkv.weight"),
                                      m->d.qkv_bias ? P.f(p + "attn.qkv.bias") : nullptr, P.f(p + "attn.proj.weight"),
                                      P.f(p + "attn.proj.bias"), P.f(p + "norm2.weight"), P.f(p + "norm2.bias"),
                                      P.f(p + "mlp.fc1.weight"), P.f(p + "mlp.fc1.bias"), P.f(p + "mlp.fc2.weight"),
                                      P.f(p + "mlp.fc2.bias"), spt_scale, base + dd.offset + (size_t)l * spt_fused_layer_bytes(), s));
      }
    }
  }
  if (m->fpt_kp_fused) {
    const Derived& dd = m->derived[m->dindex.at("fptpack")];
    const float kp_scale = m->d.qk_scale != 0.f ? m->d.qk_scale : 1.0f / sqrtf((float)(m->fpt_dim / m->H));
    for (int l = 0; l < m->depth; ++l) {
      const std::string p = "blocks." + std::to_string(l) + ".";
      MPL_TRY(launch_spt_pack_layer(P.f(p + "norm1.weight"), P.f(p + "norm1.bias"), P.f(p + "attn.qkv.weight"),
                                    m->d.qkv_bias ? P.f(p + "attn.qkv.bias") : nullptr, P.f(p + "attn.proj.weight"),
                                    P.f(p + "attn.proj.bias"), P.f(p + "norm2.weight"), P.f(p + "norm2.bias"),
                                    P.f(p + "mlp.fc1.weight"), P.f(p + "mlp.fc1.bias"), P.f(p + "mlp.fc2.weight"),
                                    P.f(p + "mlp.fc2.bias"), kp_scale, base + dd.offset + (size_t)l * spt_fused_layer_bytes(), s));
    }
  }
  if (m->fpt_tc) {
    const bool bf = m->d.precision == MPL_PREC_BF16;
    const std::string tag = bf ? "bf16:" : "split:";
    const int* perm = nullptr;
    if (m->perm) {
      int* dp = reinterpret_cast<int*>(base + m->derived[m->dindex.at("perm")].offset);
      MPL_CUDA(cudaMemcpyAsync(dp, m->perm_host.data(), m->perm_host.size() * sizeof(int), cudaMemcpyHostToDevice, s));
      perm = dp;
    }
    for (int l = 0; l < m->depth; ++l) {
      const std::string p = "blocks." + std::to_string(l) + ".";
      if (m->ln_fused) {
        const int D = m->fpt_dim, Hf = m->fpt_hidden;
        auto mut = [&](const std::string& name) { return base + m->derived[m->dindex.at(name)].offset; };
        if (m->qkv_attn) {
          const float fscale = m->d.qk_scale != 0.f ? m->d.qk_scale : 1.0f / sqrtf((float)(D / m->H));
          MPL_TRY(launch_qkv_attn_pack(P.f(p + "attn.qkv.weight"), m->d.qkv_bias ? P.f(p + "attn.qkv.bias") : nullptr,
                                       P.f(p + "norm1.weight"), P.f(p + "norm1.bias"), mut("qaw:" + p + "attn.qkv"),
                                       reinterpret_cast<float*>(mut("qacs:" + p + "attn.qkv")),
                                       reinterpret_cast<float*>(mut("qab:" + p + "attn.qkv")), m->H, D, fscale, s, perm));
        } else {
          MPL_TRY(launch_ln_fold(P.f(p + "attn.qkv.weight"), m->d.qkv_bias ? P.f(p + "attn.qkv.bias") : nullptr, P.f(p + "norm1.weight"),
                                 P.f(p + "norm1.bias"), reinterpret_cast<__nv_bfloat16*>(mut("lnw:" + p + "attn.qkv")),
                                 reinterpret_cast<float*>(mut("lncs:" + p + "attn.qkv")),
                                 reinterpret_cast<float*>(mut("lnb:" + p + "attn.qkv")), 3 * D, D, s, perm));
        }
        MPL_TRY(launch_ln_fold(P.f(p + "mlp.fc1.weight"), P.f(p + "mlp.fc1.bias"), P.f(p + "norm2.weight"), P.f(p + "norm2.bias"),
                               reinterpret_cast<__nv_bfloat16*>(mut("lnw:" + p + "mlp.fc1")),
                               reinterpret_cast<float*>(mut("lncs:" + p + "mlp.fc1")),
                               reinterpret_cast<float*>(mut("lnb:" + p + "mlp.fc1")), Hf, D, s, perm));
        if (perm != nullptr) {
          // the residual-emit GEMMs write permuted channels: rows of W and entries of the bias in packed order
          MPL_TRY(launch_to_half_rows(P.f(p + "attn.proj.weight"), mut(tag + p + "attn.proj.weight"), D, D, perm, 0, s));
          MPL_TRY(launch_to_half_rows(P.f(p + "mlp.fc2.weight"), mut(tag + p + "mlp.fc2.weight"), D, Hf, perm, 1, s));
          MPL_TRY(launch_gather_f32(P.f(p + "attn.proj.bias"), reinterpret_cast<float*>(mut("pb:" + p + "attn.proj.bias")), D, perm, s));
          MPL_TRY(launch_gather_f32(P.f(p + "mlp.fc2.bias"), reinterpret_cast<float*>(mut("pb:" + p + "mlp.fc2.bias")), D, perm, s));
          continue;
        }
      }
      for (const char* wn : {"attn.qkv.weight", "attn.proj.weight", "mlp.fc1.weight", "mlp.fc2.weight"}) {
        if (m->ln_fused && (std::string(wn) == "attn.qkv.weight" || std::string(wn) == "mlp.fc1.weight")) continue;
        const float* src = P.f(p + wn);
        const Derived& dd = m->derived[m->dindex.at(tag + p + wn)];
        if (bf && m->ln_fused && std::string(wn) == "mlp.fc2.weight") MPL_TRY(launch_to_f16(src, base + dd.offset, dd.numel, s));
        else if (bf) MPL_TRY(launch_to_bf16(src, reinterpret_cast<__nv_bfloat16*>(base + dd.offset), dd.numel, s));
        else MPL_TRY(launch_to_split(src, reinterpret_cast<__nv_bfloat16*>(base + dd.offset), dd.numel, dd.numel, s));
      }
    }
  }
  return MPL_OK;
  MPL_API_END
}

int64_t mpl_chunk_poses(const MplModel* m) { return m ? m->chunk : 0; }
int mpl_set_chunk_poses(MplModel* m, int64_t chunk) {
  if (m == nullptr || chunk < 1) {
    set_error("mpl_set_chunk_poses: chunk must be >= 1");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  m->chunk = chunk;
  for (auto& e : m->graphs) cudaGraphExecDestroy(e.exec);  // captured graphs bake the chunking in
  m->graphs.clear();
  return MPL_OK;
}

size_t mpl_workspace_bytes(const MplModel* m, int64_t max_batch) {
  if (m == nullptr || max_batch < 0) return 0;
  const int64_t Bc = std::min<int64_t>(std::max<int64_t>(max_batch, 1), m->chunk);
  return layout_workspace(m, Bc, nullptr).bytes;
}

int mpl_forward(MplModel* m, const void* packed, const float* const* poses, const float* const* rays,
                const float* const* centers, int64_t pose_stride, int64_t center_stride, float* out, float* aux1,
                float* aux2, int64_t batch, void* workspace, size_t workspace_bytes, mpl_stream_t stream) {
  MPL_API_BEGIN
  if (m == nullptr || batch < 0) {
    set_error("mpl_forward: null handle or negative batch");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) {  // empty batch: nothing to enqueue (device pointers of empty tensors are null)
    m->launches = 0;
    return MPL_OK;
  }
  if (packed == nullptr || poses == nullptr || out == nullptr) {
    set_error("mpl_forward: null argument");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  const MplDesc& d = m->d;
  // rays / centers are needed whenever a ray embedding or the ray-direction positional encoding is live
  const bool need_rays = d.input_rays_as_token || (!d.add_3D_pos_encoding_in_Spatial && !d.pose_3d_emb_learnable);
  if (need_rays && (rays == nullptr || centers == nullptr)) {
    set_error("mpl_forward: this configuration consumes rays and centers (multiview_mpl.py:469-489); got null");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (d.head_kadkhod && (aux1 == nullptr || aux2 == nullptr)) {
    set_error("mpl_forward: head_kadkhod returns (x, [x1, x2]); aux1/aux2 must be provided");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  for (int v = 0; v < m->V; ++v)
    if (poses[v] == nullptr || (rays && rays[v] == nullptr) || (centers && centers[v] == nullptr)) {
      set_error("mpl_forward: view %d pointer is null", v);
      return MPL_ERR_INVALID_ARGUMENT;
    }
  m->launches = 0;
  if (m->profile) { m->prof.clear(); m->ev_used = 0; }
  if (batch == 0) return MPL_OK;
  // Every pose is independent: the batch runs as chunks of at most m->chunk poses, one after the other on the caller's stream
  const int64_t Bc_max = std::min<int64_t>(std::max<int64_t>(batch, 1), m->chunk);
  const size_t need = layout_workspace(m, Bc_max, nullptr).bytes;
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("mpl_forward: workspace has %zu bytes, %zu needed for batch %lld", workspace_bytes, need, (long long)batch);
    return MPL_ERR_WORKSPACE;
  }
  const Workspace w = layout_workspace(m, Bc_max, reinterpret_cast<uint8_t*>(workspace));
  Packed P{m, reinterpret_cast<const uint8_t*>(packed)};
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int out_dim = 3 * m->J;
  // ---- small batches: replay the captured graph of this exact call (same batch and pointers), capture it on first sight ----
  cudaStreamCaptureStatus cap_status = cudaStreamCaptureStatusNone;
  const bool try_graph = m->graph_max_batch > 0 && batch <= m->graph_max_batch && !m->profile &&
                         cudaStreamIsCapturing(s, &cap_status) == cudaSuccess && cap_status == cudaStreamCaptureStatusNone;
  MplModel::GraphKey key;
  if (try_graph) {
    memset(&key, 0, sizeof(key));
    key.batch = batch; key.pose_stride = pose_stride; key.center_stride = center_stride;
    key.packed = packed; key.out = out; key.aux1 = aux1; key.aux2 = aux2; key.workspace = workspace;
    for (int v = 0; v < m->V; ++v) {
      key.in[0][v] = poses[v];
      key.in[1][v] = rays ? rays[v] : nullptr;
      key.in[2][v] = centers ? centers[v] : nullptr;
    }
    for (auto& e : m->graphs)
      if (memcmp(&e.key, &key, sizeof(key)) == 0) {
        e.last_used = ++m->graph_clock;
        MPL_CUDA(cudaGraphLaunch(e.exec, s));
        m->launches = e.launches;
        ++m->graph_hits;
        return MPL_OK;
      }
    if (m->cap_stream == nullptr) MPL_CUDA(cudaStreamCreateWithFlags(&m->cap_stream, cudaStreamNonBlocking));
    MPL_CUDA(cudaStreamBeginCapture(m->cap_stream, cudaStreamCaptureModeThreadLocal));
    s = m->cap_stream;  // nothing executes during capture; the instantiated graph is launched on the caller's stream below
  }
  auto end_capture = [&](int status) -> int {
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(m->cap_stream, &graph);
    if (status != MPL_OK) {
      if (graph) cudaGraphDestroy(graph);
      return status;
    }
    MPL_CUDA(e);
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    MPL_CUDA(ie);
    if (m->graphs.size() >= 16) {  // least recently used entry makes room
      size_t lru = 0;
      for (size_t i = 1; i < m->graphs.size(); ++i)
        if (m->graphs[i].last_used < m->graphs[lru].last_used) lru = i;
      cudaGraphExecDestroy(m->graphs[lru].exec);
      m->graphs.erase(m->graphs.begin() + lru);
    }
    m->graphs.push_back({key, exec, m->launches, ++m->graph_clock});
    ++m->graph_captures;
    MPL_CUDA(cudaGraphLaunch(exec, reinterpret_cast<cudaStream_t>(stream)));
    return MPL_OK;
  };
  for (int64_t b0 = 0; b0 < batch; b0 += Bc_max) {
    const int64_t Bc = std::min<int64_t>(Bc_max, batch - b0);
    const float* pp[kMaxViews];
    const float* rp[kMaxViews];
    const float* cp[kMaxViews];
    for (int v = 0; v < m->V; ++v) {
      pp[v] = poses[v] + b0 * pose_stride;
      rp[v] = rays ? rays[v] + b0 * pose_stride : nullptr;
      cp[v] = centers ? centers[v] + b0 * center_stride : nullptr;
    }
    const int st = forward_chunk(m, P, pp, rays ? rp : nullptr, centers ? cp : nullptr, pose_stride, center_stride,
                                 out + b0 * out_dim, aux1 ? aux1 + b0 * out_dim : nullptr, aux2 ? aux2 + b0 * out_dim : nullptr, Bc,
                                 w, s);
    if (st != MPL_OK) return try_graph ? end_capture(st) : st;
  }
  return try_graph ? end_capture(MPL_OK) : MPL_OK;
  MPL_API_END
}

int mpl_set_graph_batch(MplModel* m, int64_t max_batch) {
  if (m == nullptr || max_batch < 0) {
    set_error("mpl_set_graph_batch: null handle or negative batch");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  m->graph_max_batch = max_batch;
  if (max_batch == 0) {
    for (auto& e : m->graphs) cudaGraphExecDestroy(e.exec);
    m->graphs.clear();
  }
  return MPL_OK;
}

int mpl_graph_stats(const MplModel* m, int64_t* captures, int64_t* replays) {
  if (m == nullptr) return MPL_ERR_INVALID_ARGUMENT;
  if (captures) *captures = m->graph_captures;
  if (replays) *replays = m->graph_hits;
  return MPL_OK;
}

int64_t mpl_last_launch_count(const MplModel* m) { return m ? m->launches : 0; }

int mpl_mpjpe_accumulate(const float* pred, const float* gt, const float* conf3d, int64_t batch, int num_joints,
                         float unit_scale, const float* room_affine, double* acc, mpl_stream_t stream) {
  if (batch == 0 && acc != nullptr) return MPL_OK;
  if (pred == nullptr || gt == nullptr || acc == nullptr || batch < 0 || num_joints < 1) {
    set_error("mpl_mpjpe_accumulate: bad argument");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_mpjpe_accumulate(pred, gt, conf3d, nullptr, 0, batch, num_joints, unit_scale, room_affine, acc,
                                 reinterpret_cast<cudaStream_t>(stream));
}

// the group rules shared by the two grouped entry points (include/mpl_b200.h)
static bool groups_ok(const int32_t* group, int num_groups) {
  return num_groups >= 1 && num_groups <= 65536 && (group != nullptr || num_groups == 1);
}

int mpl_mpjpe_accumulate_grouped(const float* pred, const float* gt, const float* conf3d, const int32_t* group, int num_groups,
                                 int64_t batch, int num_joints, float unit_scale, const float* room_affine, double* acc,
                                 mpl_stream_t stream) {
  if (!groups_ok(group, num_groups) || pred == nullptr || gt == nullptr || acc == nullptr || batch < 0 || num_joints < 1) {
    set_error("mpl_mpjpe_accumulate_grouped: bad argument (num_groups %d, group %s, batch %lld, num_joints %d)", num_groups,
              group ? "set" : "null", (long long)batch, num_joints);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_mpjpe_accumulate(pred, gt, conf3d, group, num_groups, batch, num_joints, unit_scale, room_affine, acc,
                                 reinterpret_cast<cudaStream_t>(stream));
}

int mpl_pmpjpe_accumulate(const float* pred, const float* gt, int64_t batch, int num_joints, float unit_scale,
                          int scaling, int reflection, double* acc, mpl_stream_t stream) {
  if (batch == 0 && acc != nullptr) return MPL_OK;
  if (pred == nullptr || gt == nullptr || acc == nullptr || batch < 0 || num_joints < 1 || reflection < -1 || reflection > 1) {
    set_error("mpl_pmpjpe_accumulate: bad argument");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_pmpjpe_accumulate(pred, gt, nullptr, nullptr, 0, batch, num_joints, unit_scale, scaling != 0, reflection, acc,
                                  reinterpret_cast<cudaStream_t>(stream));
}

int mpl_pmpjpe_accumulate_masked(const float* pred, const float* gt, const float* mask, const int32_t* group, int num_groups,
                                 int64_t batch, int num_joints, float unit_scale, int scaling, int reflection, double* acc,
                                 mpl_stream_t stream) {
  if (!groups_ok(group, num_groups) || pred == nullptr || gt == nullptr || acc == nullptr || batch < 0 || num_joints < 1 ||
      reflection < -1 || reflection > 1) {
    set_error("mpl_pmpjpe_accumulate_masked: bad argument (num_groups %d, group %s, batch %lld, num_joints %d, reflection %d)",
              num_groups, group ? "set" : "null", (long long)batch, num_joints, reflection);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_pmpjpe_accumulate(pred, gt, mask, group, num_groups, batch, num_joints, unit_scale, scaling != 0, reflection,
                                  acc, reinterpret_cast<cudaStream_t>(stream));
}

// calib_stride of the *_strided entry points: 0 (one [V, 18] block for every pose) or >= 18 V (pose b at calib + b * stride)
static bool calib_stride_ok(int64_t calib_stride, int num_views) {
  return calib_stride == 0 || (calib_stride > 0 && calib_stride >= 18 * (int64_t)num_views);
}

int mpl_build_inputs(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints, float* poses,
                     float* rays, float* centers, mpl_stream_t stream) {
  return mpl_build_inputs_strided(pix, calib, 0, batch, num_views, num_joints, poses, rays, centers, stream);
}

int mpl_build_inputs_strided(const float* pix, const double* calib, int64_t calib_stride, int64_t batch, int num_views,
                             int num_joints, float* poses, float* rays, float* centers, mpl_stream_t stream) {
  if (!calib_stride_ok(calib_stride, num_views)) {
    set_error("mpl_build_inputs_strided: bad calib_stride %lld (0, or >= 18 * num_views)", (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (pix == nullptr || calib == nullptr || poses == nullptr || rays == nullptr || centers == nullptr || batch < 0) {
    set_error("mpl_build_inputs_strided: bad argument");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_build_inputs(pix, calib, calib_stride, batch, num_views, num_joints, poses, rays, centers,
                             reinterpret_cast<cudaStream_t>(stream));
}

int mpl_synth_project(uint64_t seed, int64_t start, int64_t batch, int num_views, int num_joints, const double* calib,
                      const double* room, int conf_ones, float* pix, float* target, mpl_stream_t stream) {
  return mpl_synth_project_strided(seed, start, batch, num_views, num_joints, calib, 0, room, conf_ones, pix, target, stream);
}

int mpl_synth_project_strided(uint64_t seed, int64_t start, int64_t batch, int num_views, int num_joints, const double* calib,
                              int64_t calib_stride, const double* room, int conf_ones, float* pix, float* target,
                              mpl_stream_t stream) {
  if (!calib_stride_ok(calib_stride, num_views)) {
    set_error("mpl_synth_project_strided: bad calib_stride %lld (0, or >= 18 * num_views)", (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (calib == nullptr || room == nullptr || pix == nullptr || target == nullptr || batch < 0 || start < 0 || num_views < 1 ||
      num_joints < 1) {
    set_error("mpl_synth_project_strided: bad argument");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_synth_project(seed, start, batch, num_views, num_joints, calib, calib_stride, room, conf_ones, pix, target,
                              reinterpret_cast<cudaStream_t>(stream));
}

int mpl_triangulate(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints, float min_conf,
                    float* points, int32_t* views_used, mpl_stream_t stream) {
  return mpl_triangulate_strided(pix, calib, 0, batch, num_views, num_joints, min_conf, points, views_used, stream);
}

int mpl_triangulate_strided(const float* pix, const double* calib, int64_t calib_stride, int64_t batch, int num_views,
                            int num_joints, float min_conf, float* points, int32_t* views_used, mpl_stream_t stream) {
  if (batch < 0 || num_views < 1 || num_views > kMaxViews || num_joints < 1 || !calib_stride_ok(calib_stride, num_views)) {
    set_error("mpl_triangulate_strided: bad argument (batch %lld, num_views %d, num_joints %d, calib_stride %lld)",
              (long long)batch, num_views, num_joints, (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (pix == nullptr || calib == nullptr || points == nullptr || views_used == nullptr) {
    set_error("mpl_triangulate_strided: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_triangulate(pix, calib, calib_stride, batch, num_views, num_joints, min_conf, points, views_used,
                            reinterpret_cast<cudaStream_t>(stream));
}

int mpl_triangulate_robust(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints,
                           float min_conf, float inlier_px, float* points, int32_t* inliers, mpl_stream_t stream) {
  return mpl_triangulate_robust_strided(pix, calib, 0, batch, num_views, num_joints, min_conf, inlier_px, points, inliers,
                                        stream);
}

int mpl_triangulate_robust_strided(const float* pix, const double* calib, int64_t calib_stride, int64_t batch, int num_views,
                                   int num_joints, float min_conf, float inlier_px, float* points, int32_t* inliers,
                                   mpl_stream_t stream) {
  if (batch < 0 || num_views < 1 || num_views > kMaxViews || num_joints < 1 || !std::isfinite(inlier_px) || !(inlier_px > 0.0f) ||
      !calib_stride_ok(calib_stride, num_views)) {
    set_error("mpl_triangulate_robust_strided: bad argument (batch %lld, num_views %d, num_joints %d, inlier_px %g, "
              "calib_stride %lld)", (long long)batch, num_views, num_joints, (double)inlier_px, (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (pix == nullptr || calib == nullptr || points == nullptr || inliers == nullptr) {
    set_error("mpl_triangulate_robust_strided: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_triangulate_robust(pix, calib, calib_stride, batch, num_views, num_joints, min_conf, inlier_px, points, inliers,
                                   reinterpret_cast<cudaStream_t>(stream));
}

int mpl_triangulate_refine(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints,
                           float min_conf, const int32_t* view_mask, const float* init, int max_iters, float* points,
                           float* reproj_px, mpl_stream_t stream) {
  return mpl_triangulate_refine_strided(pix, calib, 0, batch, num_views, num_joints, min_conf, view_mask, init, max_iters,
                                        points, reproj_px, stream);
}

int mpl_triangulate_refine_strided(const float* pix, const double* calib, int64_t calib_stride, int64_t batch,
                                   int num_views, int num_joints, float min_conf, const int32_t* view_mask,
                                   const float* init, int max_iters, float* points, float* reproj_px,
                                   mpl_stream_t stream) {
  if (batch < 0 || num_views < 1 || num_views > kMaxViews || num_joints < 1 || max_iters < 1 || max_iters > 100 ||
      !calib_stride_ok(calib_stride, num_views)) {
    set_error("mpl_triangulate_refine_strided: bad argument (batch %lld, num_views %d, num_joints %d, max_iters %d, "
              "calib_stride %lld)", (long long)batch, num_views, num_joints, max_iters, (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (pix == nullptr || calib == nullptr || init == nullptr || points == nullptr || reproj_px == nullptr) {
    set_error("mpl_triangulate_refine_strided: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_triangulate_refine(pix, calib, calib_stride, batch, num_views, num_joints, min_conf, view_mask, init,
                                   max_iters, points, reproj_px, reinterpret_cast<cudaStream_t>(stream));
}

int mpl_synth_detector_noise(uint64_t seed, int64_t start, int64_t batch, int num_views, int num_joints, const double* calib,
                             float sigma_px, float p_outlier, float p_miss, float* pix, mpl_stream_t stream) {
  return mpl_synth_detector_noise_strided(seed, start, batch, num_views, num_joints, calib, 0, sigma_px, p_outlier, p_miss, pix,
                                          stream);
}

int mpl_synth_detector_noise_strided(uint64_t seed, int64_t start, int64_t batch, int num_views, int num_joints,
                                     const double* calib, int64_t calib_stride, float sigma_px, float p_outlier, float p_miss,
                                     float* pix, mpl_stream_t stream) {
  // the probabilities' sum in fp64, as the kernel forms it
  if (batch < 0 || start < 0 || num_views < 1 || num_views > kMaxViews || num_joints < 1 || !std::isfinite(sigma_px) ||
      !(sigma_px >= 0.0f) || !(p_outlier >= 0.0f && p_outlier <= 1.0f) || !(p_miss >= 0.0f && p_miss <= 1.0f) ||
      !((double)p_outlier + (double)p_miss <= 1.0) || !calib_stride_ok(calib_stride, num_views)) {
    set_error("mpl_synth_detector_noise_strided: bad argument (batch %lld, start %lld, num_views %d, num_joints %d, "
              "sigma_px %g, p_outlier %g, p_miss %g, calib_stride %lld)", (long long)batch, (long long)start, num_views,
              num_joints, (double)sigma_px, (double)p_outlier, (double)p_miss, (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (calib == nullptr || pix == nullptr) {
    set_error("mpl_synth_detector_noise_strided: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_detector_noise(seed, start, batch, num_views, num_joints, calib, calib_stride, sigma_px, p_outlier, p_miss,
                               pix, reinterpret_cast<cudaStream_t>(stream));
}

// Argument checks shared by mpl_distort_pixels_strided and mpl_undistort_pixels_strided (the distortion passes margins 0).
static int lens_pixels(const char* name, bool undistort, const float* pix_in, float* pix_out, const double* calib,
                       int64_t calib_stride, const double* dist, int64_t dist_stride, double margin_x, double margin_y,
                       int64_t batch, int num_views, int num_joints, mpl_stream_t stream) {
  const bool dist_stride_ok = dist_stride == 0 || (dist_stride > 0 && dist_stride >= 5 * (int64_t)num_views);
  if (batch < 0 || num_views < 1 || num_views > kMaxViews || num_joints < 1 || !calib_stride_ok(calib_stride, num_views) ||
      !dist_stride_ok || !std::isfinite(margin_x) || !(margin_x >= 0.0) || !std::isfinite(margin_y) || !(margin_y >= 0.0)) {
    set_error("%s: bad argument (batch %lld, num_views %d, num_joints %d, calib_stride %lld, dist_stride %lld, margin %g %g)",
              name, (long long)batch, num_views, num_joints, (long long)calib_stride, (long long)dist_stride, margin_x, margin_y);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (pix_in == nullptr || pix_out == nullptr || calib == nullptr || dist == nullptr) {
    set_error("%s: null pointer", name);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_lens_pixels(undistort, pix_in, pix_out, calib, calib_stride, dist, dist_stride, margin_x, margin_y, batch,
                            num_views, num_joints, reinterpret_cast<cudaStream_t>(stream));
}

int mpl_distort_pixels(const float* pix_in, float* pix_out, const double* calib, const double* dist, int64_t batch,
                       int num_views, int num_joints, mpl_stream_t stream) {
  return mpl_distort_pixels_strided(pix_in, pix_out, calib, 0, dist, 0, batch, num_views, num_joints, stream);
}

int mpl_distort_pixels_strided(const float* pix_in, float* pix_out, const double* calib, int64_t calib_stride,
                               const double* dist, int64_t dist_stride, int64_t batch, int num_views, int num_joints,
                               mpl_stream_t stream) {
  return lens_pixels("mpl_distort_pixels_strided", false, pix_in, pix_out, calib, calib_stride, dist, dist_stride, 0.0, 0.0,
                     batch, num_views, num_joints, stream);
}

int mpl_undistort_pixels(const float* pix_in, float* pix_out, const double* calib, const double* dist, double margin_x,
                         double margin_y, int64_t batch, int num_views, int num_joints, mpl_stream_t stream) {
  return mpl_undistort_pixels_strided(pix_in, pix_out, calib, 0, dist, 0, margin_x, margin_y, batch, num_views, num_joints,
                                      stream);
}

int mpl_undistort_pixels_strided(const float* pix_in, float* pix_out, const double* calib, int64_t calib_stride,
                                 const double* dist, int64_t dist_stride, double margin_x, double margin_y, int64_t batch,
                                 int num_views, int num_joints, mpl_stream_t stream) {
  return lens_pixels("mpl_undistort_pixels_strided", true, pix_in, pix_out, calib, calib_stride, dist, dist_stride, margin_x,
                     margin_y, batch, num_views, num_joints, stream);
}

int mpl_synth_cameras(uint64_t seed, int64_t start, int64_t batch, int num_views, double f0, double w, double h,
                      const double* room, double* calib_out, mpl_stream_t stream) {
  if (batch < 0 || start < 0 || num_views < 1 || num_views > kMaxViews || !std::isfinite(f0) || !(f0 > 0.0) ||
      !std::isfinite(w) || !(w > 1.0) || !std::isfinite(h) || !(h > 1.0)) {
    set_error("mpl_synth_cameras: bad argument (batch %lld, start %lld, num_views %d, f0 %g, w %g, h %g)", (long long)batch,
              (long long)start, num_views, f0, w, h);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (room == nullptr || calib_out == nullptr) {
    set_error("mpl_synth_cameras: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_synth_cameras(seed, start, batch, num_views, f0, w, h, room, calib_out, reinterpret_cast<cudaStream_t>(stream));
}

int mpl_synth_calib_noise(uint64_t seed, int64_t start, int64_t batch, int num_views, const double* calib,
                          int64_t calib_stride, double sigma_rot, double sigma_pos, double* calib_out, mpl_stream_t stream) {
  if (num_views < 1 || num_views > kMaxViews || start < 0 || !std::isfinite(sigma_rot) || !(sigma_rot >= 0.0) ||
      !std::isfinite(sigma_pos) || !(sigma_pos >= 0.0) || !calib_stride_ok(calib_stride, num_views) || batch < 0) {
    set_error("mpl_synth_calib_noise: bad argument (batch %lld, start %lld, num_views %d, sigma_rot %g, sigma_pos %g, "
              "calib_stride %lld)", (long long)batch, (long long)start, num_views, sigma_rot, sigma_pos,
              (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (batch == 0) return MPL_OK;
  if (calib == nullptr || calib_out == nullptr) {
    set_error("mpl_synth_calib_noise: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (calib_out == calib && calib_stride != 18 * (int64_t)num_views) {
    set_error("mpl_synth_calib_noise: calib_out may be calib only with calib_stride 18 * num_views");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_synth_calib_noise(seed, start, batch, num_views, calib, calib_stride, sigma_rot, sigma_pos, calib_out,
                                  reinterpret_cast<cudaStream_t>(stream));
}

size_t mpl_calibrate_rig_workspace_bytes(int64_t batch, int num_views, int num_joints) {
  if (batch < 1 || num_views < 2 || num_views > kMaxViews || num_joints < 1) return 0;
  return rig_workspace_bytes(batch, num_views, num_joints);
}

int mpl_calibrate_rig(const float* pix, const double* calib, int64_t batch, int num_views, int num_joints, float min_conf,
                      const int32_t* view_mask, const float* init, double sigma_px, double sigma_rot, double sigma_pos,
                      int max_iters, double* calib_out, float* points, double* report, void* workspace,
                      size_t workspace_bytes, mpl_stream_t stream) {
  auto sigma_ok = [](double s) { return std::isfinite(s) && s > 0.0; };
  if (num_views < 2 || num_views > kMaxViews || num_joints < 1 || batch < 1 || !sigma_ok(sigma_px) || !sigma_ok(sigma_rot) ||
      !sigma_ok(sigma_pos) || max_iters < 1 || max_iters > 100) {
    set_error("mpl_calibrate_rig: bad argument (batch %lld, num_views %d, num_joints %d, sigma_px %g, sigma_rot %g, "
              "sigma_pos %g, max_iters %d)", (long long)batch, num_views, num_joints, sigma_px, sigma_rot, sigma_pos,
              max_iters);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (pix == nullptr || calib == nullptr || init == nullptr || calib_out == nullptr || report == nullptr ||
      workspace == nullptr) {
    set_error("mpl_calibrate_rig: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  const size_t need = rig_workspace_bytes(batch, num_views, num_joints);
  if (workspace_bytes < need) {
    set_error("mpl_calibrate_rig: workspace has %zu bytes, %zu needed", workspace_bytes, need);
    return MPL_ERR_WORKSPACE;
  }
  return launch_calibrate_rig(pix, calib, batch, num_views, num_joints, min_conf, view_mask, init, sigma_px, sigma_rot,
                              sigma_pos, max_iters, calib_out, points, report, workspace,
                              reinterpret_cast<cudaStream_t>(stream));
}

// Shape rules of the association entry points: V views, P slots per view, J joints (include/mpl_b200.h).
static bool people_shape_ok(int P, int V, int J, int min_views) {
  return V >= min_views && V <= kMaxViews && P >= 1 && P * V <= 128 && J >= 1;
}

int mpl_synth_people(uint64_t seed, int64_t start, int64_t frames, int people, int num_views, int num_joints, const float* pix,
                     float* scene, int32_t* perm, mpl_stream_t stream) {
  if (frames < 0 || start < 0 || !people_shape_ok(people, num_views, num_joints, 1)) {
    set_error("mpl_synth_people: bad argument (frames %lld, start %lld, people %d, num_views %d, num_joints %d)",
              (long long)frames, (long long)start, people, num_views, num_joints);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (frames == 0) return MPL_OK;
  if (pix == nullptr || scene == nullptr || perm == nullptr || (const void*)pix == (const void*)scene) {
    set_error("mpl_synth_people: null pointer, or scene == pix");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_synth_people(seed, start, frames, people, num_views, num_joints, pix, scene, perm,
                             reinterpret_cast<cudaStream_t>(stream));
}

int mpl_associate_people(const float* scene, const double* calib, int64_t frames, int people, int num_views, int num_joints,
                         float min_conf, int min_joints, double max_dist, int max_people, int32_t* members, int32_t* labels,
                         int32_t* num_people, mpl_stream_t stream) {
  return mpl_associate_people_strided(scene, calib, 0, frames, people, num_views, num_joints, min_conf, min_joints, max_dist,
                                      max_people, members, labels, num_people, stream);
}

int mpl_associate_people_strided(const float* scene, const double* calib, int64_t calib_stride, int64_t frames, int people,
                                 int num_views, int num_joints, float min_conf, int min_joints, double max_dist,
                                 int max_people, int32_t* members, int32_t* labels, int32_t* num_people,
                                 mpl_stream_t stream) {
  if (frames < 0 || !people_shape_ok(people, num_views, num_joints, 2) || num_joints > 32 || min_joints < 1 ||
      min_joints > num_joints || !std::isfinite(max_dist) || !(max_dist > 0.0) || max_people < 1 ||
      !calib_stride_ok(calib_stride, num_views)) {
    set_error("mpl_associate_people_strided: bad argument (frames %lld, people %d, num_views %d, num_joints %d, min_joints %d, "
              "max_dist %g, K %d, calib_stride %lld)", (long long)frames, people, num_views, num_joints, min_joints, max_dist,
              max_people, (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (frames == 0) return MPL_OK;
  if (scene == nullptr || calib == nullptr || members == nullptr || labels == nullptr || num_people == nullptr) {
    set_error("mpl_associate_people_strided: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_associate_people(scene, calib, calib_stride, frames, people, num_views, num_joints, min_conf, min_joints,
                                 max_dist, max_people, members, labels, num_people, reinterpret_cast<cudaStream_t>(stream));
}

int mpl_gather_people(const float* scene, const int32_t* members, int64_t frames, int people, int max_people, int num_views,
                      int num_joints, float* out, mpl_stream_t stream) {
  if (frames < 0 || people < 1 || max_people < 1 || num_views < 1 || num_views > kMaxViews || num_joints < 1) {
    set_error("mpl_gather_people: bad argument (frames %lld, people %d, K %d, num_views %d, num_joints %d)", (long long)frames,
              people, max_people, num_views, num_joints);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (frames == 0) return MPL_OK;
  if (scene == nullptr || members == nullptr || out == nullptr) {
    set_error("mpl_gather_people: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_gather_people(scene, members, frames, people, max_people, num_views, num_joints, out,
                              reinterpret_cast<cudaStream_t>(stream));
}

int mpl_association_score(const int32_t* members, const int32_t* labels, const int32_t* perm, int64_t frames, int people,
                          int max_people, int num_views, int32_t* owner, double* acc, mpl_stream_t stream) {
  if (frames < 0 || !people_shape_ok(people, num_views, 1, 1) || max_people < 1) {
    set_error("mpl_association_score: bad argument (frames %lld, people %d, K %d, num_views %d)", (long long)frames, people,
              max_people, num_views);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (frames == 0) return MPL_OK;
  if (members == nullptr || labels == nullptr || perm == nullptr || owner == nullptr || acc == nullptr) {
    set_error("mpl_association_score: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_association_score(members, labels, perm, frames, people, max_people, num_views, owner, acc,
                                  reinterpret_cast<cudaStream_t>(stream));
}

// Shape rules of the tracking entry points (include/mpl_b200.h): K rows per frame, J joints, max_tracks track slots.
static bool track_shape_ok(int K, int J, int max_tracks) {
  return K >= 1 && K <= 64 && J >= 1 && J <= 32 && max_tracks >= 1 && max_tracks <= 128;
}

int mpl_synth_motion(uint64_t seed, int64_t start, int64_t sequences, int frames, int people, int num_views, int num_joints,
                     const double* calib, int64_t calib_stride, const double* room, double fps, int conf_ones, float* pix,
                     float* target, mpl_stream_t stream) {
  if (sequences < 0 || start < 0 || frames < 1 || people < 1 || num_views < 1 || num_views > kMaxViews || num_joints < 1 ||
      !std::isfinite(fps) || !(fps > 0.0) || !calib_stride_ok(calib_stride, num_views)) {
    set_error("mpl_synth_motion: bad argument (sequences %lld, start %lld, frames %d, people %d, num_views %d, num_joints %d, "
              "fps %g, calib_stride %lld)", (long long)sequences, (long long)start, frames, people, num_views, num_joints, fps,
              (long long)calib_stride);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (sequences == 0) return MPL_OK;
  if (calib == nullptr || room == nullptr || pix == nullptr || target == nullptr) {
    set_error("mpl_synth_motion: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_synth_motion(seed, start, sequences, frames, people, num_views, num_joints, calib, calib_stride, room, fps,
                             conf_ones, pix, target, reinterpret_cast<cudaStream_t>(stream));
}

size_t mpl_track_state_bytes(int max_tracks, int num_joints) {
  return track_shape_ok(1, num_joints, max_tracks) ? track_state_bytes(max_tracks, num_joints) : 0;
}

int mpl_track_people(const float* points, const float* joint_mask, int64_t sequences, int64_t frames, int max_rows,
                     int num_joints, int min_joints, double max_dist, int max_age, int max_tracks, void* state,
                     int32_t* track_id, mpl_stream_t stream) {
  if (sequences < 0 || frames < 0 || frames > INT32_MAX || !track_shape_ok(max_rows, num_joints, max_tracks) ||
      min_joints < 1 || min_joints > num_joints || !std::isfinite(max_dist) || !(max_dist > 0.0) || max_age < 0) {
    set_error("mpl_track_people: bad argument (sequences %lld, frames %lld, K %d, num_joints %d, min_joints %d, max_dist %g, "
              "max_age %d, max_tracks %d)", (long long)sequences, (long long)frames, max_rows, num_joints, min_joints, max_dist,
              max_age, max_tracks);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (sequences == 0 || frames == 0) return MPL_OK;
  if (points == nullptr || state == nullptr || track_id == nullptr || (reinterpret_cast<uintptr_t>(state) & 3u) != 0) {
    set_error("mpl_track_people: null pointer, or state not 4-byte aligned");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_track_people(points, joint_mask, sequences, frames, max_rows, num_joints, min_joints, max_dist, max_age,
                             max_tracks, state, track_id, reinterpret_cast<cudaStream_t>(stream));
}

int mpl_tracking_score(const int32_t* track_id, const int32_t* owner, int64_t sequences, int64_t frames, int max_rows,
                       int people, double* acc, mpl_stream_t stream) {
  if (sequences < 0 || frames < 0 || frames > INT32_MAX || max_rows < 1 || people < 1) {
    set_error("mpl_tracking_score: bad argument (sequences %lld, frames %lld, K %d, people %d)", (long long)sequences,
              (long long)frames, max_rows, people);
    return MPL_ERR_INVALID_ARGUMENT;
  }
  if (sequences == 0 || frames == 0) return MPL_OK;
  if (track_id == nullptr || owner == nullptr || acc == nullptr) {
    set_error("mpl_tracking_score: null pointer");
    return MPL_ERR_INVALID_ARGUMENT;
  }
  return launch_tracking_score(track_id, owner, sequences, frames, max_rows, people, acc,
                               reinterpret_cast<cudaStream_t>(stream));
}

int mpl_test_gemm(const void* A, const void* W, const float* bias, void* Y, int64_t M, int N, int K, int dtype, int epilogue,
                  int out_fp32, mpl_stream_t stream) {
  MPL_API_BEGIN
  return launch_gemm_tcgen05(A, W, bias, Y, M, N, K, dtype, epilogue, out_fp32, reinterpret_cast<cudaStream_t>(stream));
  MPL_API_END
}

/* The LayerNorm-fused epilogues of the same kernel in isolation (tests/test_gemm_ln_gpu.py). */
int mpl_test_gemm_ln(const void* A, const void* W, const float* bias, void* Y, int64_t M, int N, int K, int epilogue,
                     const float* colsum, const void* stats_in, int slots_in, void* stats_out, void* x_lo, float eps,
                     int ab_fp16, int out_fp16, mpl_stream_t stream) {
  MPL_API_BEGIN
  GemmLnArgs a{};
  a.colsum = colsum;
  a.stats_in = stats_in;
  a.slots_in = slots_in;
  a.stats_out = stats_out;
  a.x_lo = x_lo;
  a.eps = eps;
  a.ab_fp16 = ab_fp16;
  a.out_fp16 = out_fp16;
  return launch_gemm_tcgen05(A, W, bias, Y, M, N, K, MPL_PREC_BF16, epilogue, 0, reinterpret_cast<cudaStream_t>(stream), &a);
  MPL_API_END
}
int mpl_test_gemm_ln_slots(int N) { return gemm_ln_slots(N); }

int mpl_test_gemm_emit_pitch(const void* A, const void* W, const float* bias, void* Y, int64_t M, int N, int K, void* stats_out,
                             void* x_lo, int ab_fp16, int ldy, mpl_stream_t stream) {
  MPL_API_BEGIN
  GemmLnArgs a{};
  a.stats_out = stats_out;
  a.x_lo = x_lo;
  a.ab_fp16 = ab_fp16;
  a.ldy = ldy;
  return launch_gemm_tcgen05(A, W, bias, Y, M, N, K, MPL_PREC_BF16, EPI_RESIDUAL_EMIT, 0, reinterpret_cast<cudaStream_t>(stream), &a);
  MPL_API_END
}

/* The fused QKV + cross-view attention kernel in isolation.  scratch: (H * 416 * D) bf16 + 2 * (H * 416) floats, 256-aligned. */
int mpl_test_qkv_attn(const void* xb, const float* W, const float* bias, const float* gamma, const float* beta,
                      const void* stats, int slots, float eps, float scale, void* att, int64_t M, int D, int H, int V,
                      void* scratch, size_t scratch_bytes, mpl_stream_t stream) {
  MPL_API_BEGIN
  if (!qkv_attn_supports(D, H, V)) {
    set_error("mpl_test_qkv_attn: unsupported shape (D=%d H=%d V=%d)", D, H, V);
    return MPL_ERR_UNSUPPORTED;
  }
  const size_t wbytes = align_up(qkv_attn_weight_elems(D, H) * 2, 256), vbytes = align_up((size_t)qkv_attn_vec_len(D, H) * 4, 256);
  if (scratch == nullptr || scratch_bytes < wbytes + 2 * vbytes) {
    set_error("mpl_test_qkv_attn: scratch has %zu bytes, %zu needed", scratch_bytes, wbytes + 2 * vbytes);
    return MPL_ERR_WORKSPACE;
  }
  uint8_t* sb = reinterpret_cast<uint8_t*>(scratch);
  float* cs = reinterpret_cast<float*>(sb + wbytes);
  float* bf = reinterpret_cast<float*>(sb + wbytes + vbytes);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  MPL_TRY(launch_qkv_attn_pack(W, bias, gamma, beta, sb, cs, bf, H, D, scale, s));
  return launch_qkv_attn(xb, sb, bf, cs, stats, slots, eps, att, M, D, H, V, s);
  MPL_API_END
}

}  // extern "C"
