// Whole-model entry points: spektral.models.GeneralGNN.__call__ and the reverse-mode
// gradient the reference takes with tf.GradientTape (src/scripts/gcn.py:320 model,
// :333-337 train step, :351 inference; upstream call graph in SURVEY.md §3.1, §8 a2).
//
//   out = pre(x)                                   MLP: [Dense -> BN -> PReLU] x P
//   for k in 1..L:  z = A . prelu(bn(out.W_k + b_k));  out = concat([z, out])
//   out = pool(out, i);  out = post(out)          MLP, last layer Dense -> BN -> softmax | sigmoid | linear
//   pool: segment_sum ('sum'), segment_mean ('avg'), attention-weighted sum ('attn_sum', one extra trainable vector
//   pool.attn_kernel [Wc] after the last post block), or none (node-level output)
//
// HBM layout.  The 'cat' skip connection is materialised ONCE: a single [N, H*(L+1)] buffer
// `cat`; Keras concatenates [z, out] (new block first), so pre() writes the LAST H columns
// and layer k writes the H columns just before the current prefix — layer k's GEMM input
// is the trailing k*H columns as a strided view (ld = H*(L+1)).  No ConcatV2 copies.  Per
// dense block only the pre-BatchNorm output h is saved for the backward; BN+PReLU are
// recomputed (fused into the aggregation's load in the conv blocks).  In the backward the
// pre-BatchNorm gradients dh_k of the L conv blocks are kept side by side in dhcat[N, H*L]:
// the gradient of one H-wide block of `cat` is then ONE long-K GEMM over all its consumers
// (trailing columns of dhcat x the matching row blocks of their kernels) with the pooled
// gradient broadcast fused into the epilogue - no read-modify-write of a concat-wide buffer.
// connectivity = 'sum' (out = z + out, Keras Add) and None (out = z) keep every layer H wide: the L+1 node
// embeddings out_0..out_L live as L+1 separate [N, H] slabs of the same `cat` allocation (each is the GEMM input of the
// next layer and is needed again for its weight gradient), the skip operand is added in the aggregation's epilogue, and
// the backward carries ONE running gradient g[N, H] = dLoss/d(out_k) that the input-gradient GEMM accumulates into.
// The caller owns the workspace; nothing is allocated here.
#include <cmath>
#include <vector>

#include "common.cuh"
#include "dropout.cuh"
#include "prep.cuh"

namespace gcs {

// linear.cu
int dense_dx_concat(const float* dh, int64_t ld, const float* const* W, const int* row_off, int n_blocks, int Hred,
                    int Nout, const float* rowbias, int64_t ld_rowbias, const int64_t* seg, const int32_t* graph_ptr,
                    int n_graphs, float* C, int64_t ldc, int64_t M, int accumulate, void* workspace,
                    int64_t workspace_bytes, cudaStream_t st);

int linear_fwd_fused(const float* A, int64_t lda, const float* W, const float* bias, const float* scale,
                     const float* shift, const float* alpha, float* C, int64_t ldc, int64_t M, int K, int N,
                     void* workspace, int64_t workspace_bytes, float* amax_out, float* stats_part, cudaStream_t st,
                     int* used);
int bn_stats_from_partials(const float* part, int64_t M, int C, float* mean, float* var, void* workspace,
                           int64_t workspace_bytes, gcs_stream stream);
namespace tc { int amax_merge(float* cell, const float* other, cudaStream_t st); }
int bn_prelu_fwd(const float* h, int64_t ldh, const float* scale, const float* shift, const float* alpha, float* out,
                 int64_t ldo, int64_t M, int32_t C, const Dropout* drop, gcs_stream stream);   // bn.cu
int bn_prelu_bwd(const float* da, int64_t ldda, const float* h, int64_t ldh, const float* mean, const float* var,
                 const float* gamma, const float* beta, const float* alpha, float eps, float* dh, int64_t lddh,
                 float* dgamma, float* dbeta, float* dalpha, float* dbias, int64_t M, int32_t C, void* workspace,
                 int64_t workspace_bytes, const Dropout* drop, gcs_stream stream);
int segment_rows_div_count(float* D, int64_t ld, const int32_t* graph_ptr, int n_graphs, int W, gcs_stream stream);   // pool.cu

enum { kPoolNone = 0, kPoolSum = 1, kPoolAvg = 2, kPoolAttnSum = 3 };

struct BlockDesc {
  int k_in, m_out;
  bool has_alpha;
  int64_t off;       // kernel offset in the trainable buffer
  int64_t stat_off;  // moving_mean offset in the state buffer
  int64_t kernel() const { return off; }
  int64_t bias() const { return off + static_cast<int64_t>(k_in) * m_out; }
  int64_t gamma() const { return bias() + m_out; }
  int64_t beta() const { return gamma() + m_out; }
  int64_t alpha() const { return beta() + m_out; }
  int64_t count() const { return static_cast<int64_t>(k_in) * m_out + (has_alpha ? 4 : 3) * m_out; }
};

// Same arithmetic as gcn-string_b200/params.py:block_specs.
static void build_blocks(const gcs_model_config& c, std::vector<BlockDesc>& out) {
  out.clear();
  int64_t off = 0, soff = 0;
  auto push = [&](int k_in, int m_out, bool has_alpha) {
    BlockDesc b{k_in, m_out, has_alpha, off, soff};
    out.push_back(b);
    off += b.count();
    soff += 2 * m_out;
  };
  int k = c.in_features;
  for (int j = 0; j < c.pre_process; ++j) { push(k, c.hidden, true); k = c.hidden; }
  const bool cat = c.connectivity == 1;
  for (int j = 0; j < c.message_passing; ++j) push(cat ? c.hidden * (j + 1) : c.hidden, c.hidden, true);
  k = cat ? c.hidden * (c.message_passing + 1) : c.hidden;
  for (int j = 0; j < c.post_process; ++j) {
    const bool last = j == c.post_process - 1;
    push(k, last ? c.output : c.hidden, !last);
    k = c.hidden;
  }
}

// The dropout of one training step (dropout.cuh): threshold and scale from the rate in double, here and nowhere else.
// A rate below 2^-32 has threshold 0 and scale 1.0f: every element is kept unscaled, and the rate-0 kernels run.
Dropout make_dropout(float rate, uint64_t seed, uint64_t step, int block) {
  const double t = std::floor(static_cast<double>(rate) * 4294967296.0);
  Dropout d;
  d.threshold = static_cast<uint32_t>(t < 4294967295.0 ? t : 4294967295.0);
  d.scale = static_cast<float>(1.0 / (1.0 - static_cast<double>(rate)));
  d.seed = seed;
  d.step = static_cast<uint32_t>(step);
  d.block = block;
  return d;
}

// The dropout of one training-mode call (block index filled in per block); threshold 0 without one, and in inference.
static int step_dropout(const gcs_dropout* d, bool training, Dropout* out) {
  *out = Dropout{};
  if (!d) return GCS_OK;
  if (!(d->rate >= 0.f && d->rate < 1.f))
    return fail(GCS_ERR_INVALID_ARGUMENT, "dropout: rate must be in [0, 1), got %g", static_cast<double>(d->rate));
  if (training) *out = make_dropout(d->rate, d->seed, d->step, 0);
  return GCS_OK;
}

static Dropout block_dropout(Dropout d, int bi) {
  d.block = bi;
  return d;
}

static int check_config(const gcs_model_config* c) {
  if (!c) return fail(GCS_ERR_INVALID_ARGUMENT, "model config is NULL");
  if (c->in_features < 1 || c->output < 1 || c->hidden < 1)
    return fail(GCS_ERR_INVALID_ARGUMENT, "model config: feature widths must be positive");
  if (c->message_passing < 1 || c->pre_process < 1 || c->post_process < 1)
    return fail(GCS_ERR_UNSUPPORTED, "model config: pre_process, message_passing, post_process must be >= 1");
  if (c->connectivity < 0 || c->connectivity > 2)
    return fail(GCS_ERR_INVALID_ARGUMENT, "model config: connectivity must be 0 (None), 1 ('cat') or 2 ('sum')");
  if (c->pool < kPoolNone || c->pool > kPoolAttnSum)
    return fail(GCS_ERR_UNSUPPORTED, "model config: pool must be 0 (None), 1 ('sum'), 2 ('avg') or 3 ('attn_sum')");
  if (c->final_activation < 0 || c->final_activation > 2)
    return fail(GCS_ERR_UNSUPPORTED, "model config: final activation must be 0 (linear), 1 (softmax) or 2 (sigmoid)");
  if (c->aggregate < 0 || c->aggregate > 2)
    return fail(GCS_ERR_INVALID_ARGUMENT, "model config: aggregate must be 0 ('sum'), 1 ('mean') or 2 ('max')");
  if (c->aggregate == 2 && c->connectivity == 2)
    return fail(GCS_ERR_UNSUPPORTED, "model config: aggregate='max' with connectivity='sum' is not built (the backward needs the "
                                     "aggregation's own output, which the skip connection overwrites)");
  if (c->final_activation == 1 && c->output > 64)
    return fail(GCS_ERR_UNSUPPORTED, "model config: softmax over more than 64 classes is not built");
  if (c->loss < 0 || c->loss > 3)
    return fail(GCS_ERR_INVALID_ARGUMENT, "model config: loss must be 0 (the head's own), 1 (MSE), 2 (MAE) or 3 (Huber)");
  if (c->loss != 0 && c->final_activation != 0)
    return fail(GCS_ERR_UNSUPPORTED, "model config: the regression losses need a linear head (final_activation = 0)");
  if (c->loss == 3 && !(std::isfinite(c->huber_delta) && c->huber_delta > 0.f))
    return fail(GCS_ERR_INVALID_ARGUMENT, "model config: huber_delta must be finite and > 0, got %g",
                static_cast<double>(c->huber_delta));
  return GCS_OK;
}

#define GCS_TIMED(label, call)                 \
  do {                                         \
    ::gcs::ScopedOpTimer timer__(label, st);   \
    GCS_TRY(call);                             \
  } while (0)

// Bump allocator over the caller's workspace; with base == nullptr it only measures.
struct Arena {
  char* base;
  int64_t used = 0;
  explicit Arena(void* b) : base(static_cast<char*>(b)) {}
  template <typename T>
  T* take(int64_t count) {
    const int64_t bytes = round_up(count * static_cast<int64_t>(sizeof(T)), 256);
    T* p = base ? reinterpret_cast<T*>(base + used) : nullptr;
    used += bytes;
    return p;
  }
};

struct Plan {
  std::vector<BlockDesc> blocks;
  int P, L, Q, H, Wc, C;
  int64_t N, rows_post;
  int B;
  // forward
  float* cat = nullptr;
  std::vector<float*> h;        // pre-BN outputs of the node-level blocks (P + L)
  std::vector<float*> act;      // materialised activations of pre blocks 0..P-2
  std::vector<float*> stat;     // per block: mean | var | scale | shift  (4 * m_out)
  float* pooled = nullptr;      // [B, Wc] (unused when pool == 0)
  int64_t attn_off = 0;         // 'attn_sum': offset of pool.attn_kernel [Wc] in the trainable buffer (after the blocks)
  int64_t n_params = 0;         // floats in the trainable buffer
  float* scores = nullptr;      // 'attn_sum', training: [N] attention scores s_n
  float* gstats = nullptr;      // 'attn_sum', training: [B][2] {max_g, softmax denominator}
  void* attn_ws = nullptr;      // 'attn_sum': partials of the split graphs
  int64_t attn_ws_bytes = 0;
  std::vector<float*> post_h;   // [rows_post, m_out]
  std::vector<float*> post_a;   // [rows_post, H], post blocks 0..Q-2
  float* logits = nullptr;      // [rows_post, C]
  void* bn_ws = nullptr;
  int64_t bn_ws_bytes = 0;
  void* lin_ws = nullptr;       // split weights of the tensor-core GEMM in flight
  int64_t lin_ws_bytes = 0;
  void* loss_ws = nullptr;      // partials of the head's loss (head_loss_workspace_bytes)
  int64_t loss_ws_bytes = 0;
  // backward
  float* gcat = nullptr;        // [N, Wc]  without pooling (node-level output) and for 'attn_sum': dLoss/d(emb(L)) in full
  float* dhcat = nullptr;       // [N, H*L] dh of the conv blocks, block k at columns [kH, (k+1)H)
  float* tmp_a = nullptr;       // [N, H]
  float* tmp_b = nullptr;       // [N, H]
  float* tmp_c = nullptr;       // [N, H]   gradient of one block of cat
  float* dlogits = nullptr;     // [rows_post, C]
  float* dpost = nullptr;       // [rows_post, max(H, C)]  dh of a post block
  float* dpost_in = nullptr;    // [rows_post, H]          gradient w.r.t. a post activation
  float* dpooled = nullptr;     // [B, Wc]
  void* lw_ws = nullptr;
  int64_t lw_ws_bytes = 0;
  void* prep_ws = nullptr;      // fp16-split weights of every tensor-core GEMM of the step (prepare_step_weights)
  int64_t prep_ws_bytes = 0;
  float* amax = nullptr;        // [0] running |max| of the node-level activations, [1] of the pre-BatchNorm gradients dh
  float* stat_part = nullptr;   // [ceil(N/32)][H][2] {sum, sum of squares} per 32-row group, left by the GEMM epilogue
};

// Sets the thread's AmaxSink for the calls inside a scope (see common.cuh: feeds the fp16 tensor-core GEMMs).
struct AmaxScope {
  AmaxSink saved;
  AmaxScope(float* produce, const float* consume, const float* consume_act = nullptr) : saved(amax_sink()) {
    amax_sink().produce = produce;
    amax_sink().consume = consume;
    amax_sink().consume_act = consume_act;
  }
  ~AmaxScope() { amax_sink() = saved; }
};

// The tensor-core GEMMs of one training step whose weight operand can be split ahead of time, in the shapes and under
// the keys run_forward / run_backward will ask for (linear.cu: find_prepared): the dense transform of every node-level
// block but the first (kind 0), the concatenated input-gradient GEMMs of the 'cat' layout (kind 1), the plain
// input-gradient GEMMs of the pre-MLP and of the 'sum' / None layouts (kind 2).  Returns the bytes they need; with
// base != NULL fills the split jobs and the lookup table.  A GEMM that is not listed (or whose wrapper decides against
// the fp16 path) prepares its own operand as before.
static int64_t list_step_weights(const gcs_model_config& c, const Plan& p, const float* params, char* base,
                                 tc::SplitJobs* jobs, PreparedTable* table) {
  const int H = p.H, L = p.L, P = p.P;
  int64_t used = 0;
  int n_jobs = 0, n_ent = 0;
  auto region = [&](int kred, int nout) { const int64_t at = used; used += round_up(tc::f16_workspace_bytes(kred, nout), 256); return at; };
  auto add_entry = [&](int kind, const float* w, int kred, int nout, int64_t at) {
    if (table) table->e[n_ent] = PreparedWeights{kind, w, kred, nout, base + at};
    ++n_ent;
  };
  auto add_job = [&](const float* W, int rows, int cols, int transpose, int64_t ldo, int64_t at, int64_t half_off, int kred, int nout) {
    if (jobs) {
      char* ws = base + at;
      jobs->j[n_jobs] = tc::SplitJob{W, rows, cols, cols, transpose, ldo, ws + 2 * half_off, ws + 2LL * kred * nout + 2 * half_off,
                                     tc::f16_cells(ws, kred, nout)};
    }
    ++n_jobs;
  };
  auto room = [&](int more) { return n_jobs + more <= tc::kMaxSplitJobs && n_ent < tc::kMaxSplitJobs; };
  if (H % 64 != 0) return 0;
  for (int bi = 1; bi < P + L; ++bi) {                          // forward: h = in . W, W [k_in, H] -> Bt [H][k_in]
    const BlockDesc& b = p.blocks[bi];
    if (b.k_in % 64 != 0 || b.m_out != H || !room(1)) continue;
    const float* W = params + b.kernel();
    const int64_t at = region(b.k_in, H);
    add_entry(0, W, b.k_in, H, at);
    add_job(W, b.k_in, H, 1, b.k_in, at, 0, b.k_in, H);
  }
  if (c.connectivity == 1) {
    // dLoss/d(block k of cat) = sum over the later layers' dh . W[rows of block k]^T: one long-K GEMM per block
    for (int k = L - 2; k >= -1; --k) {                         // k = -1: the pre-MLP output block, read by all L layers
      const int nb = L - 1 - k;
      if (nb <= 0 || !room(nb)) continue;
      const int kred = nb * H;
      const int64_t at = region(kred, H);
      for (int q = 0; q < nb; ++q) {
        const int kp = k + 1 + q;
        const float* W = params + p.blocks[P + kp].kernel() + static_cast<int64_t>(kp - 1 - k) * H * H;
        if (q == 0) add_entry(1, W, kred, H, at);
        add_job(W, H, H, 0, kred, at, static_cast<int64_t>(q) * H, kred, H);
      }
    }
  }
  for (int bi = P + L - 1; bi >= 1; --bi) {                     // plain input gradient: din = dh . W^T, W [k_in, m_out] as stored
    const bool conv = bi >= P;
    if (conv && c.connectivity == 1) continue;
    const BlockDesc& b = p.blocks[bi];
    if (b.m_out % 64 != 0 || !room(1)) continue;
    const float* W = params + b.kernel();
    const int64_t at = region(b.m_out, b.k_in);
    add_entry(2, W, b.m_out, b.k_in, at);
    add_job(W, b.k_in, b.m_out, 0, b.m_out, at, 0, b.m_out, b.k_in);
  }
  if (jobs) jobs->n = n_jobs;
  if (table) table->n = n_ent;
  return used;
}

// Splits every listed weight operand in two launches (+ one memset of the cells) at the start of a training step; the
// table stays valid until the parameters change (the optimizer step after the backward).
static int prepare_step_weights(const gcs_model_config& c, const Plan& p, const float* params, PreparedTable* table,
                                gcs_stream st) {
  table->n = 0;
  if (!p.prep_ws || p.prep_ws_bytes <= 0 || tc::f16_mode() != 1) return GCS_OK;
  tc::SplitJobs jobs;
  jobs.n = 0;
  list_step_weights(c, p, params, static_cast<char*>(p.prep_ws), &jobs, table);
  GCS_CUDA(cudaMemsetAsync(p.prep_ws, 0, p.prep_ws_bytes, as_stream(st)));
  return tc::split_f16_multi(jobs, as_stream(st));
}

// Workspace of head_loss on [rows, C] logits; the regression partials do not depend on c.loss.  With sample weights
// (GCS_WORKSPACE_SAMPLE_WEIGHTS) the larger of the weighted and the unweighted partials, so that such a plan also serves
// an unweighted step.
static int64_t head_loss_workspace_bytes(const gcs_model_config& c, int64_t rows, int C, int flags = 0) {
  if (flags & GCS_WORKSPACE_SAMPLE_WEIGHTS) {
    const int64_t w = gcs_weighted_loss_workspace_bytes(c.final_activation, rows, C);
    const int64_t u = head_loss_workspace_bytes(c, rows, C);
    return w > u ? w : u;
  }
  if (c.final_activation == 0) return gcs_regression_loss_workspace_bytes(rows, C);
  if (c.final_activation == 2) return gcs_sigmoid_bce_workspace_bytes(rows, C);
  return gcs_softmax_xent_workspace_bytes(rows, C);
}

static void make_plan(const gcs_model_config& c, int64_t N, int B, bool training, void* ws, Plan& p, int64_t* total,
                      int flags = 0) {
  build_blocks(c, p.blocks);
  p.P = c.pre_process; p.L = c.message_passing; p.Q = c.post_process;
  p.H = c.hidden; p.Wc = c.connectivity == 1 ? c.hidden * (c.message_passing + 1) : c.hidden; p.C = c.output;
  p.N = N; p.B = B;
  p.rows_post = c.pool ? B : N;
  p.attn_off = p.blocks.back().off + p.blocks.back().count();
  p.n_params = p.attn_off + (c.pool == kPoolAttnSum ? p.Wc : 0);
  Arena a(ws);
  p.amax = a.take<float>(64);
  const int64_t NH = N * p.H;
  if (training) p.stat_part = a.take<float>(ceil_div(N > 0 ? N : 1, 32) * p.H * 2);
  p.cat = a.take<float>(NH * (p.L + 1));         // 'cat': one [N, H(L+1)] matrix; otherwise L+1 slabs [N, H]
  p.h.assign(p.P + p.L, nullptr);
  if (training) {
    for (auto& q : p.h) q = a.take<float>(NH);
  } else {
    float* shared = a.take<float>(NH);
    for (auto& q : p.h) q = shared;
  }
  p.act.assign(p.P > 1 ? p.P - 1 : 0, nullptr);
  if (training) {
    for (auto& q : p.act) q = a.take<float>(NH);
  } else if (p.P > 1) {
    float* pp[2] = {a.take<float>(NH), p.P > 2 ? a.take<float>(NH) : nullptr};
    for (size_t j = 0; j < p.act.size(); ++j) p.act[j] = pp[j & 1];
  }
  p.stat.clear();
  for (const auto& b : p.blocks) p.stat.push_back(a.take<float>(4LL * b.m_out));
  if (c.pool) p.pooled = a.take<float>(static_cast<int64_t>(B) * p.Wc);
  if (c.pool == kPoolAttnSum) {
    if (training) {
      p.scores = a.take<float>(N);
      p.gstats = a.take<float>(2LL * B);
    }
    p.attn_ws_bytes = gcs_attn_pool_workspace_bytes(N, B, p.Wc);
    p.attn_ws = a.take<char>(p.attn_ws_bytes);
  }
  p.post_h.clear(); p.post_a.clear();
  for (int j = 0; j < p.Q; ++j) {
    const auto& b = p.blocks[p.P + p.L + j];
    p.post_h.push_back(a.take<float>(p.rows_post * b.m_out));
    if (j < p.Q - 1) p.post_a.push_back(a.take<float>(p.rows_post * p.H));
  }
  p.logits = a.take<float>(p.rows_post * p.C);
  int64_t bn_bytes = gcs_bn_workspace_bytes(N, p.H);
  for (int j = 0; j < p.Q; ++j) {
    const int64_t v = gcs_bn_workspace_bytes(p.rows_post, p.blocks[p.P + p.L + j].m_out);
    if (v > bn_bytes) bn_bytes = v;
  }
  p.bn_ws_bytes = bn_bytes;
  p.bn_ws = a.take<char>(bn_bytes);
  int64_t lin_bytes = c.connectivity == 1 ? gcs_linear_workspace_bytes(N, p.L * p.H, p.H) : 0;   // concatenated input-gradient GEMM
  for (const auto& b : p.blocks) {
    const int64_t v = gcs_linear_workspace_bytes(N, b.k_in, b.m_out);
    if (v > lin_bytes) lin_bytes = v;
  }
  p.lin_ws_bytes = lin_bytes;
  p.lin_ws = a.take<char>(lin_bytes);
  if (training) {
    if (!c.pool || c.pool == kPoolAttnSum) p.gcat = a.take<float>(N * p.Wc);
    p.dhcat = a.take<float>(c.connectivity == 1 ? NH * p.L : NH);
    p.tmp_a = a.take<float>(NH);
    p.tmp_b = a.take<float>(NH);
    p.tmp_c = a.take<float>(NH);
    p.dlogits = a.take<float>(p.rows_post * p.C);
    p.dpost = a.take<float>(p.rows_post * (p.H > p.C ? p.H : p.C));
    p.dpost_in = a.take<float>(p.rows_post * p.H);
    if (c.pool) p.dpooled = a.take<float>(static_cast<int64_t>(B) * p.Wc);
    int64_t lw = 0;
    for (size_t i = 0; i < p.blocks.size(); ++i) {
      const int64_t rows = static_cast<int>(i) < p.P + p.L ? N : p.rows_post;
      const int64_t v = gcs_linear_bwd_weight_workspace_bytes(rows, p.blocks[i].k_in, p.blocks[i].m_out);
      if (v > lw) lw = v;
    }
    p.lw_ws_bytes = lw;
    p.lw_ws = a.take<char>(lw);
    p.prep_ws_bytes = list_step_weights(c, p, nullptr, nullptr, nullptr, nullptr);
    p.prep_ws = a.take<char>(p.prep_ws_bytes);
  }
  // last: graph-level softmax plans keep their layout, and sample weights change no other offset
  p.loss_ws_bytes = head_loss_workspace_bytes(c, p.rows_post, p.C, flags);
  p.loss_ws = a.take<char>(p.loss_ws_bytes);
  *total = a.used;
}

static int check_batch(const gcs_model_config& c, const gcs_batch* b, bool need_labels, bool need_transpose) {
  if (!b) return fail(GCS_ERR_INVALID_ARGUMENT, "batch is NULL");
  if (b->n_nodes <= 0) return fail(GCS_ERR_INVALID_ARGUMENT, "batch has no nodes");
  if (b->nnz < 0) return fail(GCS_ERR_INVALID_ARGUMENT, "batch has negative nnz");
  if (!b->rowptr || (b->nnz > 0 && !b->colidx) || !b->x)
    return fail(GCS_ERR_INVALID_ARGUMENT, "batch: rowptr / colidx / x must be set");
  if (b->ldx < c.in_features) return fail(GCS_ERR_INVALID_ARGUMENT, "batch: ldx < in_features");
  if (c.pool && (b->n_graphs <= 0 || !b->graph_ptr))
    return fail(GCS_ERR_INVALID_ARGUMENT, "batch: pooling needs n_graphs > 0 and graph_ptr (the batch index i)");
  if (need_labels && !b->y) return fail(GCS_ERR_INVALID_ARGUMENT, "batch: training needs labels y");
  if (need_transpose && c.pool && !b->seg_ids)
    return fail(GCS_ERR_INVALID_ARGUMENT, "batch: the backward of the pool needs seg_ids (the batch index i)");
  if (need_transpose && (!b->rowptr_t || (b->nnz > 0 && !b->colidx_t)))
    return fail(GCS_ERR_INVALID_ARGUMENT, "batch: the backward needs the transposed CSR (alias it if symmetric)");
  if (need_transpose && b->values && !b->values_t)
    return fail(GCS_ERR_INVALID_ARGUMENT, "batch: the backward needs the edge weights in transposed order (values_t)");
  return GCS_OK;
}

// Y = pattern(A) . f(X) (+ residual) for the batch: per-graph shared-memory slabs when the batch says how long its graphs
// are (gcs_spmm_sum_graphs), the global-memory kernels otherwise.  transposed selects pattern(A)^T (the backward).
static int aggregate(const gcs_batch& bt, bool transposed, const float* X, int64_t ldx, const float* scale, const float* shift,
                     const float* alpha, const float* residual, int64_t ldr, float* Y, int64_t ldy, int H, gcs_stream st,
                     int agg = 0) {
  if (agg != 0 || bt.values)                         // weighted / mean / max (SURVEY.md 8 f3): the general row kernel
    return gcs_spmm_aggregate(transposed ? bt.rowptr_t : bt.rowptr, transposed ? bt.colidx_t : bt.colidx,
                              transposed ? bt.values_t : bt.values, nullptr, nullptr, bt.n_nodes, X, ldx, scale, shift, alpha,
                              residual, ldr, Y, ldy, H, agg, st);
  const int height = bt.rb_height ? bt.rb_height : 4;
  return gcs_spmm_sum_graphs(bt.graph_ptr, bt.n_graphs, bt.max_graph_nodes, transposed ? bt.rowptr_t : bt.rowptr,
                             transposed ? bt.colidx_t : bt.colidx, transposed ? bt.rb4_blk_ptr_t : bt.rb4_blk_ptr,
                             transposed ? bt.rb4_ent_t : bt.rb4_ent, height, bt.n_nodes, X, ldx, scale, shift, alpha, residual,
                             ldr, Y, ldy, H, st);
}

// dLoss/d(a_k) from dz = dLoss/d(z_k), z_k = agg(a_k): the transposed aggregation.  Z: the forward output z_k (max only).
// With dropout the forward aggregated the materialised a = prelu(dropout(bn(h))) (run_forward); the kernels that read
// f(X) again get the same a, rebuilt by the same kernel into `scratch` [N, H] (ld lds) and read with the transform off.
static int aggregate_bwd(const gcs_model_config& c, const Plan& p, const gcs_batch& bt, int bi, const float* params,
                         const float* dz, int64_t lddz, const float* Z, int64_t ldz, const Dropout& drop, float* scratch,
                         int64_t lds, gcs_stream st) {
  const int H = p.H;
  if (c.aggregate == 0 && !bt.values)
    return aggregate(bt, true, dz, lddz, nullptr, nullptr, nullptr, nullptr, 0, p.tmp_a, H, H, st);
  const float* scale = p.stat[bi] + 2 * H;
  const float* X = p.h[bi];
  int64_t ldx = H;
  const float* alpha = params + p.blocks[bi].alpha();
  if (drop.threshold) {
    const Dropout d = block_dropout(drop, bi);
    AmaxScope off(nullptr, amax_sink().consume, amax_sink().consume_act);
    GCS_TIMED("dropout_act", bn_prelu_fwd(p.h[bi], H, scale, scale + H, alpha, scratch, lds, p.N, H, &d, st));
    X = scratch;
    ldx = lds;
    scale = nullptr;
    alpha = nullptr;
  }
  return gcs_spmm_aggregate_bwd(bt.rowptr_t, bt.colidx_t, bt.values ? bt.values_t : nullptr, bt.rowptr, bt.colidx, bt.values,
                                bt.n_nodes, dz, lddz, c.aggregate, X, ldx, scale, scale ? scale + H : nullptr, alpha, Z,
                                ldz, p.tmp_b, H, p.tmp_a, H, H, st);
}

// BatchNorm statistics -> folded scale/shift for block bi over `rows` rows of h.
static int block_norm(const gcs_model_config& c, const Plan& p, int bi, const float* params, float* state,
                      const float* h, int64_t ldh, int64_t rows, bool training, gcs_stream st,
                      const float* stat_part = nullptr) {
  const BlockDesc& b = p.blocks[bi];
  float* mean = p.stat[bi];
  float* var = mean + b.m_out;
  float* scale = var + b.m_out;
  float* shift = scale + b.m_out;
  float* mm = state + b.stat_off;
  float* mv = mm + b.m_out;
  if (training) {
    if (stat_part) GCS_TIMED("bn_stats", bn_stats_from_partials(stat_part, rows, b.m_out, mean, var, p.bn_ws, p.bn_ws_bytes, st));
    else GCS_TIMED("bn_stats", gcs_bn_stats(h, ldh, rows, b.m_out, mean, var, p.bn_ws, p.bn_ws_bytes, st));
    GCS_TRY(gcs_bn_fold(mean, var, params + b.gamma(), params + b.beta(), c.bn_epsilon, c.bn_momentum, mm, mv,
                        scale, shift, b.m_out, st));
  } else {
    GCS_TRY(gcs_bn_fold(mm, mv, params + b.gamma(), params + b.beta(), c.bn_epsilon, c.bn_momentum, nullptr,
                        nullptr, scale, shift, b.m_out, st));
  }
  return GCS_OK;
}

// Everything up to the logits ([rows_post, C] in p.logits).
static int run_forward(const gcs_model_config& c, const Plan& p, const float* params, float* state,
                       const gcs_batch& bt, bool training, const Dropout& drop, gcs_stream st) {
  const int H = p.H, Wc = p.Wc, L = p.L, P = p.P;
  const int64_t N = p.N;
  const bool cat = c.connectivity == 1;
  // out_k, the node embedding after k conv layers: the trailing (k+1)H columns of `cat`, or slab k
  auto emb = [&](int k) { return cat ? p.cat + static_cast<int64_t>(L - k) * H : p.cat + static_cast<int64_t>(k) * N * H; };
  const int64_t ld_emb = cat ? Wc : H;
  // Every node-level activation written from here on folds its |max| into amax[0]; the dense transforms that read
  // them (all but the one on the raw features) take it as the |max| of their A operand (fp16 split, linear_tc.cu).
  GCS_CUDA(cudaMemsetAsync(p.amax, 0, sizeof(float), as_stream(st)));
  AmaxScope node_scope(p.amax, nullptr);
  // pre-processing MLP
  const float* in = bt.x;
  int64_t ld_in = bt.ldx;
  for (int j = 0; j < P; ++j) {
    const BlockDesc& b = p.blocks[j];
    amax_sink().consume = j > 0 ? p.amax : nullptr;
    float* out = j < P - 1 ? p.act[j] : emb(0);
    const int64_t ld_out = j < P - 1 ? H : ld_emb;
    const float* scale = p.stat[j] + 2 * H;
    int fused = 0;
    if (!training) {
      // inference: moving-statistics BatchNorm folded into the GEMM, PReLU in its epilogue (one pass instead of three);
      // the |max| of the result goes through a scratch cell so that the GEMM does not raise the cell it reads
      GCS_TRY(block_norm(c, p, j, params, state, nullptr, H, N, false, st));
      GCS_TIMED("linear_fwd", linear_fwd_fused(in, ld_in, params + b.kernel(), params + b.bias(), scale, scale + H,
                                               params + b.alpha(), out, ld_out, N, b.k_in, H, p.lin_ws, p.lin_ws_bytes,
                                               p.amax + 2, nullptr, as_stream(st), &fused));
      if (fused) GCS_TRY(tc::amax_merge(p.amax, p.amax + 2, as_stream(st)));
    }
    if (!fused) {
      // training: the GEMM epilogue leaves the BatchNorm sums of its output (no separate pass over h) where it can
      int with_stats = 0;
      if (training)
        GCS_TIMED("linear_fwd", linear_fwd_fused(in, ld_in, params + b.kernel(), params + b.bias(), nullptr, nullptr, nullptr,
                                                 p.h[j], H, N, b.k_in, H, p.lin_ws, p.lin_ws_bytes, nullptr, p.stat_part,
                                                 as_stream(st), &with_stats));
      if (!with_stats)
        GCS_TIMED("linear_fwd", gcs_linear_fwd(in, ld_in, params + b.kernel(), params + b.bias(), p.h[j], H, N, b.k_in, H, p.lin_ws, p.lin_ws_bytes, st));
      GCS_TRY(block_norm(c, p, j, params, state, p.h[j], H, N, training, st, with_stats ? p.stat_part : nullptr));
      const Dropout d = block_dropout(drop, j);
      GCS_TIMED("bn_prelu_fwd", bn_prelu_fwd(p.h[j], H, scale, scale + H, params + b.alpha(), out, ld_out, N, H, &d, st));
    }
    in = out;
    ld_in = ld_out;
  }
  // message passing with in-place concat
  amax_sink().consume = p.amax;
  for (int k = 0; k < L; ++k) {
    const int bi = P + k;
    const BlockDesc& b = p.blocks[bi];
    const float* cin = emb(k);
    const float* scale = p.stat[bi] + 2 * H;
    int fused = 0;
    if (!training) {
      // inference: p.h[bi] receives prelu(bn(out . W + b)) straight from the GEMM; the aggregation is a plain gather
      GCS_TRY(block_norm(c, p, bi, params, state, nullptr, H, N, false, st));
      GCS_TIMED("linear_fwd", linear_fwd_fused(cin, ld_emb, params + b.kernel(), params + b.bias(), scale, scale + H,
                                               params + b.alpha(), p.h[bi], H, N, b.k_in, H, p.lin_ws, p.lin_ws_bytes,
                                               nullptr, nullptr, as_stream(st), &fused));
    }
    if (fused) {
      GCS_TIMED("spmm_fwd", aggregate(bt, false, p.h[bi], H, nullptr, nullptr, nullptr, c.connectivity == 2 ? emb(k) : nullptr, H,
                                      emb(k + 1), ld_emb, H, st, c.aggregate));
      continue;
    }
    int with_stats = 0;
    if (training)
      GCS_TIMED("linear_fwd", linear_fwd_fused(cin, ld_emb, params + b.kernel(), params + b.bias(), nullptr, nullptr, nullptr,
                                               p.h[bi], H, N, b.k_in, H, p.lin_ws, p.lin_ws_bytes, nullptr, p.stat_part,
                                               as_stream(st), &with_stats));
    if (!with_stats)
      GCS_TIMED("linear_fwd", gcs_linear_fwd(cin, ld_emb, params + b.kernel(), params + b.bias(), p.h[bi], H, N, b.k_in, H, p.lin_ws, p.lin_ws_bytes, st));
    GCS_TRY(block_norm(c, p, bi, params, state, p.h[bi], H, N, training, st, with_stats ? p.stat_part : nullptr));
    const float* ax = p.h[bi];
    const float* ascale = scale;
    const float* aalpha = params + b.alpha();
    if (drop.threshold) {
      // dropout: a = prelu(dropout(bn(h))) written once per node and aggregated as it is, instead of one mask draw per
      // gathered entry inside the aggregation kernels (DESIGN.md 3.12).  a is no GEMM operand: its |max| is not folded.
      // tmp_a, a backward buffer of the training plan, is free during the forward.
      const Dropout d = block_dropout(drop, bi);
      AmaxScope off(nullptr, amax_sink().consume, amax_sink().consume_act);
      GCS_TIMED("dropout_act", bn_prelu_fwd(p.h[bi], H, scale, scale + H, aalpha, p.tmp_a, H, N, H, &d, st));
      ax = p.tmp_a;
      ascale = nullptr;
      aalpha = nullptr;
    }
    // z_k is the leading block of out_{k+1} ('cat'), or out_{k+1} = z_k (+ out_k for 'sum') in the next slab
    GCS_TIMED("spmm_fwd", aggregate(bt, false, ax, H, ascale, ascale ? ascale + H : nullptr, aalpha,
                                    c.connectivity == 2 ? emb(k) : nullptr, H, emb(k + 1), ld_emb, H, st, c.aggregate));
  }
  // global pool
  amax_sink() = AmaxSink();                                 // pooled rows and the post-MLP: tf32 kernels / CUDA cores
  const float* pin = emb(L);
  int64_t ld_pin = Wc;
  if (c.pool == kPoolSum)
    GCS_TIMED("pool_fwd", gcs_segment_sum_fwd(emb(L), Wc, bt.graph_ptr, bt.n_graphs, Wc, p.pooled, Wc, st));
  else if (c.pool == kPoolAvg)
    GCS_TIMED("pool_fwd", gcs_segment_mean_fwd(emb(L), Wc, bt.graph_ptr, bt.n_graphs, Wc, p.pooled, Wc, st));
  else if (c.pool == kPoolAttnSum)
    GCS_TIMED("pool_fwd", gcs_attn_sum_pool_fwd(emb(L), Wc, N, params + p.attn_off, bt.graph_ptr, bt.n_graphs, Wc, p.pooled, Wc,
                                                p.scores, p.gstats, p.attn_ws, p.attn_ws_bytes, st));
  if (c.pool) pin = p.pooled;
  // post-processing MLP
  const int64_t R = p.rows_post;
  for (int j = 0; j < p.Q; ++j) {
    const int bi = P + L + j;
    const BlockDesc& b = p.blocks[bi];
    GCS_TRY(gcs_linear_fwd(pin, ld_pin, params + b.kernel(), params + b.bias(), p.post_h[j], b.m_out, R, b.k_in,
                           b.m_out, p.lin_ws, p.lin_ws_bytes, st));
    GCS_TRY(block_norm(c, p, bi, params, state, p.post_h[j], b.m_out, R, training, st));
    const float* scale = p.stat[bi] + 2 * b.m_out;
    const Dropout d = block_dropout(drop, bi);     // the last block too: Keras' dropout acts on the logits
    if (j < p.Q - 1) {
      GCS_TRY(bn_prelu_fwd(p.post_h[j], b.m_out, scale, scale + b.m_out, params + b.alpha(), p.post_a[j], H, R,
                           b.m_out, &d, st));
      pin = p.post_a[j];
      ld_pin = H;
    } else {
      GCS_TRY(bn_prelu_fwd(p.post_h[j], b.m_out, scale, scale + b.m_out, nullptr, p.logits, p.C, R, p.C, &d, st));
    }
  }
  return GCS_OK;
}

// Backward of one dense block given da = dLoss/d(block output): parameter gradients into
// `grads`, dh left in `dh`; optionally the input gradient.
static int block_backward(const gcs_model_config& c, const Plan& p, int bi, const float* params, float* grads,
                          const float* da, int64_t ldda, const float* h, int64_t ldh, int64_t rows,
                          const float* in, int64_t ld_in, float* dh, int64_t lddh, float* din, int64_t lddin,
                          int accumulate, const Dropout& drop, gcs_stream st) {
  const BlockDesc& b = p.blocks[bi];
  const Dropout d = block_dropout(drop, bi);
  const float* mean = p.stat[bi];
  const float* var = mean + b.m_out;
  float* const dh_amax = const_cast<float*>(amax_sink().consume);      // set for the node-level blocks only
  amax_sink().produce = dh_amax;
  GCS_TIMED("bn_prelu_bwd", bn_prelu_bwd(da, ldda, h, ldh, mean, var, params + b.gamma(), params + b.beta(),
                                         b.has_alpha ? params + b.alpha() : nullptr, c.bn_epsilon, dh, lddh,
                                         grads + b.gamma(), grads + b.beta(),
                                         b.has_alpha ? grads + b.alpha() : nullptr, grads + b.bias(), rows, b.m_out,
                                         p.bn_ws, p.bn_ws_bytes, &d, st));
  amax_sink().produce = nullptr;
  // the bias gradient (column sums of dh) came out of the BatchNorm backward's apply pass
  GCS_TIMED("linear_bwd_weight", gcs_linear_bwd_weight(in, ld_in, dh, lddh, grads + b.kernel(), nullptr, rows,
                                                       b.k_in, b.m_out, p.lw_ws, p.lw_ws_bytes, st));
  if (din)
    GCS_TIMED("linear_bwd_input", gcs_linear_bwd_input(dh, lddh, params + b.kernel(), din, lddin, rows, b.k_in,
                                                       b.m_out, accumulate, p.lin_ws, p.lin_ws_bytes, st));
  return GCS_OK;
}

// Called by run_backward whenever a trailing range of the flat gradient buffer is final: [begin, end) in floats, the
// ranges tile the buffer from its end to its start.  The data-parallel step uses it to start the all-reduce of the
// layers already differentiated while the earlier layers are still in the backward.
struct GradReady {
  int (*fn)(void* user, int64_t begin, int64_t end);
  void* user;
};

// The head on p.logits: softmax with categorical cross-entropy, sigmoid with binary cross-entropy, or a linear head
// with the regression loss c.loss selects (MSE by default).  probs gets the head's output (the probabilities, or a copy
// of a linear head's logits).  With labels y it also leaves loss_acc and dLoss/dlogits (scaled by grad_scale) in
// p.dlogits; with y = NULL, only probs.  Per-row weights w (with y) select the weighted form of the same head.
static int head_loss(const gcs_model_config& c, const Plan& p, const float* y, float* probs, float* loss_acc,
                     float grad_scale, gcs_stream st, const float* w = nullptr) {
  float* dlogits = y ? p.dlogits : nullptr;
  if (y && w)
    return gcs_weighted_loss(c.final_activation, c.loss ? c.loss : 1, c.huber_delta, p.logits, y, w, p.rows_post, p.C,
                             probs, loss_acc, dlogits, grad_scale, p.loss_ws, p.loss_ws_bytes, st);
  if (c.final_activation == 0)
    return gcs_regression_loss(c.loss ? c.loss : 1, c.huber_delta, p.logits, y, p.rows_post, p.C, probs, loss_acc,
                               dlogits, grad_scale, p.loss_ws, p.loss_ws_bytes, st);
  if (c.final_activation == 2)
    return gcs_sigmoid_bce(p.logits, y, p.rows_post, p.C, probs, loss_acc, dlogits, grad_scale, p.loss_ws,
                           p.loss_ws_bytes, st);
  GCS_CHECK_ARG(p.rows_post < INT32_MAX, "softmax head: too many output rows");
  return gcs_softmax_xent_ws(p.logits, y, static_cast<int32_t>(p.rows_post), p.C, probs, loss_acc, dlogits, grad_scale,
                             p.loss_ws, p.loss_ws_bytes, st);
}

// Reverse pass given dlogits = dLoss/d(logits) [rows_post, C]; needs the activations a
// training-mode run_forward left in the workspace.
static int run_backward(const gcs_model_config& c, const Plan& p, const float* params, float* grads,
                        const gcs_batch& bt, const float* dlogits, const Dropout& drop, gcs_stream st,
                        const GradReady* ready = nullptr) {
  const int H = p.H, Wc = p.Wc, L = p.L, P = p.P, Q = p.Q;
  const int64_t N = p.N, R = p.rows_post;
  const bool cat = c.connectivity == 1;
  auto emb = [&](int k) { return cat ? p.cat + static_cast<int64_t>(L - k) * H : p.cat + static_cast<int64_t>(k) * N * H; };
  const int64_t ld_emb = cat ? Wc : H;
  // dh of every node-level block folds its |max| into amax[1] (BatchNorm backward apply pass); the input-gradient
  // GEMMs read dh as their A operand
  GCS_CUDA(cudaMemsetAsync(p.amax + 1, 0, sizeof(float), as_stream(st)));
  // ---- post-processing MLP, last block first
  const float* da = dlogits;
  int64_t ldda = p.C;
  for (int j = Q - 1; j >= 0; --j) {
    const int bi = P + L + j;
    const BlockDesc& b = p.blocks[bi];
    const float* in = j == 0 ? (c.pool ? p.pooled : emb(L)) : p.post_a[j - 1];
    const int64_t ld_in = j == 0 ? Wc : H;
    float* din;
    int64_t lddin;
    if (j == 0) { din = c.pool ? p.dpooled : p.gcat; lddin = Wc; }
    else { din = p.dpost_in; lddin = H; }
    GCS_TRY(block_backward(c, p, bi, params, grads, da, ldda, p.post_h[j], b.m_out, R, in, ld_in, p.dpost, b.m_out,
                           din, lddin, 0, drop, st));
    da = din;
    ldda = lddin;
  }
  // From here on the node-level code sees either a pooled gradient dpooled [B, Wc] that every node of graph g receives
  // ('sum'; 'avg' after dividing row g by n_g) or, for 'attn_sum' and without pooling, dLoss/d(emb(L)) in full in gcat.
  const bool pooled_grad = c.pool == kPoolSum || c.pool == kPoolAvg;
  if (c.pool == kPoolAvg)
    GCS_TIMED("pool_bwd", segment_rows_div_count(p.dpooled, Wc, bt.graph_ptr, bt.n_graphs, Wc, st));
  else if (c.pool == kPoolAttnSum)
    GCS_TIMED("pool_bwd", gcs_attn_sum_pool_bwd(p.dpooled, Wc, emb(L), Wc, N, params + p.attn_off, bt.graph_ptr, bt.n_graphs, Wc,
                                                p.pooled, Wc, p.scores, p.gstats, p.gcat, Wc, grads + p.attn_off, p.attn_ws,
                                                p.attn_ws_bytes, st));
  int64_t grads_final_from = p.n_params;                    // everything from here on is final
  auto notify = [&](int first_block) -> int {                // blocks first_block .. have all been differentiated
    const int64_t begin = p.blocks[first_block].off;
    if (ready && begin < grads_final_from) GCS_TRY(ready->fn(ready->user, begin, grads_final_from));
    grads_final_from = begin < grads_final_from ? begin : grads_final_from;
    return GCS_OK;
  };
  AmaxScope node_scope(nullptr, p.amax + 1, p.amax);        // weight gradients: activations under amax[0], dh under amax[1]
  // ---- message passing, last layer first.  Block z_k of cat (columns [(L-1-k)H, (L-k)H)) is read by
  // the pool and by every later conv layer k' > k (rows [(k'-1-k)H, (k'-k)H) of its kernel).
  const int64_t ldd = static_cast<int64_t>(L) * H;
  std::vector<const float*> Wp(L);
  std::vector<int> roff(L);
  cudaStream_t cst = as_stream(st);
  for (int k = L - 1; k >= 0 && cat; --k) {
    const int bi = P + k;
    const int nb = L - 1 - k;
    for (int q = 0; q < nb; ++q) {
      const int kp = k + 1 + q;
      Wp[q] = params + p.blocks[P + kp].kernel();
      roff[q] = (kp - 1 - k) * H;
    }
    const float* dz;
    int64_t lddz;
    if (pooled_grad) {
      const float* rb = p.dpooled + static_cast<int64_t>(L - 1 - k) * H;
      if (nb == 0) {
        GCS_TIMED("pool_bwd", gcs_segment_sum_bwd(rb, Wc, bt.graph_ptr, bt.n_graphs, H, p.tmp_c, H, st));
      } else {
        GCS_TIMED("linear_bwd_input", dense_dx_concat(p.dhcat + static_cast<int64_t>(k + 1) * H, ldd, Wp.data(), roff.data(), nb, H, H,
                                                      rb, Wc, bt.seg_ids, bt.graph_ptr, bt.n_graphs, p.tmp_c, H, N, 0,
                                                      p.lin_ws, p.lin_ws_bytes, cst));
      }
      dz = p.tmp_c;
      lddz = H;
    } else {
      float* blk = p.gcat + static_cast<int64_t>(L - 1 - k) * H;
      if (nb > 0)
        GCS_TIMED("linear_bwd_input", dense_dx_concat(p.dhcat + static_cast<int64_t>(k + 1) * H, ldd, Wp.data(), roff.data(), nb, H, H,
                                                      nullptr, 0, nullptr, nullptr, 0, blk, Wc, N, 1, p.lin_ws,
                                                      p.lin_ws_bytes, cst));
      dz = blk;
      lddz = Wc;
    }
    // the dh slot of block k is written by its block_backward below: free scratch for the aggregation backward
    GCS_TIMED("spmm_bwd", aggregate_bwd(c, p, bt, bi, params, dz, lddz, p.cat + static_cast<int64_t>(L - 1 - k) * H, Wc, drop,
                                        p.dhcat + static_cast<int64_t>(k) * H, ldd, st));
    GCS_TRY(block_backward(c, p, bi, params, grads, p.tmp_a, H, p.h[bi], H, N, p.cat + static_cast<int64_t>(L - k) * H, Wc,
                           p.dhcat + static_cast<int64_t>(k) * H, ldd, nullptr, 0, 0, drop, st));
    if (k == L - 1 || k == (L - 1) / 2) GCS_TRY(notify(bi));   // two buckets inside the message-passing stack
  }
  // ---- pre-processing MLP: its output block (last H columns of cat) is read by the pool and by
  // every conv layer k' (rows [k'H, (k'+1)H) of its kernel)
  for (int kp = 0; kp < L; ++kp) {
    Wp[kp] = params + p.blocks[P + kp].kernel();
    roff[kp] = kp * H;
  }
  const float* da_pre;
  int64_t ldda_pre;
  if (!cat) {
    // one running gradient g = dLoss/d(out_k): through z_k into the conv block, and - for 'sum' - straight on to out_{k-1}
    float* g = p.gcat;
    if (pooled_grad) {
      GCS_TIMED("pool_bwd", gcs_segment_sum_bwd(p.dpooled, Wc, bt.graph_ptr, bt.n_graphs, H, p.tmp_c, H, st));
      g = p.tmp_c;
    }
    for (int k = L - 1; k >= 0; --k) {
      GCS_TIMED("spmm_bwd", aggregate_bwd(c, p, bt, P + k, params, g, H, emb(k + 1), H, drop, p.dhcat, H, st));
      GCS_TRY(block_backward(c, p, P + k, params, grads, p.tmp_a, H, p.h[P + k], H, N, emb(k), ld_emb, p.dhcat, H, g, H,
                             c.connectivity == 2 ? 1 : 0, drop, st));
      if (k == L - 1 || k == (L - 1) / 2) GCS_TRY(notify(P + k));
    }
    da_pre = g;
    ldda_pre = H;
  } else if (pooled_grad) {
    GCS_TIMED("linear_bwd_input", dense_dx_concat(p.dhcat, ldd, Wp.data(), roff.data(), L, H, H, p.dpooled + static_cast<int64_t>(L) * H, Wc,
                                                  bt.seg_ids, bt.graph_ptr, bt.n_graphs, p.tmp_c, H, N, 0, p.lin_ws,
                                                  p.lin_ws_bytes, cst));
    da_pre = p.tmp_c;
    ldda_pre = H;
  } else {
    float* blk = p.gcat + static_cast<int64_t>(L) * H;
    GCS_TIMED("linear_bwd_input", dense_dx_concat(p.dhcat, ldd, Wp.data(), roff.data(), L, H, H, nullptr, 0, nullptr, nullptr, 0, blk,
                                                  Wc, N, 1, p.lin_ws, p.lin_ws_bytes, cst));
    da_pre = blk;
    ldda_pre = Wc;
  }
  da = da_pre;
  ldda = ldda_pre;
  for (int j = P - 1; j >= 0; --j) {
    if (j == 0) amax_sink().consume_act = nullptr;           // the raw features are not covered by amax[0]
    const float* in = j == 0 ? bt.x : p.act[j - 1];
    const int64_t ld_in = j == 0 ? bt.ldx : H;
    GCS_TRY(block_backward(c, p, j, params, grads, da, ldda, p.h[j], H, N, in, ld_in, p.tmp_b, H,
                           j > 0 ? p.tmp_a : nullptr, H, 0, drop, st));
    da = p.tmp_a;
    ldda = H;
  }
  GCS_TRY(notify(0));
  return GCS_OK;
}

}  // namespace gcs

using namespace gcs;

extern "C" int64_t gcs_model_num_params(const gcs_model_config* cfg) {
  if (check_config(cfg) != GCS_OK) return -1;
  std::vector<BlockDesc> blocks;
  build_blocks(*cfg, blocks);
  const int64_t wc = cfg->connectivity == 1 ? static_cast<int64_t>(cfg->hidden) * (cfg->message_passing + 1) : cfg->hidden;
  return blocks.back().off + blocks.back().count() + (cfg->pool == kPoolAttnSum ? wc : 0);
}

extern "C" int64_t gcs_model_num_state(const gcs_model_config* cfg) {
  if (check_config(cfg) != GCS_OK) return -1;
  std::vector<BlockDesc> blocks;
  build_blocks(*cfg, blocks);
  return blocks.back().stat_off + 2LL * blocks.back().m_out;
}

extern "C" int64_t gcs_model_workspace_bytes_ex(const gcs_model_config* cfg, int64_t n_nodes, int64_t nnz,
                                                int32_t n_graphs, int32_t training, int32_t flags) {
  (void)nnz;
  if (check_config(cfg) != GCS_OK || n_nodes < 0 || n_graphs < 0 || (flags & ~GCS_WORKSPACE_SAMPLE_WEIGHTS)) return -1;
  Plan p;
  int64_t total = 0;
  make_plan(*cfg, n_nodes, n_graphs, training != 0, nullptr, p, &total, flags);
  return total;
}

extern "C" int64_t gcs_model_workspace_bytes(const gcs_model_config* cfg, int64_t n_nodes, int64_t nnz,
                                             int32_t n_graphs, int32_t training) {
  return gcs_model_workspace_bytes_ex(cfg, n_nodes, nnz, n_graphs, training, 0);
}

extern "C" int gcs_model_forward_ex(const gcs_model_config* cfg, const float* params, float* state,
                                    const gcs_batch* batch, int32_t training, float* out, void* workspace,
                                    int64_t workspace_bytes, gcs_stream stream, const gcs_dropout* dropout) {
  GCS_TRY(check_config(cfg));
  Dropout drop;
  GCS_TRY(step_dropout(dropout, training != 0, &drop));
  GCS_TRY(check_batch(*cfg, batch, false, false));
  GCS_CHECK_ARG(params && state && out && workspace, "gcs_model_forward: null pointer");
  GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "gcs_model_forward: workspace must be 256-byte aligned");
  Plan p;
  int64_t total = 0;
  make_plan(*cfg, batch->n_nodes, batch->n_graphs, training != 0, workspace, p, &total);
  if (workspace_bytes < total)
    return fail(GCS_ERR_WORKSPACE, "gcs_model_forward: workspace %lld < %lld bytes", (long long)workspace_bytes, (long long)total);
  GCS_TRY(run_forward(*cfg, p, params, state, *batch, training != 0, drop, stream));
  return head_loss(*cfg, p, nullptr, out, nullptr, 0.f, stream);
}

extern "C" int gcs_model_forward(const gcs_model_config* cfg, const float* params, float* state,
                                 const gcs_batch* batch, int32_t training, float* out, void* workspace,
                                 int64_t workspace_bytes, gcs_stream stream) {
  return gcs_model_forward_ex(cfg, params, state, batch, training, out, workspace, workspace_bytes, stream, nullptr);
}

extern "C" int gcs_model_train_step_ex(const gcs_model_config* cfg, const float* params, float* state,
                                       const gcs_batch* batch, float grad_scale, float* grads, float* probs,
                                       float* loss_acc, void* workspace, int64_t workspace_bytes,
                                       gcs_stream stream, const gcs_dropout* dropout) {
  GCS_TRY(check_config(cfg));
  Dropout drop;
  GCS_TRY(step_dropout(dropout, true, &drop));
  GCS_TRY(check_batch(*cfg, batch, true, true));
  GCS_CHECK_ARG(params && state && grads && loss_acc && workspace, "gcs_model_train_step: null pointer");
  GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "gcs_model_train_step: workspace must be 256-byte aligned");
  const gcs_model_config& c = *cfg;
  const gcs_batch& bt = *batch;
  Plan p;
  int64_t total = 0;
  make_plan(c, bt.n_nodes, bt.n_graphs, true, workspace, p, &total, bt.sample_weight ? GCS_WORKSPACE_SAMPLE_WEIGHTS : 0);
  if (workspace_bytes < total)
    return fail(GCS_ERR_WORKSPACE, "gcs_model_train_step: workspace %lld < %lld bytes", (long long)workspace_bytes, (long long)total);
  GCS_CHECK_ARG(p.rows_post < INT32_MAX, "gcs_model_train_step: too many output rows");
  PreparedTable prepared;
  GCS_TRY(prepare_step_weights(c, p, params, &prepared, stream));
  PreparedScope prepared_scope(&prepared);
  GCS_TRY(run_forward(c, p, params, state, bt, true, drop, stream));
  GCS_TRY(head_loss(c, p, bt.y, probs, loss_acc, grad_scale, stream, bt.sample_weight));

  return run_backward(c, p, params, grads, bt, p.dlogits, drop, stream);
}

extern "C" int gcs_model_train_step(const gcs_model_config* cfg, const float* params, float* state,
                                    const gcs_batch* batch, float grad_scale, float* grads, float* probs,
                                    float* loss_acc, void* workspace, int64_t workspace_bytes,
                                    gcs_stream stream) {
  return gcs_model_train_step_ex(cfg, params, state, batch, grad_scale, grads, probs, loss_acc, workspace,
                                 workspace_bytes, stream, nullptr);
}

// Data-parallel train step: gcs_model_train_step + the gradient all-reduce, started bucket by bucket on comm_stream as
// the backward finishes trailing ranges of the flat gradient buffer, so that only the last bucket's reduction is exposed.
// On return (asynchronously) `stream` waits for the reductions: whatever follows on it - the optimizer step - sees the
// summed gradients.
namespace {
struct DpSync {
  gcs_comm* comm; float* grads; cudaStream_t compute, comm_stream; cudaEvent_t ev[8]; int used;
};
int dp_bucket(void* user, int64_t begin, int64_t end) {
  DpSync* d = static_cast<DpSync*>(user);
  if (d->used >= 8) return fail(GCS_ERR_INVALID_ARGUMENT, "gcs_model_train_step_dp: too many gradient buckets");
  cudaEvent_t e = d->ev[d->used++];
  GCS_CUDA(cudaEventRecord(e, d->compute));
  GCS_CUDA(cudaStreamWaitEvent(d->comm_stream, e, 0));
  return gcs_allreduce_grads(d->comm, d->grads + begin, end - begin, d->comm_stream);
}
cudaEvent_t* dp_events() {           // per host thread: recorded and waited on within one call, reusable afterwards
  thread_local cudaEvent_t ev[9];
  thread_local bool made = false;
  if (!made) {
    for (auto& e : ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    made = true;
  }
  return ev;
}
}  // namespace

namespace {
int dp_sync_bn(double* buf, int64_t n, gcs_stream stream, void* user) {   // synchronised BatchNorm over the step's communicator
  return gcs_allreduce_f64(static_cast<gcs_comm*>(user), buf, n, stream);
}
struct HookScope {                                                        // call-scoped: restored on every exit path
  SyncHook saved;
  bool active;
  HookScope(gcs_comm* comm, bool on) : saved(sync_hook()), active(on) {
    if (on) { sync_hook().fn = dp_sync_bn; sync_hook().user = comm; sync_hook().world = gcs_comm_world_size(comm); }
  }
  ~HookScope() { if (active) sync_hook() = saved; }
};
}  // namespace

extern "C" int gcs_model_train_step_dp_ex(const gcs_model_config* cfg, const float* params, float* state,
                                          const gcs_batch* batch, float grad_scale, float* grads, float* probs,
                                          float* loss_acc, void* workspace, int64_t workspace_bytes, gcs_stream stream,
                                          gcs_comm* comm, gcs_stream comm_stream, int32_t sync_batchnorm,
                                          const gcs_dropout* dropout) {
  GCS_TRY(check_config(cfg));
  Dropout drop;
  GCS_TRY(step_dropout(dropout, true, &drop));
  GCS_TRY(check_batch(*cfg, batch, true, true));
  GCS_CHECK_ARG(params && state && grads && loss_acc && workspace && comm, "gcs_model_train_step_dp: null pointer");
  GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "gcs_model_train_step_dp: workspace must be 256-byte aligned");
  GCS_CHECK_ARG(comm_stream != stream, "gcs_model_train_step_dp: the collective needs its own stream");
  const gcs_model_config& c = *cfg;
  const gcs_batch& bt = *batch;
  Plan p;
  int64_t total = 0;
  make_plan(c, bt.n_nodes, bt.n_graphs, true, workspace, p, &total, bt.sample_weight ? GCS_WORKSPACE_SAMPLE_WEIGHTS : 0);
  if (workspace_bytes < total)
    return fail(GCS_ERR_WORKSPACE, "gcs_model_train_step_dp: workspace %lld < %lld bytes", (long long)workspace_bytes, (long long)total);
  GCS_CHECK_ARG(p.rows_post < INT32_MAX, "gcs_model_train_step_dp: too many output rows");
  HookScope hook(comm, sync_batchnorm != 0 && gcs_comm_world_size(comm) > 1);
  PreparedTable prepared;
  GCS_TRY(prepare_step_weights(c, p, params, &prepared, stream));
  PreparedScope prepared_scope(&prepared);
  GCS_TRY(run_forward(c, p, params, state, bt, true, drop, stream));
  GCS_TRY(head_loss(c, p, bt.y, probs, loss_acc, grad_scale, stream, bt.sample_weight));
  cudaEvent_t* ev = dp_events();
  DpSync sync{comm, grads, as_stream(stream), as_stream(comm_stream), {}, 0};
  for (int i = 0; i < 8; ++i) sync.ev[i] = ev[i];
  GradReady ready{dp_bucket, &sync};
  GCS_TRY(run_backward(c, p, params, grads, bt, p.dlogits, drop, stream, &ready));
  GCS_CUDA(cudaEventRecord(ev[8], as_stream(comm_stream)));
  GCS_CUDA(cudaStreamWaitEvent(as_stream(stream), ev[8], 0));
  return GCS_OK;
}

extern "C" int gcs_model_train_step_dp(const gcs_model_config* cfg, const float* params, float* state,
                                       const gcs_batch* batch, float grad_scale, float* grads, float* probs,
                                       float* loss_acc, void* workspace, int64_t workspace_bytes, gcs_stream stream,
                                       gcs_comm* comm, gcs_stream comm_stream, int32_t sync_batchnorm) {
  return gcs_model_train_step_dp_ex(cfg, params, state, batch, grad_scale, grads, probs, loss_acc, workspace,
                                    workspace_bytes, stream, comm, comm_stream, sync_batchnorm, nullptr);
}

extern "C" int64_t gcs_model_logits_offset(const gcs_model_config* cfg, int64_t n_nodes, int32_t n_graphs,
                                           int32_t training) {
  if (check_config(cfg) != GCS_OK || n_nodes < 0 || n_graphs < 0) return -1;
  Plan p;
  int64_t total = 0;
  // measure against a fake non-null base so that pointers are offsets + 256
  make_plan(*cfg, n_nodes, n_graphs, training != 0, reinterpret_cast<void*>(256), p, &total);
  return reinterpret_cast<char*>(p.logits) - reinterpret_cast<char*>(256);
}

extern "C" int gcs_model_backward_ex(const gcs_model_config* cfg, const float* params, const gcs_batch* batch,
                                     const float* dlogits, float* grads, void* workspace, int64_t workspace_bytes,
                                     gcs_stream stream, const gcs_dropout* dropout) {
  GCS_TRY(check_config(cfg));
  Dropout drop;
  GCS_TRY(step_dropout(dropout, true, &drop));
  GCS_TRY(check_batch(*cfg, batch, false, true));
  GCS_CHECK_ARG(params && dlogits && grads && workspace, "gcs_model_backward: null pointer");
  GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "gcs_model_backward: workspace must be 256-byte aligned");
  Plan p;
  int64_t total = 0;
  make_plan(*cfg, batch->n_nodes, batch->n_graphs, true, workspace, p, &total);
  if (workspace_bytes < total)
    return fail(GCS_ERR_WORKSPACE, "gcs_model_backward: workspace %lld < %lld bytes", (long long)workspace_bytes, (long long)total);
  return run_backward(*cfg, p, params, grads, *batch, dlogits, drop, stream);
}

extern "C" int gcs_model_backward(const gcs_model_config* cfg, const float* params, const gcs_batch* batch,
                                  const float* dlogits, float* grads, void* workspace, int64_t workspace_bytes,
                                  gcs_stream stream) {
  return gcs_model_backward_ex(cfg, params, batch, dlogits, grads, workspace, workspace_bytes, stream, nullptr);
}

// Test hook (not part of the drop-in surface): where a training-mode forward leaves block `block`'s pre-BatchNorm output
// h [rows, width] and its statistics (mean | var | scale | shift, width floats each) inside the workspace (byte offsets).
extern "C" int gcs_model_debug_block_buffers(const gcs_model_config* cfg, int64_t n_nodes, int32_t n_graphs, int32_t block,
                                             int64_t* h_offset, int64_t* stat_offset, int64_t* rows, int32_t* width) {
  GCS_TRY(check_config(cfg));
  GCS_CHECK_ARG(h_offset && stat_offset && rows && width, "gcs_model_debug_block_buffers: null pointer");
  Plan p;
  int64_t total = 0;
  char* const base = reinterpret_cast<char*>(256);
  make_plan(*cfg, n_nodes, n_graphs, true, base, p, &total);
  GCS_CHECK_ARG(block >= 0 && block < static_cast<int>(p.blocks.size()), "gcs_model_debug_block_buffers: no such block");
  const int node_blocks = p.P + p.L;
  const float* h = block < node_blocks ? p.h[block] : p.post_h[block - node_blocks];
  *h_offset = reinterpret_cast<const char*>(h) - base;
  *stat_offset = reinterpret_cast<const char*>(p.stat[block]) - base;
  *rows = block < node_blocks ? n_nodes : p.rows_post;
  *width = p.blocks[block].m_out;
  return GCS_OK;
}

// Test hook (not part of the drop-in surface): the keep mask of dense block `block` in step `step`, out[r, c] = 1 where
// element (r, c) is kept, from the same device function the kernels apply (dropout.cuh).  threshold = 0 for rate 0.
namespace gcs {
__global__ void dropout_keep_kernel(Dropout d, int64_t M, int C, uint8_t* __restrict__ out) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= M * C) return;
  const int64_t r = i / C;
  const int c = static_cast<int>(i - r * C);
  out[i] = static_cast<uint8_t>((dropout_keep4(d, r, c >> 2) >> (c & 3)) & 1u);
}
}  // namespace gcs

extern "C" int gcs_debug_dropout_keep(uint64_t seed, uint64_t step, int32_t block, int64_t rows, int32_t cols, float rate,
                                      uint8_t* out, gcs_stream stream) {
  GCS_CHECK_ARG(out && rows >= 0 && cols > 0 && block >= 0, "gcs_debug_dropout_keep: bad argument");
  GCS_CHECK_ARG(rate >= 0.f && rate < 1.f, "gcs_debug_dropout_keep: rate must be in [0, 1)");
  if (rows == 0) return GCS_OK;
  const gcs::Dropout d = gcs::make_dropout(rate, seed, step, block);
  const int64_t n = rows * cols;
  gcs::dropout_keep_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, gcs::as_stream(stream)>>>(d, rows, cols, out);
  GCS_CHECK_LAUNCH("dropout_keep_kernel");
  return GCS_OK;
}
