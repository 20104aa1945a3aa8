// K5 — the loss heads of the model, forward and the gradient w.r.t. the logits, with loss_acc = {loss, metric}:
//   softmax + CategoricalCrossentropy + categorical_accuracy (reference: src/scripts/gcn.py:326 loss_fn, :335 loss,
//   :339 accuracy; SURVEY.md §8 a10).  Keras recovers the logits of the softmax and evaluates
//   softmax_cross_entropy_with_logits per row:
//     loss_b = logsumexp(z_b) * sum(y_b) - y_b . z_b ;  loss = mean_b loss_b
//            (evaluated as log(sum exp(z - m)) * sum(y) - y . (z - m), m = max z)
//     dz_b   = (softmax(z_b) * sum(y_b) - y_b) * grad_scale
//   sigmoid + BinaryCrossentropy + binary_accuracy (binary and multi-label targets), per element
//   (sigmoid_cross_entropy_with_logits):
//     l = max(z, 0) - z*y + log1p(exp(-|z|))   acc = mean(y == (p > 0.5))   dz = (p - y) * grad_scale / C
//   MeanSquaredError / MeanAbsoluteError / Huber of a linear head, metric mean_absolute_error; with e = z - y:
//     MSE    l = e^2                                              dl/dz = 2e
//     MAE    l = |e|                                              dl/dz = sign(e)   (sign(0) = 0, as in TF)
//     Huber  l = 0.5 e^2 if |e| <= delta, else delta|e| - 0.5 delta^2   dl/dz = e, or delta sign(e)
//     mae = mean(|e|)   dz = dl/dz * grad_scale / C
//   The elementwise losses are the mean over the C columns, then over the rows: sum(l) / (rows * C).
// One kernel body serves every loss (loss_kernel<Policy>).  A thread walks its items grid-stride - a row for the
// softmax, a unit of four elements of the flat [rows * C] array for the others - with fp32 math per item and fp64 sums
// per thread; the block adds {loss, metric} in a fixed-order tree.  A grid of one block writes loss_acc itself;
// otherwise the per-block partials go to a workspace that loss_finish_kernel adds in a fixed order.  The grid size
// depends on the problem size alone and there are no atomics, so every result is bit-identical run to run.
// With per-row sample weights w (the weighted policies, gcs_weighted_loss), as Keras' sample_weight with the default
// "sum_over_batch_size" reduction: loss = sum_r w_r l_r / rows, dz_r = w_r * dz_r, and the metric is the weighted mean
// sum w m / sum w (0 when sum w = 0).  Each block then adds {sum w l, sum w m, sum w} in fp64 (WSums), in the same
// fixed-order tree.
#include <cmath>

#include "common.cuh"

namespace gcs {

constexpr int kMaxClasses = 64;
constexpr int64_t kXentGridThreshold = 65536;   // rows above which gcs_softmax_xent_ws runs a grid of blocks
constexpr int kXentMaxBlocks = 1024;
constexpr int kElemMaxBlocks = 6 * 148;         // one wave of 6 resident blocks per SM (at <= 40 registers) on a
                                                // B200's 148 SMs; a constant, not the device's count
constexpr int kFinishThreads = 1024;            // one partial per finish thread
static_assert(kXentMaxBlocks <= kFinishThreads && kElemMaxBlocks <= kFinishThreads, "one partial per finish thread");

enum { kRegMse = 1, kRegMae = 2, kRegHuber = 3 };

struct LossArgs {
  const float* logits;
  const float* y;         // NULL: probabilities / predictions only
  float* probs;
  float* dlogits;
  int64_t n;              // what the loss is the mean over: rows for the softmax, rows * C elements otherwise
  int C;
  float scale;            // gradient scale: grad_scale for the softmax, grad_scale / C otherwise
  float delta = 0.f;      // Huber's delta
  bool vec = false;       // every pointer is 16-byte aligned: the unit walk uses 128-bit accesses (set by launch_loss)
};

// The arguments of the weighted policies.  The weight pointer lives in this extension rather than in LossArgs itself, so
// that the unweighted kernels keep their parameter layout and compiled code.
struct WLossArgs : LossArgs {
  const float* w;         // [rows] one weight per row (read with scalar loads; any alignment)
};

// One row b: writes probs / dlogits, adds the row's loss and hit to loss / hit (when y != NULL).  W: the row has weight
// w, which multiplies its loss (in fp64) and its dlogits, after the unweighted expression (exact for w = 1).
template <bool W = false>
__device__ __forceinline__ void xent_row(const LossArgs& a, int64_t b, double& loss, int& hit, float w = 1.f) {
  const int C = a.C;
  const float* z = a.logits + b * C;
  float m = z[0];
  int arg_p = 0;
  for (int c = 1; c < C; ++c)
    if (z[c] > m) { m = z[c]; arg_p = c; }       // first maximum, like tf.argmax
  float e[kMaxClasses];
  float rest = 0.f;                                // sum over c != argmax; e[argmax] = 1 exactly
  for (int c = 0; c < C; ++c) {
    e[c] = expf(z[c] - m);
    if (c != arg_p) rest += e[c];
  }
  const float sum = 1.0f + rest;
  const float log_sum = log1pf(rest);              // lse = m + log_sum, accurate for confident rows
  const float inv = 1.0f / sum;
  float ysum = 0.f, yz = 0.f, ymax = 0.f;
  int arg_y = 0;
  if (a.y) {
    const float* yy = a.y + b * C;
    ymax = yy[0];
    for (int c = 0; c < C; ++c) {
      ysum += yy[c];
      yz = fmaf(yy[c], z[c] - m, yz);            // y . (z - m): no cancellation against lse
      if (c > 0 && yy[c] > ymax) { ymax = yy[c]; arg_y = c; }
    }
    if (W) loss += static_cast<double>(log_sum * ysum - yz) * static_cast<double>(w);
    else loss += static_cast<double>(log_sum * ysum - yz);
    hit += (arg_y == arg_p);
  }
  for (int c = 0; c < C; ++c) {
    const float p = e[c] * inv;
    if (a.probs) a.probs[b * C + c] = p;
    if (a.dlogits) {
      if (W) a.dlogits[b * C + c] = (p * ysum - a.y[b * C + c]) * a.scale * w;
      else a.dlogits[b * C + c] = (p * ysum - a.y[b * C + c]) * a.scale;
    }
  }
}

// The metric of one unit of four, m[k] being element k's.  A hit count needs no order: the four elements add to one
// counter.  fp32 values get a slot each and are added as (v0 + v1) + (v2 + v3), like the loss.
struct UnitCount {
  int n = 0;
  __device__ int& operator[](int) { return n; }
  __device__ int total() const { return n; }
};
struct UnitSum {
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  __device__ float& operator[](int k) { return v[k]; }
  __device__ float total() const { return (v[0] + v[1]) + (v[2] + v[3]); }
};

// One element of the sigmoid head: out = sigmoid(z); with labels also dz, the hit (added to hit) and the element's
// loss (returned, 0 without labels).  One exp per element: e = exp(-|z|) gives both log1p(e) and p = 1/(1+e) or
// e/(1+e), finite for any z.
struct BceElem {
  using Unit = UnitCount;
  static constexpr bool kNeedsY = false;
  __device__ __forceinline__ static float elem(float z, float yv, bool want_y, const LossArgs& a, float& out, float& dz,
                                               int& hit) {
    const float e = expf(-fabsf(z));
    const float inv = 1.0f / (1.0f + e);
    out = z >= 0.f ? inv : e * inv;
    if (!want_y) return 0.f;
    hit += (yv == (out > 0.5f ? 1.0f : 0.0f));
    dz = (out - yv) * a.scale;
    return fmaf(-z, yv, fmaxf(z, 0.f)) + log1pf(e);
  }
};

// One element of a regression loss (only run with targets): out = z; returns the loss, leaves dz and |e| in ae.
template <int KIND>
struct RegElem {
  using Unit = UnitSum;
  static constexpr bool kNeedsY = true;            // the host copies the predictions itself when y is NULL
  __device__ __forceinline__ static float elem(float z, float yv, bool, const LossArgs& a, float& out, float& dz,
                                               float& ae) {
    out = z;
    const float e = z - yv;
    const float abs_e = fabsf(e);
    const float sgn = e > 0.f ? 1.f : (e < 0.f ? -1.f : 0.f);
    ae = abs_e;
    if (KIND == kRegMse) {
      dz = (2.f * e) * a.scale;
      return e * e;
    }
    if (KIND == kRegMae) {
      dz = sgn * a.scale;
      return abs_e;
    }
    if (abs_e <= a.delta) {
      dz = e * a.scale;
      return 0.5f * e * e;
    }
    dz = (a.delta * sgn) * a.scale;
    return a.delta * abs_e - 0.5f * a.delta * a.delta;
  }
};

// Unit u = elements [4u, min(4u + 4, n)): one 128-bit access per operand when a.vec allows it, otherwise scalar
// accesses of the same four elements, so the sums do not depend on alignment.  Each branch adds its own unit sums next
// to the element math, which keeps the compiler's contraction of e.g. MSE's e0 * e0 + e1 * e1 into one FFMA.
template <class E, class Metric>
__device__ __forceinline__ void unit_walk(const LossArgs& a, int64_t u, double& loss, Metric& metric) {
  const bool want_y = E::kNeedsY || a.y != nullptr;
  const int64_t i0 = u << 2;
  typename E::Unit m;
  if (a.vec && i0 + 4 <= a.n) {
    const float4 z = *reinterpret_cast<const float4*>(a.logits + i0);
    const float4 yv = want_y ? *reinterpret_cast<const float4*>(a.y + i0) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 o, d;
    const float l0 = E::elem(z.x, yv.x, want_y, a, o.x, d.x, m[0]);
    const float l1 = E::elem(z.y, yv.y, want_y, a, o.y, d.y, m[1]);
    const float l2 = E::elem(z.z, yv.z, want_y, a, o.z, d.z, m[2]);
    const float l3 = E::elem(z.w, yv.w, want_y, a, o.w, d.w, m[3]);
    loss += static_cast<double>((l0 + l1) + (l2 + l3));
    metric += m.total();
    if (a.probs) *reinterpret_cast<float4*>(a.probs + i0) = o;
    if (a.dlogits) *reinterpret_cast<float4*>(a.dlogits + i0) = d;
  } else {
    float l[4] = {0.f, 0.f, 0.f, 0.f};               // the vector path's order of the four additions
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (i0 + k >= a.n) break;
      float o, d;
      l[k] = E::elem(a.logits[i0 + k], want_y ? a.y[i0 + k] : 0.f, want_y, a, o, d, m[k]);
      if (a.probs) a.probs[i0 + k] = o;
      if (a.dlogits) a.dlogits[i0 + k] = d;
    }
    loss += static_cast<double>((l[0] + l[1]) + (l[2] + l[3]));
    metric += m.total();
  }
}

// {sum of w * metric, sum of w} of the weighted policies, per thread and per block (fp64).
struct WSums {
  double m, w;
  WSums() = default;                               // trivial: block_reduce keeps an array of them in shared memory
  __device__ WSums(int zero) : m(zero), w(zero) {}
  __device__ WSums& operator+=(const WSums& o) {
    m += o.m;
    w += o.w;
    return *this;
  }
};

// The weighted unit u.  When its elements all carry the same weight w0 (every unit of a row when C % 4 == 0; any unit
// when the weights agree) it is unit_walk itself on a gradient scale of scale * w0, and its sums times w0 in fp64: with
// w0 = 1 loss, dlogits and metric are the unweighted kernel's bits.  A unit that spans rows of different weights takes
// each element alone, with scalar accesses.
template <class E, class Acc>
__device__ __forceinline__ void unit_walk_weighted(const WLossArgs& a, int64_t u, double& loss, WSums& ws) {
  const int64_t i0 = u << 2;
  const int cnt = a.n - i0 < 4 ? static_cast<int>(a.n - i0) : 4;
  const int64_t r0 = i0 / a.C;
  const int c0 = static_cast<int>(i0 - r0 * a.C);
  float w[4];
  bool same = true;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    w[k] = k < cnt ? a.w[r0 + (c0 + k) / a.C] : 0.f;
    same = same && (k >= cnt || w[k] == w[0]);
  }
  if (same) {
    LossArgs b = a;
    b.scale = a.scale * w[0];
    double l = 0.0;
    Acc m = 0;
    unit_walk<E>(b, u, l, m);
    loss += l * static_cast<double>(w[0]);
    ws.m += static_cast<double>(m) * static_cast<double>(w[0]);
    ws.w += static_cast<double>(cnt) * static_cast<double>(w[0]);
    return;
  }
  float wl[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k >= cnt) break;
    const int64_t i = i0 + k;
    LossArgs b = a;
    b.scale = a.scale * w[k];
    typename E::Unit m;
    float o, d;
    wl[k] = E::elem(a.logits[i], a.y[i], true, b, o, d, m[0]) * w[k];
    if (a.probs) a.probs[i] = o;
    if (a.dlogits) a.dlogits[i] = d;
    ws.m += static_cast<double>(m.total()) * static_cast<double>(w[k]);
    ws.w += static_cast<double>(w[k]);
  }
  loss += static_cast<double>((wl[0] + wl[1]) + (wl[2] + wl[3]));
}

// loss_acc from the block sums (n > 0).  The sums are taken by reference: thread 0 reads each from shared memory
// where it is used, which keeps the kernels at their register counts.
struct XentFinish {
  using Metric = int;                              // hit count, per thread and per block
  using Acc = int;
  __device__ static void finish(const double& s, const int& hits, int64_t rows, float* loss_acc) {
    loss_acc[0] = static_cast<float>(s / static_cast<double>(rows));
    loss_acc[1] = static_cast<float>(hits) / static_cast<float>(rows);
  }
};

template <class M, class A>                        // per block M, per thread A: hit counts (sigmoid) or sums of |e|
struct MeanFinish {
  using Metric = M;
  using Acc = A;
  __device__ static void finish(const double& s, const M& m, int64_t n, float* loss_acc) {
    loss_acc[0] = static_cast<float>(s / static_cast<double>(n));
    loss_acc[1] = static_cast<float>(static_cast<double>(m) / static_cast<double>(n));
  }
};

// The weighted policies: loss = sum w l / n (n = rows, or rows * C: the mean over the columns is inside), metric =
// sum w m / sum w, or 0 when sum w = 0.
struct WeightedFinish {
  using Metric = WSums;
  using Acc = WSums;
  __device__ static void finish(const double& s, const WSums& m, int64_t n, float* loss_acc) {
    loss_acc[0] = static_cast<float>(s / static_cast<double>(n));
    loss_acc[1] = m.w != 0.0 ? static_cast<float>(m.m / m.w) : 0.f;
  }
};

// Policies of loss_kernel: block size, minimum resident blocks (0: no bound), most blocks of a grid, the kernel's
// arguments (Args), the elements of an item (a row for the softmax, whose n counts rows), one item, and the finish.
// W selects the weighted form of a policy.
template <int THREADS, int MAX_BLOCKS, bool W = false>
struct Xent {
  static constexpr int kThreads = THREADS, kMinBlocks = 0, kMaxBlocks = MAX_BLOCKS, kItem = 1;
  using Args = LossArgs;
  using Finish = XentFinish;
  __device__ static void item(const LossArgs& a, int64_t b, double& loss, int& hit) { xent_row(a, b, loss, hit); }
};
template <int THREADS, int MAX_BLOCKS>
struct Xent<THREADS, MAX_BLOCKS, true> {
  static constexpr int kThreads = THREADS, kMinBlocks = 0, kMaxBlocks = MAX_BLOCKS, kItem = 1;
  using Args = WLossArgs;
  using Finish = WeightedFinish;
  __device__ static void item(const WLossArgs& a, int64_t b, double& loss, WSums& ws) {
    const float w = a.w[b];
    int hit = 0;
    xent_row<true>(a, b, loss, hit, w);
    if (hit) ws.m += static_cast<double>(w);
    ws.w += static_cast<double>(w);
  }
};
using XentBlock = Xent<1024, 1>;                   // gcs_softmax_xent: one block for any row count
using XentGrid = Xent<256, kXentMaxBlocks>;        // gcs_softmax_xent_ws above kXentGridThreshold rows
using XentBlockW = Xent<1024, 1, true>;            // gcs_weighted_loss, the same rule
using XentGridW = Xent<256, kXentMaxBlocks, true>;

template <class E, class F, bool W = false>
struct Elementwise {
  static constexpr int kThreads = 256, kMinBlocks = 6, kMaxBlocks = kElemMaxBlocks, kItem = 4;
  using Args = LossArgs;
  using Finish = F;
  __device__ static void item(const LossArgs& a, int64_t u, double& loss, typename F::Acc& m) {
    unit_walk<E>(a, u, loss, m);
  }
};
template <class E, class F>                        // F: the unweighted finish, whose per-thread metric a unit produces
struct Elementwise<E, F, true> {
  static constexpr int kThreads = 256, kMinBlocks = 0, kMaxBlocks = kElemMaxBlocks, kItem = 4;
  using Args = WLossArgs;
  using Finish = WeightedFinish;
  __device__ static void item(const WLossArgs& a, int64_t u, double& loss, WSums& ws) {
    unit_walk_weighted<E, typename F::Acc>(a, u, loss, ws);
  }
};
using Bce = Elementwise<BceElem, MeanFinish<long long, int>>;
template <int KIND>
using Reg = Elementwise<RegElem<KIND>, MeanFinish<double, double>>;
using BceW = Elementwise<BceElem, MeanFinish<long long, int>, true>;
template <int KIND>
using RegW = Elementwise<RegElem<KIND>, MeanFinish<double, double>, true>;

template <int THREADS, class M>
struct BlockSums {
  double loss[THREADS];
  M m[THREADS];
};

// Fixed-order tree over the block of {loss, m}; the block's sums end in loss[0], m[0].
template <int THREADS, class M>
__device__ __forceinline__ const BlockSums<THREADS, M>& block_reduce(double loss, M m) {
  __shared__ BlockSums<THREADS, M> s;
  const int t = threadIdx.x;
  s.loss[t] = loss;
  s.m[t] = m;
  __syncthreads();
  for (int off = THREADS >> 1; off > 0; off >>= 1) {
    if (t < off) {
      s.loss[t] += s.loss[t + off];
      s.m[t] += s.m[t + off];
    }
    __syncthreads();
  }
  return s;
}

template <class F>
__device__ __forceinline__ void write_loss_acc(const double& s, const typename F::Metric& m, int64_t n,
                                               float* loss_acc) {
  if (n > 0) {
    F::finish(s, m, n, loss_acc);
  } else {
    loss_acc[0] = 0.f;
    loss_acc[1] = 0.f;
  }
}

// Items i = blockIdx.x * blockDim.x + threadIdx.x + k * gridDim.x * blockDim.x, elements [i * kItem, ...).  The
// block's sums go to loss_acc (a grid of one block) or to part_loss / part_m[blockIdx.x].
template <class P>
__global__ void __launch_bounds__(P::kThreads, P::kMinBlocks) loss_kernel(
    const typename P::Args a, double* __restrict__ part_loss, typename P::Finish::Metric* __restrict__ part_m,
    float* __restrict__ loss_acc) {
  double loss = 0.0;
  typename P::Finish::Acc m = 0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * P::kThreads;
#pragma unroll 1                                   // unrolled, the one-block softmax kernel spills
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * P::kThreads + threadIdx.x; i * P::kItem < a.n; i += stride)
    P::item(a, i, loss, m);
  if (!part_loss && !loss_acc) return;
  const auto& s = block_reduce<P::kThreads, typename P::Finish::Metric>(loss, m);
  if (threadIdx.x == 0) {
    if (loss_acc) {
      write_loss_acc<typename P::Finish>(s.loss[0], s.m[0], a.n, loss_acc);
    } else {
      part_loss[blockIdx.x] = s.loss[0];
      part_m[blockIdx.x] = s.m[0];
    }
  }
}

// One thread per partial (n_parts <= kFinishThreads), zero-padded, fixed-order tree sum; n = 0 gives {0, 0}.
template <class F>
__global__ void __launch_bounds__(kFinishThreads) loss_finish_kernel(
    const double* __restrict__ part_loss, const typename F::Metric* __restrict__ part_m, int n_parts, int64_t n,
    float* __restrict__ loss_acc) {
  const int t = threadIdx.x;
  const auto& s = block_reduce<kFinishThreads>(t < n_parts ? part_loss[t] : 0.0,
                                               t < n_parts ? part_m[t] : typename F::Metric(0));
  if (t == 0) write_loss_acc<F>(s.loss[0], s.m[0], n, loss_acc);
}

// The grid: a count that depends on n alone; 0 when there is nothing to walk, except that a policy of one block runs
// its block for any n (gcs_softmax_xent writes loss_acc = {0, 0} for B = 0 from its own kernel).
template <class P>
static int grid_blocks(int64_t n) {
  if (P::kMaxBlocks == 1) return 1;
  const int64_t blocks = ceil_div(ceil_div(n, P::kItem), static_cast<int64_t>(P::kThreads));
  return static_cast<int>(blocks < P::kMaxBlocks ? blocks : P::kMaxBlocks);
}

// Bytes of the partials: the fp64 loss sums of the grid's blocks, then their metrics; none for a grid of one block.
template <class P>
static int64_t partial_bytes(int64_t n) {
  const int blocks = grid_blocks<P>(n);
  return blocks > 1 ? static_cast<int64_t>(blocks) * (sizeof(double) + sizeof(typename P::Finish::Metric)) : 0;
}

// Runs loss_kernel<P> and, for a grid of several blocks with loss_acc requested, loss_finish_kernel<P> over the
// partials in `workspace`; with nothing to walk only the finish kernel, for loss_acc = {0, 0}.
template <class P>
static int launch_loss(const char* who, typename P::Args a, float* loss_acc, void* workspace, int64_t workspace_bytes,
                       cudaStream_t st) {
  const int blocks = grid_blocks<P>(a.n);
  double* part_loss = nullptr;
  using F = typename P::Finish;
  typename F::Metric* part_m = nullptr;
  if (loss_acc && blocks > 1) {
    const int64_t need = partial_bytes<P>(a.n);
    if (!workspace || workspace_bytes < need)
      return fail(GCS_ERR_WORKSPACE, "%s: workspace %lld < %lld bytes", who, (long long)workspace_bytes,
                  (long long)need);
    GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 7u) == 0, "%s: workspace must be 8-byte aligned", who);
    part_loss = static_cast<double*>(workspace);
    part_m = reinterpret_cast<typename F::Metric*>(part_loss + blocks);
  }
  if (blocks == 0) {
    if (loss_acc) {
      loss_finish_kernel<F><<<1, kFinishThreads, 0, st>>>(nullptr, nullptr, 0, 0, loss_acc);
      GCS_CHECK_LAUNCH("loss_finish_kernel");
    }
    return GCS_OK;
  }
  a.vec = aligned16(a.logits) && aligned16(a.y) && aligned16(a.probs) && aligned16(a.dlogits);
  loss_kernel<P><<<blocks, P::kThreads, 0, st>>>(a, part_loss, part_m, blocks == 1 ? loss_acc : nullptr);
  GCS_CHECK_LAUNCH("loss_kernel");
  if (part_loss) {
    loss_finish_kernel<F><<<1, kFinishThreads, 0, st>>>(part_loss, part_m, blocks, a.n, loss_acc);
    GCS_CHECK_LAUNCH("loss_finish_kernel");
  }
  return GCS_OK;
}

static bool elementwise_size_ok(int64_t rows, int32_t C) { return rows >= 0 && C >= 1 && rows <= INT64_MAX / C; }

}  // namespace gcs

using namespace gcs;

extern "C" int gcs_softmax_xent(const float* logits, const float* y, int32_t B, int32_t C, float* probs,
                                float* loss_acc, float* dlogits, float grad_scale, gcs_stream stream) {
  GCS_CHECK_ARG(B >= 0 && C > 0 && C <= kMaxClasses, "gcs_softmax_xent: C=%d outside [1, %d]", C, kMaxClasses);
  GCS_CHECK_ARG(logits || B == 0, "gcs_softmax_xent: null logits");
  GCS_CHECK_ARG(y || (!dlogits && !loss_acc), "gcs_softmax_xent: loss / gradient requested without labels");
  return launch_loss<XentBlock>("gcs_softmax_xent", {logits, y, probs, dlogits, B, C, grad_scale}, loss_acc, nullptr, 0,
                                as_stream(stream));
}

extern "C" int64_t gcs_softmax_xent_workspace_bytes(int64_t B, int32_t C) {
  (void)C;
  if (B < 0) return -1;
  return B <= kXentGridThreshold ? 0 : partial_bytes<XentGrid>(B);
}

extern "C" int gcs_softmax_xent_ws(const float* logits, const float* y, int32_t B, int32_t C, float* probs,
                                   float* loss_acc, float* dlogits, float grad_scale, void* workspace,
                                   int64_t workspace_bytes, gcs_stream stream) {
  if (B <= kXentGridThreshold)
    return gcs_softmax_xent(logits, y, B, C, probs, loss_acc, dlogits, grad_scale, stream);
  GCS_CHECK_ARG(C > 0 && C <= kMaxClasses, "gcs_softmax_xent_ws: C=%d outside [1, %d]", C, kMaxClasses);
  GCS_CHECK_ARG(logits, "gcs_softmax_xent_ws: null logits");
  GCS_CHECK_ARG(y || (!dlogits && !loss_acc), "gcs_softmax_xent_ws: loss / gradient requested without labels");
  return launch_loss<XentGrid>("gcs_softmax_xent_ws", {logits, y, probs, dlogits, B, C, grad_scale}, loss_acc,
                               workspace, workspace_bytes, as_stream(stream));
}

extern "C" int64_t gcs_sigmoid_bce_workspace_bytes(int64_t rows, int32_t C) {
  return elementwise_size_ok(rows, C) ? partial_bytes<Bce>(rows * C) : -1;
}

extern "C" int gcs_sigmoid_bce(const float* logits, const float* y, int64_t rows, int32_t C, float* probs,
                               float* loss_acc, float* dlogits, float grad_scale, void* workspace,
                               int64_t workspace_bytes, gcs_stream stream) {
  GCS_CHECK_ARG(elementwise_size_ok(rows, C), "gcs_sigmoid_bce: rows=%lld, C=%d", (long long)rows, C);
  GCS_CHECK_ARG(logits || rows == 0, "gcs_sigmoid_bce: null logits");
  GCS_CHECK_ARG(y || (!dlogits && !loss_acc), "gcs_sigmoid_bce: loss / gradient requested without labels");
  const LossArgs a{logits, y, probs, dlogits, rows * C, C, grad_scale / static_cast<float>(C)};
  return launch_loss<Bce>("gcs_sigmoid_bce", a, loss_acc, workspace, workspace_bytes, as_stream(stream));
}

extern "C" int64_t gcs_regression_loss_workspace_bytes(int64_t rows, int32_t C) {
  return elementwise_size_ok(rows, C) ? partial_bytes<Reg<kRegMse>>(rows * C) : -1;   // the same for every kind
}

extern "C" int gcs_regression_loss(int32_t kind, float huber_delta, const float* pred, const float* y, int64_t rows,
                                   int32_t C, float* probs, float* loss_acc, float* dlogits, float grad_scale,
                                   void* workspace, int64_t workspace_bytes, gcs_stream stream) {
  GCS_CHECK_ARG(kind >= kRegMse && kind <= kRegHuber, "gcs_regression_loss: kind=%d (1 = MSE, 2 = MAE, 3 = Huber)",
                kind);
  GCS_CHECK_ARG(kind != kRegHuber || (std::isfinite(huber_delta) && huber_delta > 0.f),
                "gcs_regression_loss: huber_delta must be finite and > 0, got %g", static_cast<double>(huber_delta));
  GCS_CHECK_ARG(elementwise_size_ok(rows, C), "gcs_regression_loss: rows=%lld, C=%d", (long long)rows, C);
  GCS_CHECK_ARG(pred || rows == 0, "gcs_regression_loss: null predictions");
  GCS_CHECK_ARG(y || (!dlogits && !loss_acc), "gcs_regression_loss: loss / gradient requested without targets");
  const LossArgs a{pred, y, probs, dlogits, rows * C, C, grad_scale / static_cast<float>(C), huber_delta};
  cudaStream_t st = as_stream(stream);
  if (!y) {                                          // predictions only: a linear head's output is its input
    if (probs && probs != pred && a.n > 0)
      GCS_CUDA(cudaMemcpyAsync(probs, pred, sizeof(float) * a.n, cudaMemcpyDeviceToDevice, st));
    return GCS_OK;
  }
  const char* who = "gcs_regression_loss";
  if (kind == kRegMse) return launch_loss<Reg<kRegMse>>(who, a, loss_acc, workspace, workspace_bytes, st);
  if (kind == kRegMae) return launch_loss<Reg<kRegMae>>(who, a, loss_acc, workspace, workspace_bytes, st);
  return launch_loss<Reg<kRegHuber>>(who, a, loss_acc, workspace, workspace_bytes, st);
}

// head: gcs_model_config.final_activation codes (0 = linear with a regression loss, 1 = softmax, 2 = sigmoid).
extern "C" int64_t gcs_weighted_loss_workspace_bytes(int32_t head, int64_t rows, int32_t C) {
  if (head < 0 || head > 2 || !elementwise_size_ok(rows, C)) return -1;
  if (head == 1) return rows <= kXentGridThreshold ? 0 : partial_bytes<XentGridW>(rows);
  return partial_bytes<BceW>(rows * C);                                  // the same for every elementwise head
}

extern "C" int gcs_weighted_loss(int32_t head, int32_t kind, float huber_delta, const float* logits, const float* y,
                                 const float* sample_weight, int64_t rows, int32_t C, float* probs, float* loss_acc,
                                 float* dlogits, float grad_scale, void* workspace, int64_t workspace_bytes,
                                 gcs_stream stream) {
  const char* who = "gcs_weighted_loss";
  GCS_CHECK_ARG(head >= 0 && head <= 2, "%s: head=%d (0 = linear, 1 = softmax, 2 = sigmoid)", who, head);
  GCS_CHECK_ARG(head != 0 || (kind >= kRegMse && kind <= kRegHuber), "%s: kind=%d (1 = MSE, 2 = MAE, 3 = Huber)", who,
                kind);
  GCS_CHECK_ARG(head != 0 || kind != kRegHuber || (std::isfinite(huber_delta) && huber_delta > 0.f),
                "%s: huber_delta must be finite and > 0, got %g", who, static_cast<double>(huber_delta));
  GCS_CHECK_ARG(elementwise_size_ok(rows, C), "%s: rows=%lld, C=%d", who, (long long)rows, C);
  GCS_CHECK_ARG(head != 1 || C <= kMaxClasses, "%s: softmax C=%d outside [1, %d]", who, C, kMaxClasses);
  GCS_CHECK_ARG(sample_weight, "%s: null sample_weight (the unweighted entry points take no weights)", who);
  GCS_CHECK_ARG((logits && y) || rows == 0, "%s: null logits or labels", who);
  cudaStream_t st = as_stream(stream);
  WLossArgs a;
  static_cast<LossArgs&>(a) = LossArgs{logits, y, probs, dlogits, rows, C, grad_scale};
  a.w = sample_weight;
  if (head == 1) {
    if (rows <= kXentGridThreshold) return launch_loss<XentBlockW>(who, a, loss_acc, workspace, workspace_bytes, st);
    return launch_loss<XentGridW>(who, a, loss_acc, workspace, workspace_bytes, st);
  }
  a.n = rows * C;
  a.scale = grad_scale / static_cast<float>(C);
  if (head == 2) return launch_loss<BceW>(who, a, loss_acc, workspace, workspace_bytes, st);
  a.delta = huber_delta;
  if (kind == kRegMse) return launch_loss<RegW<kRegMse>>(who, a, loss_acc, workspace, workspace_bytes, st);
  if (kind == kRegMae) return launch_loss<RegW<kRegMae>>(who, a, loss_acc, workspace, workspace_bytes, st);
  return launch_loss<RegW<kRegHuber>>(who, a, loss_acc, workspace, workspace_bytes, st);
}
