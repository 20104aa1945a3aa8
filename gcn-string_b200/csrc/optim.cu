// K10 — fused multi-tensor optimizer steps over the flat parameter buffer.
//   SGD  (what the reference runs: tf.keras.optimizers.SGD, src/scripts/gcn.py:325,338):
//        w <- w - lr * g
//   SGD with momentum (Keras ResourceApplyKerasMomentum), slot accum:
//        accum <- momentum accum - lr g ; w <- w + accum     (nesterov: w <- w + momentum accum - lr g)
//   Adam (Keras semantics, what the upstream example the script derives from uses and what
//        BASELINE.json's north_star names; SURVEY.md §8 a11):
//        m <- b1 m + (1-b1) g ; v <- b2 v + (1-b2) g^2 ; lr_t = lr sqrt(1-b2^t)/(1-b1^t)
//        w <- w - lr_t m / (sqrt(v) + eps)            (eps OUTSIDE the corrected root)
//        amsgrad: vhat <- max(vhat, v) ; w <- w - lr_t m / (sqrt(vhat) + eps)
// grad_scale folds the 1/world_size (or count weighting) after the NCCL all-reduce in.
//
// Gradient clipping (Keras clipvalue, clipnorm, global_clipnorm) acts on g * grad_scale, in that order: clipvalue
// clamps each element, then the norm factor scales it.  Norms come from a chunk table over the flat buffer (no chunk
// crosses a tensor): clip_partials_kernel writes one fp64 sum of squares per chunk, then every block of the update
// kernel takes one chunk and sums the partials it needs (its tensor's chunks, or all of them) in a fixed order.
// Two launches, no atomics, no host synchronisation; every block of a tensor forms the same factor bit for bit.
#include "common.cuh"

#include <math.h>

namespace gcs {

constexpr int kOptThreads = 256;
enum NormKind { kNoNorm = 0, kTensorNorm = 1, kGlobalNorm = 2 };

struct ClipArgs {
  float value;               // clipvalue bound
  float norm;                // clipnorm / global_clipnorm threshold
  const int64_t* rows;       // [n_chunks][4]: begin, end, lo, hi
  double* partials;          // row k of this call owns partials[base + k]
  int32_t base;
  int32_t n_partials;        // global norm: partials[0, n_partials)
};

// Comparisons rather than fminf / fmaxf, so that a NaN stays NaN instead of becoming a bound.
__device__ __forceinline__ float clip_value(float x, float v) { return x > v ? v : (x < -v ? -v : x); }

template <bool CLIPV>
__device__ __forceinline__ float scaled_grad(const float* __restrict__ g, int64_t k, float grad_scale,
                                             const ClipArgs& c) {
  const float x = g[k] * grad_scale;
  return CLIPV ? clip_value(x, c.value) : x;
}

// Fixed-order block sum: shuffle tree inside each warp, then thread 0 adds the warp sums in order.  Valid in thread 0.
__device__ __forceinline__ double block_sum(double x) {
  __shared__ double warp_sums[kOptThreads / 32];
  for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = x;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kOptThreads / 32; ++w) s += warp_sums[w];
  return s;
}

// One block per chunk: sum of squares of clipvalue(g * grad_scale) over [begin, end).
template <bool CLIPV>
__global__ void __launch_bounds__(kOptThreads) clip_partials_kernel(const float* __restrict__ g, float grad_scale,
                                                                    ClipArgs c) {
  const int64_t* r = c.rows + 4 * static_cast<int64_t>(blockIdx.x);
  const int64_t end = r[1];
  double s = 0.0;
  for (int64_t k = r[0] + threadIdx.x; k < end; k += kOptThreads) {
    const double x = scaled_grad<CLIPV>(g, k, grad_scale, c);
    s += x * x;
  }
  s = block_sum(s);
  if (threadIdx.x == 0) c.partials[c.base + blockIdx.x] = s;
}

// Clip factor from partials[lo, hi): exactly 1 when the norm is <= the threshold, else c / norm (0 for an infinite
// per-tensor norm, NaN for a NaN one).  A global norm that is not finite gives NaN, as tf.clip_by_global_norm.
template <int NORM>
__device__ __forceinline__ float clip_factor(const ClipArgs& c, int64_t lo, int64_t hi) {
  __shared__ float factor;
  double s = 0.0;
  for (int64_t k = lo + threadIdx.x; k < hi; k += kOptThreads) s += c.partials[k];
  s = block_sum(s);
  if (threadIdx.x == 0) {
    const double norm = sqrt(s);
    const double cn = static_cast<double>(c.norm);
    if (NORM == kGlobalNorm && !isfinite(norm))
      factor = __int_as_float(0x7fffffff);
    else
      factor = norm <= cn ? 1.0f : static_cast<float>(cn / norm);
  }
  __syncthreads();
  return factor;
}

// ---- update rules: (k, clipped gradient) -> new w and slots -------------------------------------------------------
enum SgdKind { kPlainSgd = 0, kMomentum = 1, kNesterov = 2 };

template <int KIND>
struct SgdStep {
  float* __restrict__ w;
  float* __restrict__ accum;
  float lr, momentum;
  __device__ __forceinline__ void operator()(int64_t k, float gk) const {
    if (KIND == kPlainSgd) {
      w[k] = w[k] - lr * gk;
    } else {
      const float a = momentum * accum[k] - lr * gk;
      accum[k] = a;
      w[k] = KIND == kNesterov ? w[k] + (momentum * a - lr * gk) : w[k] + a;
    }
  }
};

template <bool AMSGRAD>
struct AdamStep {
  float* __restrict__ w;
  float* __restrict__ m;
  float* __restrict__ v;
  float* __restrict__ vhat;
  float lr_t, beta1, beta2, omb1, omb2, eps;
  __device__ __forceinline__ void operator()(int64_t k, float gk) const {
    const float mk = beta1 * m[k] + omb1 * gk;
    const float vk = beta2 * v[k] + omb2 * gk * gk;
    m[k] = mk;
    v[k] = vk;
    if (AMSGRAD) {
      const float vh = fmaxf(vhat[k], vk);
      vhat[k] = vh;
      w[k] = w[k] - lr_t * mk / (sqrtf(vh) + eps);
    } else {
      w[k] = w[k] - lr_t * mk / (sqrtf(vk) + eps);
    }
  }
};

// Without a norm: grid-stride over [0, n).  With one: block b takes chunk b and forms its factor first.
template <class Step, bool CLIPV, int NORM>
__global__ void __launch_bounds__(kOptThreads) opt_kernel(Step step, const float* __restrict__ g, int64_t n,
                                                          float grad_scale, ClipArgs c) {
  if constexpr (NORM == kNoNorm) {
    for (int64_t k = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; k < n;
         k += static_cast<int64_t>(gridDim.x) * blockDim.x)
      step(k, scaled_grad<CLIPV>(g, k, grad_scale, c));
  } else {
    const int64_t* r = c.rows + 4 * static_cast<int64_t>(blockIdx.x);
    const int64_t end = r[1];
    const float f = NORM == kTensorNorm ? clip_factor<NORM>(c, r[2], r[3]) : clip_factor<NORM>(c, 0, c.n_partials);
    for (int64_t k = r[0] + threadIdx.x; k < end; k += kOptThreads) step(k, scaled_grad<CLIPV>(g, k, grad_scale, c) * f);
  }
}

}  // namespace gcs

using namespace gcs;

static inline unsigned opt_blocks(int64_t n) {
  int64_t b = ceil_div(n, 256);
  const int64_t cap = 8LL * sm_count();
  return static_cast<unsigned>(b < 1 ? 1 : (b > cap ? cap : b));
}

static int check_clip(const gcs_grad_clip* clip, bool need_norm, const char* who) {
  const int mode = clip->mode;
  GCS_CHECK_ARG((mode & ~(GCS_CLIP_VALUE | GCS_CLIP_NORM | GCS_CLIP_GLOBAL_NORM | GCS_CLIP_PARTIALS_READY)) == 0,
                "%s: unknown clip mode bits 0x%x", who, mode);
  GCS_CHECK_ARG(!((mode & GCS_CLIP_NORM) && (mode & GCS_CLIP_GLOBAL_NORM)),
                "%s: GCS_CLIP_NORM and GCS_CLIP_GLOBAL_NORM exclude each other", who);
  GCS_CHECK_ARG(!(mode & GCS_CLIP_VALUE) || clip->clipvalue >= 0.0f, "%s: clipvalue must be >= 0", who);
  const bool norm = mode & (GCS_CLIP_NORM | GCS_CLIP_GLOBAL_NORM);
  GCS_CHECK_ARG(!need_norm || norm, "%s: no norm mode set", who);
  if (norm) {
    GCS_CHECK_ARG(clip->clipnorm >= 0.0f, "%s: clipnorm must be >= 0", who);
    GCS_CHECK_ARG(clip->chunks && clip->partials && clip->n_chunks >= 1 && clip->chunk_base >= 0 &&
                      clip->n_partials >= clip->chunk_base + clip->n_chunks,
                  "%s: bad chunk table (chunks, partials, n_chunks >= 1, chunk_base + n_chunks <= n_partials)", who);
  }
  return GCS_OK;
}

static ClipArgs clip_args(const gcs_grad_clip* clip) {
  if (!clip) return ClipArgs{0.f, 0.f, nullptr, nullptr, 0, 0};
  return ClipArgs{clip->clipvalue, clip->clipnorm, clip->chunks, clip->partials, clip->chunk_base, clip->n_partials};
}

static int launch_partials(const float* g, float grad_scale, const gcs_grad_clip* clip, cudaStream_t st) {
  const ClipArgs c = clip_args(clip);
  if (clip->mode & GCS_CLIP_VALUE)
    clip_partials_kernel<true><<<clip->n_chunks, kOptThreads, 0, st>>>(g, grad_scale, c);
  else
    clip_partials_kernel<false><<<clip->n_chunks, kOptThreads, 0, st>>>(g, grad_scale, c);
  GCS_CHECK_LAUNCH("clip_partials_kernel");
  return GCS_OK;
}

// Optional norm pass, then the update kernel of `step` for the clip options in `clip` (NULL: none).
template <class Step>
static int launch_step(Step step, const float* g, int64_t n, float grad_scale, const gcs_grad_clip* clip,
                       cudaStream_t st) {
  const int mode = clip ? clip->mode : 0;
  const bool cv = mode & GCS_CLIP_VALUE;
  const int norm = (mode & GCS_CLIP_NORM) ? kTensorNorm : (mode & GCS_CLIP_GLOBAL_NORM) ? kGlobalNorm : kNoNorm;
  if (norm != kNoNorm && !(mode & GCS_CLIP_PARTIALS_READY)) GCS_TRY(launch_partials(g, grad_scale, clip, st));
  const ClipArgs c = clip_args(clip);
  const unsigned grid = norm == kNoNorm ? opt_blocks(n) : static_cast<unsigned>(clip->n_chunks);
#define GCS_OPT_LAUNCH(CV, NORM) opt_kernel<Step, CV, NORM><<<grid, kOptThreads, 0, st>>>(step, g, n, grad_scale, c)
  switch (norm * 2 + (cv ? 1 : 0)) {
    case 0: GCS_OPT_LAUNCH(false, kNoNorm); break;
    case 1: GCS_OPT_LAUNCH(true, kNoNorm); break;
    case 2: GCS_OPT_LAUNCH(false, kTensorNorm); break;
    case 3: GCS_OPT_LAUNCH(true, kTensorNorm); break;
    case 4: GCS_OPT_LAUNCH(false, kGlobalNorm); break;
    default: GCS_OPT_LAUNCH(true, kGlobalNorm); break;
  }
#undef GCS_OPT_LAUNCH
  GCS_CHECK_LAUNCH("opt_kernel");
  return GCS_OK;
}

extern "C" int gcs_sgd_step(float* w, const float* g, int64_t n, float lr, float grad_scale, gcs_stream stream) {
  GCS_CHECK_ARG(n >= 0 && (n == 0 || (w && g)), "gcs_sgd_step: bad argument");
  if (n == 0) return GCS_OK;
  return launch_step(SgdStep<kPlainSgd>{w, nullptr, lr, 0.0f}, g, n, grad_scale, nullptr, as_stream(stream));
}

extern "C" int gcs_sgd_step_ex(float* w, const float* g, float* accum, int64_t n, float lr, float momentum,
                               int32_t nesterov, float grad_scale, const gcs_grad_clip* clip, gcs_stream stream) {
  GCS_CHECK_ARG(n >= 0 && (n == 0 || (w && g)), "gcs_sgd_step_ex: bad argument");
  GCS_CHECK_ARG(momentum >= 0.0f && momentum <= 1.0f, "gcs_sgd_step_ex: momentum must lie in [0, 1]");
  GCS_CHECK_ARG(momentum == 0.0f || n == 0 || accum, "gcs_sgd_step_ex: momentum > 0 needs the accum slot");
  if (clip) GCS_TRY(check_clip(clip, false, "gcs_sgd_step_ex"));
  if (n == 0) return GCS_OK;
  const cudaStream_t st = as_stream(stream);
  if (momentum == 0.0f)          // Keras runs plain gradient descent whatever nesterov says
    return launch_step(SgdStep<kPlainSgd>{w, nullptr, lr, 0.0f}, g, n, grad_scale, clip, st);
  if (nesterov) return launch_step(SgdStep<kNesterov>{w, accum, lr, momentum}, g, n, grad_scale, clip, st);
  return launch_step(SgdStep<kMomentum>{w, accum, lr, momentum}, g, n, grad_scale, clip, st);
}

// lr_t and the (1 - beta) terms: hyper-parameters arrive as doubles so that 1 - beta is rounded once, not computed in fp32
template <bool AMSGRAD>
static AdamStep<AMSGRAD> adam_args(float* w, float* m, float* v, float* vhat, double lr, double beta1, double beta2,
                                   double eps, int64_t step) {
  const double t = static_cast<double>(step);
  const float lr_t = static_cast<float>(lr * sqrt(1.0 - pow(beta2, t)) / (1.0 - pow(beta1, t)));
  return AdamStep<AMSGRAD>{w, m, v, vhat, lr_t, static_cast<float>(beta1), static_cast<float>(beta2),
                           static_cast<float>(1.0 - beta1), static_cast<float>(1.0 - beta2), static_cast<float>(eps)};
}

extern "C" int gcs_adam_step(float* w, const float* g, float* m, float* v, int64_t n, double lr, double beta1,
                             double beta2, double eps, int64_t step, float grad_scale, gcs_stream stream) {
  GCS_CHECK_ARG(n >= 0 && step >= 1 && (n == 0 || (w && g && m && v)), "gcs_adam_step: bad argument (step is 1-based)");
  if (n == 0) return GCS_OK;
  return launch_step(adam_args<false>(w, m, v, nullptr, lr, beta1, beta2, eps, step), g, n, grad_scale, nullptr,
                     as_stream(stream));
}

extern "C" int gcs_adam_step_ex(float* w, const float* g, float* m, float* v, float* vhat, int64_t n, double lr,
                                double beta1, double beta2, double eps, int64_t step, float grad_scale,
                                const gcs_grad_clip* clip, gcs_stream stream) {
  GCS_CHECK_ARG(n >= 0 && step >= 1 && (n == 0 || (w && g && m && v)),
                "gcs_adam_step_ex: bad argument (step is 1-based)");
  if (clip) GCS_TRY(check_clip(clip, false, "gcs_adam_step_ex"));
  if (n == 0) return GCS_OK;
  const cudaStream_t st = as_stream(stream);
  if (vhat) return launch_step(adam_args<true>(w, m, v, vhat, lr, beta1, beta2, eps, step), g, n, grad_scale, clip, st);
  return launch_step(adam_args<false>(w, m, v, nullptr, lr, beta1, beta2, eps, step), g, n, grad_scale, clip, st);
}

extern "C" int gcs_grad_clip_partials(const float* g, int64_t n, float grad_scale, const gcs_grad_clip* clip,
                                      gcs_stream stream) {
  GCS_CHECK_ARG(n >= 0 && clip && (n == 0 || g), "gcs_grad_clip_partials: bad argument");
  GCS_TRY(check_clip(clip, true, "gcs_grad_clip_partials"));
  if (n == 0) return GCS_OK;
  return launch_partials(g, grad_scale, clip, as_stream(stream));
}
