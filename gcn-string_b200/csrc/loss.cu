// K5 — softmax + CategoricalCrossentropy (mean) + categorical_accuracy, forward and the
// gradient w.r.t. the logits (reference: src/scripts/gcn.py:326 loss_fn, :335 loss,
// :339 accuracy; SURVEY.md §8 a10).  Keras recovers the logits of the softmax activation
// and evaluates softmax_cross_entropy_with_logits:
//   loss_b = logsumexp(z_b) * sum(y_b) - y_b . z_b ;  loss = mean_b loss_b
//          (evaluated as log(sum exp(z - m)) * sum(y) - y . (z - m), m = max z)
//   dz_b   = (softmax(z_b) * sum(y_b) - y_b) * grad_scale
// Two kernels share the per-row code (xent_row), so probs / dlogits are bit-identical between them:
//   softmax_xent_kernel       one CTA, fixed-order tree reduction.  Graph-level batches are tiny ([1024, 2]).
//   softmax_xent_grid_kernel  a grid of CTAs for node-level batches (~508 k rows at the cfg3 shape, where one CTA
//                             would walk ~500 rows per thread); per-CTA fp64 loss / int hit partials go to a workspace
//                             and softmax_xent_finish_kernel adds them in a fixed order.  The grid size depends on the
//                             row count alone: deterministic run to run.
// gcs_softmax_xent_ws picks between them by row count (kXentGridThreshold).
#include "common.cuh"

namespace gcs {

constexpr int kMaxClasses = 64;
constexpr int64_t kXentGridThreshold = 65536;   // rows above which gcs_softmax_xent_ws runs the grid kernel
constexpr int kXentGridThreads = 256;
constexpr int kXentMaxBlocks = 1024;            // = the finish kernel's block size: one partial per thread

// One row b: writes probs / dlogits, adds the row's loss and hit to *loss / *hit (when y != NULL).
__device__ __forceinline__ void xent_row(const float* __restrict__ logits, const float* __restrict__ y, int64_t b, int C,
                                         float* __restrict__ probs, float* __restrict__ dlogits, float grad_scale,
                                         double* loss, int* hit) {
  const float* z = logits + b * C;
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
  if (y) {
    const float* yy = y + b * C;
    ymax = yy[0];
    for (int c = 0; c < C; ++c) {
      ysum += yy[c];
      yz = fmaf(yy[c], z[c] - m, yz);            // y . (z - m): no cancellation against lse
      if (c > 0 && yy[c] > ymax) { ymax = yy[c]; arg_y = c; }
    }
    *loss += static_cast<double>(log_sum * ysum - yz);
    *hit += (arg_y == arg_p);
  }
  for (int c = 0; c < C; ++c) {
    const float p = e[c] * inv;
    if (probs) probs[b * C + c] = p;
    if (dlogits) dlogits[b * C + c] = (p * ysum - y[b * C + c]) * grad_scale;
  }
}

__global__ void __launch_bounds__(1024) softmax_xent_kernel(
    const float* __restrict__ logits, const float* __restrict__ y, int B, int C,
    float* __restrict__ probs, float* __restrict__ loss_acc, float* __restrict__ dlogits,
    float grad_scale) {
  __shared__ double s_loss[1024];
  __shared__ int s_hit[1024];
  double loss = 0.0;
  int hit = 0;
  for (int b = threadIdx.x; b < B; b += blockDim.x)
    xent_row(logits, y, b, C, probs, dlogits, grad_scale, &loss, &hit);
  s_loss[threadIdx.x] = loss;
  s_hit[threadIdx.x] = hit;
  __syncthreads();
  for (int off = blockDim.x >> 1; off > 0; off >>= 1) {
    if (threadIdx.x < off) {
      s_loss[threadIdx.x] += s_loss[threadIdx.x + off];
      s_hit[threadIdx.x] += s_hit[threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0 && loss_acc) {
    loss_acc[0] = B > 0 ? static_cast<float>(s_loss[0] / B) : 0.f;
    loss_acc[1] = B > 0 ? static_cast<float>(s_hit[0]) / static_cast<float>(B) : 0.f;
  }
}

// Rows b = blockIdx.x * blockDim.x + threadIdx.x + k * gridDim.x * blockDim.x; the CTA's loss / hit sums go to
// part_loss[blockIdx.x] / part_hit[blockIdx.x].
__global__ void __launch_bounds__(kXentGridThreads) softmax_xent_grid_kernel(
    const float* __restrict__ logits, const float* __restrict__ y, int B, int C, float* __restrict__ probs,
    float* __restrict__ dlogits, float grad_scale, double* __restrict__ part_loss, int* __restrict__ part_hit) {
  __shared__ double s_loss[kXentGridThreads];
  __shared__ int s_hit[kXentGridThreads];
  double loss = 0.0;
  int hit = 0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; b < B; b += stride)
    xent_row(logits, y, b, C, probs, dlogits, grad_scale, &loss, &hit);
  if (!part_loss) return;
  s_loss[threadIdx.x] = loss;
  s_hit[threadIdx.x] = hit;
  __syncthreads();
  for (int off = blockDim.x >> 1; off > 0; off >>= 1) {
    if (threadIdx.x < off) {
      s_loss[threadIdx.x] += s_loss[threadIdx.x + off];
      s_hit[threadIdx.x] += s_hit[threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    part_loss[blockIdx.x] = s_loss[0];
    part_hit[blockIdx.x] = s_hit[0];
  }
}

// One thread per partial (n_parts <= kXentMaxBlocks), fixed-order tree sum.
__global__ void __launch_bounds__(kXentMaxBlocks) softmax_xent_finish_kernel(
    const double* __restrict__ part_loss, const int* __restrict__ part_hit, int n_parts, int B, float* __restrict__ loss_acc) {
  __shared__ double s_loss[kXentMaxBlocks];
  __shared__ int s_hit[kXentMaxBlocks];
  const int t = threadIdx.x;
  s_loss[t] = t < n_parts ? part_loss[t] : 0.0;
  s_hit[t] = t < n_parts ? part_hit[t] : 0;
  __syncthreads();
  for (int off = kXentMaxBlocks >> 1; off > 0; off >>= 1) {
    if (t < off) {
      s_loss[t] += s_loss[t + off];
      s_hit[t] += s_hit[t + off];
    }
    __syncthreads();
  }
  if (t == 0) {
    loss_acc[0] = static_cast<float>(s_loss[0] / B);
    loss_acc[1] = static_cast<float>(s_hit[0]) / static_cast<float>(B);
  }
}

static int xent_grid_blocks(int64_t B) {
  const int64_t blocks = ceil_div(B, static_cast<int64_t>(kXentGridThreads));
  return static_cast<int>(blocks < kXentMaxBlocks ? blocks : kXentMaxBlocks);
}

}  // namespace gcs

using namespace gcs;

extern "C" int gcs_softmax_xent(const float* logits, const float* y, int32_t B, int32_t C, float* probs,
                                float* loss_acc, float* dlogits, float grad_scale, gcs_stream stream) {
  GCS_CHECK_ARG(B >= 0 && C > 0 && C <= kMaxClasses, "gcs_softmax_xent: C=%d outside [1, %d]", C, kMaxClasses);
  GCS_CHECK_ARG(logits || B == 0, "gcs_softmax_xent: null logits");
  GCS_CHECK_ARG(y || (!dlogits && !loss_acc), "gcs_softmax_xent: loss / gradient requested without labels");
  softmax_xent_kernel<<<1, 1024, 0, as_stream(stream)>>>(logits, y, B, C, probs, loss_acc, dlogits, grad_scale);
  GCS_CHECK_LAUNCH("softmax_xent_kernel");
  return GCS_OK;
}

extern "C" int64_t gcs_softmax_xent_workspace_bytes(int64_t B, int32_t C) {
  (void)C;
  if (B < 0) return -1;
  if (B <= kXentGridThreshold) return 0;
  return static_cast<int64_t>(xent_grid_blocks(B)) * (sizeof(double) + sizeof(int));
}

extern "C" int gcs_softmax_xent_ws(const float* logits, const float* y, int32_t B, int32_t C, float* probs,
                                   float* loss_acc, float* dlogits, float grad_scale, void* workspace,
                                   int64_t workspace_bytes, gcs_stream stream) {
  if (B <= kXentGridThreshold)
    return gcs_softmax_xent(logits, y, B, C, probs, loss_acc, dlogits, grad_scale, stream);
  GCS_CHECK_ARG(C > 0 && C <= kMaxClasses, "gcs_softmax_xent_ws: C=%d outside [1, %d]", C, kMaxClasses);
  GCS_CHECK_ARG(logits, "gcs_softmax_xent_ws: null logits");
  GCS_CHECK_ARG(y || (!dlogits && !loss_acc), "gcs_softmax_xent_ws: loss / gradient requested without labels");
  const int blocks = xent_grid_blocks(B);
  double* part_loss = nullptr;
  int* part_hit = nullptr;
  if (loss_acc) {
    const int64_t need = gcs_softmax_xent_workspace_bytes(B, C);
    if (!workspace || workspace_bytes < need)
      return fail(GCS_ERR_WORKSPACE, "gcs_softmax_xent_ws: workspace %lld < %lld bytes", (long long)workspace_bytes,
                  (long long)need);
    GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 7u) == 0, "gcs_softmax_xent_ws: workspace must be 8-byte aligned");
    part_loss = static_cast<double*>(workspace);
    part_hit = reinterpret_cast<int*>(part_loss + blocks);
  }
  cudaStream_t st = as_stream(stream);
  softmax_xent_grid_kernel<<<blocks, kXentGridThreads, 0, st>>>(logits, y, B, C, probs, dlogits, grad_scale, part_loss,
                                                                part_hit);
  GCS_CHECK_LAUNCH("softmax_xent_grid_kernel");
  if (loss_acc) {
    softmax_xent_finish_kernel<<<1, kXentMaxBlocks, 0, st>>>(part_loss, part_hit, blocks, B, loss_acc);
    GCS_CHECK_LAUNCH("softmax_xent_finish_kernel");
  }
  return GCS_OK;
}
