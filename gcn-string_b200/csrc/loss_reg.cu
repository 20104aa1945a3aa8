// K5c — regression losses of a linear head: MeanSquaredError, MeanAbsoluteError and Huber (Keras, mean over the C
// columns, then over the rows), the mean_absolute_error metric and the gradient w.r.t. the predictions z, for
// GeneralGNN(C) with its default activation=None.  With e = z - y in float32:
//   MSE    l = e^2                                              dl/dz = 2e
//   MAE    l = |e|                                              dl/dz = sign(e)   (sign(0) = 0, as in TF)
//   Huber  l = 0.5 e^2 if |e| <= delta, else delta|e| - 0.5 delta^2   dl/dz = e, or delta sign(e)
//   loss = sum(l) / (rows * C)   mae = sum(|e|) / (rows * C)   dz = dl/dz * grad_scale / C
// Every quantity is elementwise: the same walk as loss_bce.cu over the flat [rows * C] array in units of four elements
// (one 128-bit access per operand when every pointer allows it; the same four elements with scalar accesses otherwise,
// so the sums do not depend on alignment), fp32 per element, fp64 per thread.  The per-block fp64 sums go to a workspace
// that regression_loss_finish_kernel adds in a fixed order; the grid size depends on rows * C alone (bit-identical run
// to run, no atomics).  A grid of one block writes loss_acc itself.
#include <cmath>

#include "common.cuh"

namespace gcs {

constexpr int kRegThreads = 256;
constexpr int kRegBlocksPerSm = 6;
constexpr int kRegMaxBlocks = kRegBlocksPerSm * 148;   // one wave on a B200's 148 SMs; a constant, not the device's count
constexpr int kRegFinishThreads = 1024;                // >= kRegMaxBlocks: one partial per thread

enum { kRegMse = 1, kRegMae = 2, kRegHuber = 3 };

// One element: returns its loss, leaves dz and |e|.
template <int KIND>
__device__ __forceinline__ float reg_elem(float z, float yv, float delta, float scale, float& dz, float& ae) {
  const float e = z - yv;
  const float a = fabsf(e);
  const float sgn = e > 0.f ? 1.f : (e < 0.f ? -1.f : 0.f);
  ae = a;
  if (KIND == kRegMse) {
    dz = (2.f * e) * scale;
    return e * e;
  }
  if (KIND == kRegMae) {
    dz = sgn * scale;
    return a;
  }
  if (a <= delta) {
    dz = e * scale;
    return 0.5f * e * e;
  }
  dz = (delta * sgn) * scale;
  return delta * a - 0.5f * delta * delta;
}

// Unit u = elements [4u, min(4u + 4, n)); units u = blockIdx.x * blockDim.x + threadIdx.x + k * gridDim.x * blockDim.x.
template <int KIND>
__global__ void __launch_bounds__(kRegThreads, kRegBlocksPerSm) regression_loss_kernel(
    const float* __restrict__ pred, const float* __restrict__ y, int64_t n, bool vec, float delta,
    float* __restrict__ probs, float* __restrict__ dlogits, float scale, double* __restrict__ part,
    float* __restrict__ loss_acc) {
  __shared__ double s_loss[kRegThreads];
  __shared__ double s_abs[kRegThreads];
  double loss = 0.0, abs_sum = 0.0;                 // per thread: fp64 over units, fp32 within a unit
  const int64_t units = (n + 3) >> 2;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t u = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; u < units; u += stride) {
    const int64_t i0 = u << 2;
    if (vec && i0 + 4 <= n) {
      const float4 z = *reinterpret_cast<const float4*>(pred + i0);
      const float4 yv = *reinterpret_cast<const float4*>(y + i0);
      float4 d;
      float a0, a1, a2, a3;
      const float l0 = reg_elem<KIND>(z.x, yv.x, delta, scale, d.x, a0);
      const float l1 = reg_elem<KIND>(z.y, yv.y, delta, scale, d.y, a1);
      const float l2 = reg_elem<KIND>(z.z, yv.z, delta, scale, d.z, a2);
      const float l3 = reg_elem<KIND>(z.w, yv.w, delta, scale, d.w, a3);
      loss += static_cast<double>((l0 + l1) + (l2 + l3));
      abs_sum += static_cast<double>((a0 + a1) + (a2 + a3));
      if (probs) *reinterpret_cast<float4*>(probs + i0) = z;
      if (dlogits) *reinterpret_cast<float4*>(dlogits + i0) = d;
    } else {
      float l[4] = {0.f, 0.f, 0.f, 0.f};             // the vector path's order of the four additions
      float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (i0 + k >= n) break;
        const float z = pred[i0 + k];
        float d;
        l[k] = reg_elem<KIND>(z, y[i0 + k], delta, scale, d, a[k]);
        if (probs) probs[i0 + k] = z;
        if (dlogits) dlogits[i0 + k] = d;
      }
      loss += static_cast<double>((l[0] + l[1]) + (l[2] + l[3]));
      abs_sum += static_cast<double>((a[0] + a[1]) + (a[2] + a[3]));
    }
  }
  if (!part && !loss_acc) return;
  s_loss[threadIdx.x] = loss;
  s_abs[threadIdx.x] = abs_sum;
  __syncthreads();
  for (int off = blockDim.x >> 1; off > 0; off >>= 1) {
    if (threadIdx.x < off) {
      s_loss[threadIdx.x] += s_loss[threadIdx.x + off];
      s_abs[threadIdx.x] += s_abs[threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (loss_acc) {                                  // a grid of one block: the final result
      loss_acc[0] = static_cast<float>(s_loss[0] / static_cast<double>(n));
      loss_acc[1] = static_cast<float>(s_abs[0] / static_cast<double>(n));
    } else {
      part[blockIdx.x] = s_loss[0];
      part[gridDim.x + blockIdx.x] = s_abs[0];
    }
  }
}

// One thread per partial (n_parts <= kRegFinishThreads), fixed-order tree sum; n = 0 gives {0, 0}.
__global__ void __launch_bounds__(kRegFinishThreads) regression_loss_finish_kernel(const double* __restrict__ part,
                                                                                   int n_parts, int64_t n,
                                                                                   float* __restrict__ loss_acc) {
  __shared__ double s_loss[kRegFinishThreads];
  __shared__ double s_abs[kRegFinishThreads];
  const int t = threadIdx.x;
  s_loss[t] = t < n_parts ? part[t] : 0.0;
  s_abs[t] = t < n_parts ? part[n_parts + t] : 0.0;
  __syncthreads();
  for (int off = kRegFinishThreads >> 1; off > 0; off >>= 1) {
    if (t < off) {
      s_loss[t] += s_loss[t + off];
      s_abs[t] += s_abs[t + off];
    }
    __syncthreads();
  }
  if (t == 0) {
    loss_acc[0] = n > 0 ? static_cast<float>(s_loss[0] / static_cast<double>(n)) : 0.f;
    loss_acc[1] = n > 0 ? static_cast<float>(s_abs[0] / static_cast<double>(n)) : 0.f;
  }
}

static_assert(kRegMaxBlocks <= kRegFinishThreads, "one partial per finish thread");

static int reg_blocks(int64_t n) {
  const int64_t blocks = ceil_div(ceil_div(n, static_cast<int64_t>(4)), static_cast<int64_t>(kRegThreads));
  return static_cast<int>(blocks < kRegMaxBlocks ? blocks : kRegMaxBlocks);
}

template <int KIND>
static void launch_regression(int blocks, cudaStream_t st, const float* pred, const float* y, int64_t n, bool vec,
                              float delta, float* probs, float* dlogits, float scale, double* part, float* loss_acc) {
  regression_loss_kernel<KIND><<<blocks, kRegThreads, 0, st>>>(pred, y, n, vec, delta, probs, dlogits, scale, part,
                                                               loss_acc);
}

}  // namespace gcs

using namespace gcs;

extern "C" int64_t gcs_regression_loss_workspace_bytes(int64_t rows, int32_t C) {
  if (rows < 0 || C < 1 || rows > INT64_MAX / C) return -1;
  const int blocks = reg_blocks(rows * C);
  return blocks > 1 ? static_cast<int64_t>(blocks) * 2 * sizeof(double) : 0;
}

extern "C" int gcs_regression_loss(int32_t kind, float huber_delta, const float* pred, const float* y, int64_t rows,
                                   int32_t C, float* probs, float* loss_acc, float* dlogits, float grad_scale,
                                   void* workspace, int64_t workspace_bytes, gcs_stream stream) {
  GCS_CHECK_ARG(kind >= kRegMse && kind <= kRegHuber, "gcs_regression_loss: kind=%d (1 = MSE, 2 = MAE, 3 = Huber)", kind);
  GCS_CHECK_ARG(kind != kRegHuber || (std::isfinite(huber_delta) && huber_delta > 0.f),
                "gcs_regression_loss: huber_delta must be finite and > 0, got %g", static_cast<double>(huber_delta));
  GCS_CHECK_ARG(rows >= 0 && C >= 1 && rows <= INT64_MAX / C, "gcs_regression_loss: rows=%lld, C=%d", (long long)rows, C);
  GCS_CHECK_ARG(pred || rows == 0, "gcs_regression_loss: null predictions");
  GCS_CHECK_ARG(y || (!dlogits && !loss_acc), "gcs_regression_loss: loss / gradient requested without targets");
  const int64_t n = rows * C;
  cudaStream_t st = as_stream(stream);
  if (!y) {                                          // predictions only: a linear head's output is its input
    if (probs && probs != pred && n > 0)
      GCS_CUDA(cudaMemcpyAsync(probs, pred, sizeof(float) * n, cudaMemcpyDeviceToDevice, st));
    return GCS_OK;
  }
  const int blocks = reg_blocks(n);
  double* part = nullptr;
  if (loss_acc && blocks > 1) {
    const int64_t need = gcs_regression_loss_workspace_bytes(rows, C);
    if (!workspace || workspace_bytes < need)
      return fail(GCS_ERR_WORKSPACE, "gcs_regression_loss: workspace %lld < %lld bytes", (long long)workspace_bytes,
                  (long long)need);
    GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 7u) == 0,
                  "gcs_regression_loss: workspace must be 8-byte aligned");
    part = static_cast<double*>(workspace);
  }
  if (n == 0) {
    if (loss_acc) {
      regression_loss_finish_kernel<<<1, kRegFinishThreads, 0, st>>>(nullptr, 0, 0, loss_acc);
      GCS_CHECK_LAUNCH("regression_loss_finish_kernel");
    }
    return GCS_OK;
  }
  auto aligned = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  const bool vec = aligned(pred) && aligned(y) && aligned(probs) && aligned(dlogits);
  const float scale = grad_scale / static_cast<float>(C);
  float* one_block = blocks == 1 ? loss_acc : nullptr;
  if (kind == kRegMse)
    launch_regression<kRegMse>(blocks, st, pred, y, n, vec, huber_delta, probs, dlogits, scale, part, one_block);
  else if (kind == kRegMae)
    launch_regression<kRegMae>(blocks, st, pred, y, n, vec, huber_delta, probs, dlogits, scale, part, one_block);
  else
    launch_regression<kRegHuber>(blocks, st, pred, y, n, vec, huber_delta, probs, dlogits, scale, part, one_block);
  GCS_CHECK_LAUNCH("regression_loss_kernel");
  if (part) {
    regression_loss_finish_kernel<<<1, kRegFinishThreads, 0, st>>>(part, blocks, n, loss_acc);
    GCS_CHECK_LAUNCH("regression_loss_finish_kernel");
  }
  return GCS_OK;
}
