// K5b — sigmoid + BinaryCrossentropy (mean over classes, then over rows) + binary_accuracy, forward and the gradient
// w.r.t. the logits: the head of GeneralGNN(activation='sigmoid') for binary and multi-label targets.  Keras recovers
// the logits of the sigmoid activation and evaluates sigmoid_cross_entropy_with_logits per element:
//   l  = max(z, 0) - z*y + log1p(exp(-|z|))          loss = sum(l) / (rows * C)  (= mean_b mean_c l)
//   p  = sigmoid(z)                                   acc  = sum(y == (p > 0.5)) / (rows * C)
//   dz = (p - y) * grad_scale / C
// Every quantity is elementwise, so the kernel walks the flat [rows * C] array in units of four elements (one 128-bit
// load per operand when the pointers allow; the same four elements with scalar loads otherwise, so the sums do not
// depend on alignment).  One exp per element: e = exp(-|z|) gives both log1p(e) and p = 1/(1+e) or e/(1+e), finite for
// any |z|.  The per-block fp64 loss sums and integer hit counts go to a workspace that sigmoid_bce_finish_kernel adds in
// a fixed order; the grid size depends on rows * C alone (bit-identical run to run, no atomics).  A grid of one block
// writes loss_acc itself.
#include "common.cuh"

namespace gcs {

constexpr int kBceThreads = 256;
constexpr int kBceBlocksPerSm = 6;       // resident blocks per SM at the kernel's 40 registers
constexpr int kBceMaxBlocks = kBceBlocksPerSm * 148;   // one wave on a B200's 148 SMs; a constant, not the device's count
constexpr int kBceFinishThreads = 1024;  // >= kBceMaxBlocks: one partial per thread

// One element: p = sigmoid(z); with labels also dz, the hit and the element's loss (returned, 0 without labels).
__device__ __forceinline__ float bce_elem(float z, float yv, bool want_y, float scale, float& p, float& dz, int& hit) {
  const float e = expf(-fabsf(z));
  const float inv = 1.0f / (1.0f + e);
  p = z >= 0.f ? inv : e * inv;
  if (!want_y) return 0.f;
  hit += (yv == (p > 0.5f ? 1.0f : 0.0f));
  dz = (p - yv) * scale;
  return fmaf(-z, yv, fmaxf(z, 0.f)) + log1pf(e);
}

// Unit u = elements [4u, min(4u + 4, n)); units u = blockIdx.x * blockDim.x + threadIdx.x + k * gridDim.x * blockDim.x.
__global__ void __launch_bounds__(kBceThreads, kBceBlocksPerSm) sigmoid_bce_kernel(
    const float* __restrict__ logits, const float* __restrict__ y, int64_t n, bool vec, float* __restrict__ probs,
    float* __restrict__ dlogits, float scale, double* __restrict__ part_loss, long long* __restrict__ part_hit,
    float* __restrict__ loss_acc) {
  __shared__ double s_loss[kBceThreads];
  __shared__ long long s_hit[kBceThreads];
  double loss = 0.0;                                // per thread: fp64 over units, fp32 within a unit
  int hit = 0;
  const bool want_y = y != nullptr;
  const int64_t units = (n + 3) >> 2;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t u = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; u < units; u += stride) {
    const int64_t i0 = u << 2;
    if (vec && i0 + 4 <= n) {
      const float4 z = *reinterpret_cast<const float4*>(logits + i0);
      const float4 yv = want_y ? *reinterpret_cast<const float4*>(y + i0) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 p, d;
      const float l0 = bce_elem(z.x, yv.x, want_y, scale, p.x, d.x, hit);
      const float l1 = bce_elem(z.y, yv.y, want_y, scale, p.y, d.y, hit);
      const float l2 = bce_elem(z.z, yv.z, want_y, scale, p.z, d.z, hit);
      const float l3 = bce_elem(z.w, yv.w, want_y, scale, p.w, d.w, hit);
      loss += static_cast<double>((l0 + l1) + (l2 + l3));
      if (probs) *reinterpret_cast<float4*>(probs + i0) = p;
      if (dlogits) *reinterpret_cast<float4*>(dlogits + i0) = d;
    } else {
      float l[4] = {0.f, 0.f, 0.f, 0.f};             // the vector path's order of the four additions
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (i0 + k >= n) break;
        float p, d;
        l[k] = bce_elem(logits[i0 + k], want_y ? y[i0 + k] : 0.f, want_y, scale, p, d, hit);
        if (probs) probs[i0 + k] = p;
        if (dlogits) dlogits[i0 + k] = d;
      }
      loss += static_cast<double>((l[0] + l[1]) + (l[2] + l[3]));
    }
  }
  if (!part_loss && !loss_acc) return;
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
    if (loss_acc) {                                  // a grid of one block: the final result
      loss_acc[0] = static_cast<float>(s_loss[0] / static_cast<double>(n));
      loss_acc[1] = static_cast<float>(static_cast<double>(s_hit[0]) / static_cast<double>(n));
    } else {
      part_loss[blockIdx.x] = s_loss[0];
      part_hit[blockIdx.x] = s_hit[0];
    }
  }
}

// One thread per partial (n_parts <= kBceFinishThreads), fixed-order tree sum; n = 0 gives {0, 0}.
__global__ void __launch_bounds__(kBceFinishThreads) sigmoid_bce_finish_kernel(
    const double* __restrict__ part_loss, const long long* __restrict__ part_hit, int n_parts, int64_t n,
    float* __restrict__ loss_acc) {
  __shared__ double s_loss[kBceFinishThreads];
  __shared__ long long s_hit[kBceFinishThreads];
  const int t = threadIdx.x;
  s_loss[t] = t < n_parts ? part_loss[t] : 0.0;
  s_hit[t] = t < n_parts ? part_hit[t] : 0;
  __syncthreads();
  for (int off = kBceFinishThreads >> 1; off > 0; off >>= 1) {
    if (t < off) {
      s_loss[t] += s_loss[t + off];
      s_hit[t] += s_hit[t + off];
    }
    __syncthreads();
  }
  if (t == 0) {
    loss_acc[0] = n > 0 ? static_cast<float>(s_loss[0] / static_cast<double>(n)) : 0.f;
    loss_acc[1] = n > 0 ? static_cast<float>(static_cast<double>(s_hit[0]) / static_cast<double>(n)) : 0.f;
  }
}

static_assert(kBceMaxBlocks <= kBceFinishThreads, "one partial per finish thread");

static int bce_blocks(int64_t n) {
  const int64_t blocks = ceil_div(ceil_div(n, static_cast<int64_t>(4)), static_cast<int64_t>(kBceThreads));
  return static_cast<int>(blocks < kBceMaxBlocks ? blocks : kBceMaxBlocks);
}

}  // namespace gcs

using namespace gcs;

extern "C" int64_t gcs_sigmoid_bce_workspace_bytes(int64_t rows, int32_t C) {
  if (rows < 0 || C < 1 || rows > INT64_MAX / C) return -1;
  const int blocks = bce_blocks(rows * C);
  return blocks > 1 ? static_cast<int64_t>(blocks) * (sizeof(double) + sizeof(long long)) : 0;
}

extern "C" int gcs_sigmoid_bce(const float* logits, const float* y, int64_t rows, int32_t C, float* probs, float* loss_acc,
                               float* dlogits, float grad_scale, void* workspace, int64_t workspace_bytes,
                               gcs_stream stream) {
  GCS_CHECK_ARG(rows >= 0 && C >= 1 && rows <= INT64_MAX / C, "gcs_sigmoid_bce: rows=%lld, C=%d", (long long)rows, C);
  GCS_CHECK_ARG(logits || rows == 0, "gcs_sigmoid_bce: null logits");
  GCS_CHECK_ARG(y || (!dlogits && !loss_acc), "gcs_sigmoid_bce: loss / gradient requested without labels");
  const int64_t n = rows * C;
  const int blocks = bce_blocks(n);
  double* part_loss = nullptr;
  long long* part_hit = nullptr;
  if (loss_acc && blocks > 1) {
    const int64_t need = gcs_sigmoid_bce_workspace_bytes(rows, C);
    if (!workspace || workspace_bytes < need)
      return fail(GCS_ERR_WORKSPACE, "gcs_sigmoid_bce: workspace %lld < %lld bytes", (long long)workspace_bytes,
                  (long long)need);
    GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 7u) == 0, "gcs_sigmoid_bce: workspace must be 8-byte aligned");
    part_loss = static_cast<double*>(workspace);
    part_hit = reinterpret_cast<long long*>(part_loss + blocks);
  }
  cudaStream_t st = as_stream(stream);
  if (n == 0) {
    if (loss_acc) {
      sigmoid_bce_finish_kernel<<<1, kBceFinishThreads, 0, st>>>(nullptr, nullptr, 0, 0, loss_acc);
      GCS_CHECK_LAUNCH("sigmoid_bce_finish_kernel");
    }
    return GCS_OK;
  }
  auto aligned = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  const bool vec = aligned(logits) && aligned(y) && aligned(probs) && aligned(dlogits);
  const float scale = grad_scale / static_cast<float>(C);
  sigmoid_bce_kernel<<<blocks, kBceThreads, 0, st>>>(logits, y, n, vec, probs, dlogits, scale, part_loss, part_hit,
                                                     blocks == 1 ? loss_acc : nullptr);
  GCS_CHECK_LAUNCH("sigmoid_bce_kernel");
  if (part_loss) {
    sigmoid_bce_finish_kernel<<<1, kBceFinishThreads, 0, st>>>(part_loss, part_hit, blocks, n, loss_acc);
    GCS_CHECK_LAUNCH("sigmoid_bce_finish_kernel");
  }
  return GCS_OK;
}
