// K4 / K6 — GlobalSumPool: tf.math.segment_sum(X, i) over sorted graph ids and its gradient
// dX[n] = dOut[i[n]]  (SURVEY.md §8 a9; reference call path gcn.py:320 -> GeneralGNN.pool).
// GlobalAvgPool (GeneralGNN(pool='avg')): tf.math.segment_mean(X, i) = the same sum divided by
// the graph's row count (0 for an empty graph), gradient dX[n] = dOut[i[n]] / n_{i[n]}.  MEAN is
// a template flag, so the sum instantiations are the kernels they were.
// One streaming pass over [N, W]; HBM-bound.  Deterministic: fixed row->warp assignment and
// a fixed-order cross-warp sum.
#include "common.cuh"

namespace gcs {

constexpr int kPoolWarps = 8;

// grid (graph, column tile of 128 floats).  Lane l owns float4 column (tile*32 + l); warp w
// sums rows w, w+8, ... of the graph; the 8 partials are added in warp order.
template <bool MEAN>
__global__ void __launch_bounds__(kPoolWarps * 32) segment_sum_fwd_kernel(
    const float* __restrict__ X, int64_t ldx, const int32_t* __restrict__ graph_ptr, int W,
    float* __restrict__ out, int64_t ldo) {
  __shared__ float4 part[kPoolWarps][32];
  const int g = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = (blockIdx.y * 32 + lane) * 4;
  const int r0 = __ldg(graph_ptr + g), r1 = __ldg(graph_ptr + g + 1);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < W) {
    const float* p = X + c;
    int r = r0 + warp;
    for (; r + 3 * kPoolWarps < r1; r += 4 * kPoolWarps) {   // 4 independent loads in flight
      const float4 a = __ldg(reinterpret_cast<const float4*>(p + static_cast<int64_t>(r) * ldx));
      const float4 b = __ldg(reinterpret_cast<const float4*>(p + static_cast<int64_t>(r + kPoolWarps) * ldx));
      const float4 d = __ldg(reinterpret_cast<const float4*>(p + static_cast<int64_t>(r + 2 * kPoolWarps) * ldx));
      const float4 e = __ldg(reinterpret_cast<const float4*>(p + static_cast<int64_t>(r + 3 * kPoolWarps) * ldx));
      acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
      acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
      acc.x += d.x; acc.y += d.y; acc.z += d.z; acc.w += d.w;
      acc.x += e.x; acc.y += e.y; acc.z += e.z; acc.w += e.w;
    }
    for (; r < r1; r += kPoolWarps) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(p + static_cast<int64_t>(r) * ldx));
      acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
    }
  }
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && c < W) {
    float4 s = part[0][lane];
#pragma unroll
    for (int w = 1; w < kPoolWarps; ++w) {
      const float4 t = part[w][lane];
      s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
    }
    if (MEAN && r1 > r0) {
      const float n = static_cast<float>(r1 - r0);
      s.x /= n; s.y /= n; s.z /= n; s.w /= n;
    }
    *reinterpret_cast<float4*>(out + static_cast<int64_t>(g) * ldo + c) = s;
  }
}

// Scalar variant for widths / alignments the float4 path cannot take.
template <bool MEAN>
__global__ void __launch_bounds__(kPoolWarps * 32) segment_sum_fwd_scalar_kernel(
    const float* __restrict__ X, int64_t ldx, const int32_t* __restrict__ graph_ptr, int W,
    float* __restrict__ out, int64_t ldo) {
  __shared__ float part[kPoolWarps][32];
  const int g = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.y * 32 + lane;
  const int r0 = __ldg(graph_ptr + g), r1 = __ldg(graph_ptr + g + 1);
  float acc = 0.f;
  if (c < W)
    for (int r = r0 + warp; r < r1; r += kPoolWarps) acc += __ldg(X + static_cast<int64_t>(r) * ldx + c);
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && c < W) {
    float s = part[0][lane];
    for (int w = 1; w < kPoolWarps; ++w) s += part[w][lane];
    if (MEAN && r1 > r0) s /= static_cast<float>(r1 - r0);
    out[static_cast<int64_t>(g) * ldo + c] = s;
  }
}

// grid (graph, column tile): broadcast dOut[g] (/ n_g for MEAN) to every row of the graph.
template <int VEC, bool MEAN>
__global__ void __launch_bounds__(256) segment_sum_bwd_kernel(
    const float* __restrict__ dout, int64_t ldo, const int32_t* __restrict__ graph_ptr, int W,
    float* __restrict__ dX, int64_t ldx) {
  const int g = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = (blockIdx.y * 32 + lane) * VEC;
  if (c >= W) return;
  const int r0 = __ldg(graph_ptr + g), r1 = __ldg(graph_ptr + g + 1);
  if (VEC == 4) {
    float4 v = __ldg(reinterpret_cast<const float4*>(dout + static_cast<int64_t>(g) * ldo + c));
    if (MEAN && r1 > r0) {
      const float n = static_cast<float>(r1 - r0);
      v.x /= n; v.y /= n; v.z /= n; v.w /= n;
    }
    for (int r = r0 + warp; r < r1; r += 8)
      *reinterpret_cast<float4*>(dX + static_cast<int64_t>(r) * ldx + c) = v;
  } else {
    float v = __ldg(dout + static_cast<int64_t>(g) * ldo + c);
    if (MEAN && r1 > r0) v /= static_cast<float>(r1 - r0);
    for (int r = r0 + warp; r < r1; r += 8) dX[static_cast<int64_t>(r) * ldx + c] = v;
  }
}

}  // namespace gcs

using namespace gcs;

namespace gcs {

template <bool MEAN>
static int segment_fwd(const float* X, int64_t ldx, const int32_t* graph_ptr, int32_t n_graphs, int32_t W, float* out,
                       int64_t ldo, gcs_stream stream, const char* name) {
  GCS_CHECK_ARG(n_graphs >= 0 && W > 0, "%s: bad size", name);
  if (n_graphs == 0) return GCS_OK;
  GCS_CHECK_ARG(X && graph_ptr && out && ldx >= W && ldo >= W, "%s: bad pointer / leading dimension", name);
  const bool vec = (W % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && aligned16(X) && aligned16(out);
  if (vec) {
    dim3 grid(n_graphs, static_cast<unsigned>(ceil_div(W, 128)));
    segment_sum_fwd_kernel<MEAN><<<grid, kPoolWarps * 32, 0, as_stream(stream)>>>(X, ldx, graph_ptr, W, out, ldo);
  } else {
    dim3 grid(n_graphs, static_cast<unsigned>(ceil_div(W, 32)));
    segment_sum_fwd_scalar_kernel<MEAN><<<grid, kPoolWarps * 32, 0, as_stream(stream)>>>(X, ldx, graph_ptr, W, out, ldo);
  }
  GCS_CHECK_LAUNCH("segment_sum_fwd_kernel");
  return GCS_OK;
}

template <bool MEAN>
static int segment_bwd(const float* dout, int64_t ldo, const int32_t* graph_ptr, int32_t n_graphs, int32_t W, float* dX,
                       int64_t ldx, gcs_stream stream, const char* name) {
  GCS_CHECK_ARG(n_graphs >= 0 && W > 0, "%s: bad size", name);
  if (n_graphs == 0) return GCS_OK;
  GCS_CHECK_ARG(dout && graph_ptr && dX && ldx >= W && ldo >= W, "%s: bad pointer / leading dimension", name);
  const bool vec = (W % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && aligned16(dX) && aligned16(dout);
  if (vec) {
    dim3 grid(n_graphs, static_cast<unsigned>(ceil_div(W, 128)));
    segment_sum_bwd_kernel<4, MEAN><<<grid, 256, 0, as_stream(stream)>>>(dout, ldo, graph_ptr, W, dX, ldx);
  } else {
    dim3 grid(n_graphs, static_cast<unsigned>(ceil_div(W, 32)));
    segment_sum_bwd_kernel<1, MEAN><<<grid, 256, 0, as_stream(stream)>>>(dout, ldo, graph_ptr, W, dX, ldx);
  }
  GCS_CHECK_LAUNCH("segment_sum_bwd_kernel");
  return GCS_OK;
}

// grid (graph, column tile of 256): D[g] /= max(n_g, 1) in place - the pooled gradient of GlobalAvgPool turned into
// the one of GlobalSumPool, so that the model's backward continues on the sum pool's code (model.cu).
__global__ void __launch_bounds__(256) segment_rows_div_count_kernel(float* __restrict__ D, int64_t ld,
                                                                     const int32_t* __restrict__ graph_ptr, int W) {
  const int g = blockIdx.x;
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c >= W) return;
  const int n = __ldg(graph_ptr + g + 1) - __ldg(graph_ptr + g);
  if (n > 1) D[static_cast<int64_t>(g) * ld + c] /= static_cast<float>(n);
}

int segment_rows_div_count(float* D, int64_t ld, const int32_t* graph_ptr, int n_graphs, int W, gcs_stream stream) {
  if (n_graphs <= 0) return GCS_OK;
  dim3 grid(n_graphs, static_cast<unsigned>(ceil_div(W, 256)));
  segment_rows_div_count_kernel<<<grid, 256, 0, as_stream(stream)>>>(D, ld, graph_ptr, W);
  GCS_CHECK_LAUNCH("segment_rows_div_count_kernel");
  return GCS_OK;
}

}  // namespace gcs

extern "C" int gcs_segment_sum_fwd(const float* X, int64_t ldx, const int32_t* graph_ptr, int32_t n_graphs,
                                   int32_t W, float* out, int64_t ldo, gcs_stream stream) {
  return segment_fwd<false>(X, ldx, graph_ptr, n_graphs, W, out, ldo, stream, "gcs_segment_sum_fwd");
}

extern "C" int gcs_segment_sum_bwd(const float* dout, int64_t ldo, const int32_t* graph_ptr, int32_t n_graphs,
                                   int32_t W, float* dX, int64_t ldx, gcs_stream stream) {
  return segment_bwd<false>(dout, ldo, graph_ptr, n_graphs, W, dX, ldx, stream, "gcs_segment_sum_bwd");
}

extern "C" int gcs_segment_mean_fwd(const float* X, int64_t ldx, const int32_t* graph_ptr, int32_t n_graphs,
                                    int32_t W, float* out, int64_t ldo, gcs_stream stream) {
  return segment_fwd<true>(X, ldx, graph_ptr, n_graphs, W, out, ldo, stream, "gcs_segment_mean_fwd");
}

extern "C" int gcs_segment_mean_bwd(const float* dout, int64_t ldo, const int32_t* graph_ptr, int32_t n_graphs,
                                    int32_t W, float* dX, int64_t ldx, gcs_stream stream) {
  return segment_bwd<true>(dout, ldo, graph_ptr, n_graphs, W, dX, ldx, stream, "gcs_segment_mean_bwd");
}
