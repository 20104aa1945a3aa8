// Kernels of the attribution backward (gradients with respect to the model's inputs, DESIGN.md §3.13): the gradient
// of the per-entry edge weights, the input gradient of the first dense block, the BatchNorm/PReLU backward on moving
// statistics (inference mode), and the Jacobian of the head's activation.  None of them runs in a forward, a train
// step or a parameter-only backward.
#include "common.cuh"

namespace gcs {

enum { kEgSum = 0, kEgMean = 1, kEgMax = 2 };

// ---------------------------------------------------------------------------------------------
// Edge-weight gradient, an SDDMM over the forward pattern.  For Z = agg_e(w_e * a[j_e]) with a = f(X) and stored entry
// e = (i, j) of row i:
//   sum : dw_e = sum_c dZ[i, c] * a[j, c]
//   mean: the same / (entries of row i)
//   max : sum over the columns where w_e * a[j, c] == Z[i, c] of dZ[i, c] * a[j, c] / ties[i, c]
// One warp per row i with dZ[i] (and, for max, Z[i] and ties[i]) in registers, lane = columns lane + 32 k; each entry
// gathers a[j], and its dot product is reduced by a fixed xor-shuffle tree.  One writer per entry and a fixed order:
// bit-identical from run to run.  accumulate != 0 adds to dw (the layers of a model, in a fixed order).
template <int NT, bool MAX>
__global__ void __launch_bounds__(256) spmm_edge_grad_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, const float* __restrict__ values,
    int64_t n_rows, const float* __restrict__ dZ, int64_t lddz, int mean, const float* __restrict__ X, int64_t ldx,
    const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ alpha,
    const float* __restrict__ Z, int64_t ldz, const float* __restrict__ ties, int64_t ldt, int H,
    float* __restrict__ dw, int accumulate) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (i >= n_rows) return;
  const int eb = __ldg(rowptr + i), ee = __ldg(rowptr + i + 1);
  if (eb == ee) return;
  float g[NT], sc[NT], sh[NT], al[NT], z[NT], rt[NT];
#pragma unroll
  for (int k = 0; k < NT; ++k) {
    const int c = lane + 32 * k;
    const bool in = c < H;
    g[k] = in ? __ldg(dZ + i * lddz + c) : 0.f;
    sc[k] = scale && in ? __ldg(scale + c) : 1.f;
    sh[k] = scale && in ? __ldg(shift + c) : 0.f;
    al[k] = scale && in ? __ldg(alpha + c) : 1.f;
    z[k] = MAX && in ? __ldg(Z + i * ldz + c) : 0.f;
    rt[k] = MAX && in ? 1.f / __ldg(ties + i * ldt + c) : 0.f;
  }
  auto row = [&](int e) {
    const int64_t j = __ldg(colidx + e);
    const float w = values ? __ldg(values + e) : 1.f;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NT; ++k) {
      const int c = lane + 32 * k;
      if (c >= H) continue;
      float a = __ldg(X + j * ldx + c);
      if (scale) a = bn_prelu(a, sc[k], sh[k], al[k]);
      if (MAX) {
        // the same comparison as the forward maximum and spmm_agg_bwd_kernel
        if ((values ? a * w : a) == z[k]) s = fmaf(g[k] * a, rt[k], s);
      } else {
        s = fmaf(g[k], a, s);
      }
    }
    return s;
  };
  const float inv = mean ? 1.f / static_cast<float>(ee - eb) : 1.f;
  auto finish = [&](int e, float s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      if (mean) s *= inv;
      dw[e] = accumulate ? dw[e] + s : s;
    }
  };
  int e = eb;
  for (; e + 2 <= ee; e += 2) {            // two gathers in flight
    const float s0 = row(e), s1 = row(e + 1);
    finish(e, s0);
    finish(e + 1, s1);
  }
  if (e < ee) finish(e, row(e));
}

// ---------------------------------------------------------------------------------------------
// Input gradient of a dense layer with a THIN input (the first Dense of the pre-processing MLP, K = F <= 32 features):
// dX[M, K] = dH[M, N] . W[K, N]^T.  The tensor-core kernels need the output width to be a multiple of 64, and the
// tiled FFMA kernel leaves most of its 128-wide tile empty.  Here one thread owns one row of dX (K4 * 4 accumulators)
// and walks its row of dH in 32-byte sectors (two 128-bit loads per step), W^T sits in shared memory as [N][K4] float4
// read by broadcast.  fp32 FMAs in a fixed order per element: deterministic.  A grid of a few CTAs per SM strides over
// the rows, so W is staged once per CTA.
template <int K4>
__global__ void __launch_bounds__(256) dx_thin_kernel(const float* __restrict__ dH, int64_t ldh, const float* __restrict__ W,
                                                      int K, int N, float* __restrict__ dX, int64_t lddx, int64_t M) {
  extern __shared__ float4 sW[];                       // sW[n * K4 + q] = W[4q .. 4q+3][n]
  for (int t = threadIdx.x; t < N * K4; t += blockDim.x) {
    const int n = t / K4, q = t - n * K4;
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = 4 * q + u < K ? __ldg(W + static_cast<int64_t>(4 * q + u) * N + n) : 0.f;
    sW[t] = make_float4(v[0], v[1], v[2], v[3]);
  }
  __syncthreads();
  for (int64_t m = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; m < M;
       m += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float acc[4 * K4];
#pragma unroll
    for (int k = 0; k < 4 * K4; ++k) acc[k] = 0.f;
    const float* row = dH + m * ldh;
    for (int n = 0; n < N; n += 8) {
      const float4 d0 = __ldg(reinterpret_cast<const float4*>(row + n));
      const float4 d1 = __ldg(reinterpret_cast<const float4*>(row + n + 4));
      const float d[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
      for (int u = 0; u < 8; ++u) {
#pragma unroll
        for (int q = 0; q < K4; ++q) {
          const float4 w = sW[(n + u) * K4 + q];
          acc[4 * q + 0] = fmaf(d[u], w.x, acc[4 * q + 0]);
          acc[4 * q + 1] = fmaf(d[u], w.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(d[u], w.z, acc[4 * q + 2]);
          acc[4 * q + 3] = fmaf(d[u], w.w, acc[4 * q + 3]);
        }
      }
    }
    float* out = dX + m * lddx;
#pragma unroll
    for (int k = 0; k < 4 * K4; ++k)
      if (k < K) out[k] = acc[k];
  }
}

// ---------------------------------------------------------------------------------------------
// BatchNorm + PReLU backward on moving statistics (inference mode, frozen BatchNorm): with the folded scale / shift
// of the forward (scale = gamma * rsqrt(moving_variance + eps)), z = h * scale + shift and
//   dh = scale * slope(z) * da,   slope = 1 (z > 0), alpha (z < 0), 0 (z == 0); alpha == NULL: no PReLU (slope 1).
// No batch-statistics terms and no parameter gradients.  z is formed exactly as bn_prelu_fwd_kernel forms it, so the
// branch of every element is the one the forward took.  Folds |dh| into amax (the tensor-core GEMMs that read dh).
__global__ void __launch_bounds__(256) bn_prelu_bwd_frozen_kernel(
    const float* __restrict__ da, int64_t ldda, const float* __restrict__ h, int64_t ldh, const float* __restrict__ scale,
    const float* __restrict__ shift, const float* __restrict__ alpha, float* __restrict__ dh, int64_t lddh, int64_t M,
    int C, float* __restrict__ amax) {
  float mx = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float sc = __ldg(scale + c), sh = __ldg(shift + c), al = alpha ? __ldg(alpha + c) : 1.f;
    for (int64_t r = blockIdx.x; r < M; r += gridDim.x) {
      const float g = __ldg(da + r * ldda + c);
      const float z = fmaf(__ldg(h + r * ldh + c), sc, sh);
      const float dz = alpha ? (z > 0.f ? g : (z < 0.f ? g * al : 0.f)) : g;
      const float o = sc * dz;
      dh[r * lddh + c] = o;
      mx = fmaxf(mx, fabsf(o));
    }
  }
  amax_commit(mx, amax);
}

// ---------------------------------------------------------------------------------------------
// dlogits = J_act^T . dprobs for the head's activation, one thread per row: softmax p * (d - p . d), sigmoid
// d * p * (1 - p), linear d.
__global__ void __launch_bounds__(256) output_grad_kernel(int act, const float* __restrict__ p, const float* __restrict__ d,
                                                          int64_t rows, int C, float* __restrict__ out) {
  const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float* pr = p + r * C;
  const float* dr = d + r * C;
  float* o = out + r * C;
  if (act == 1) {
    float dot = 0.f;
    for (int c = 0; c < C; ++c) dot = fmaf(__ldg(pr + c), __ldg(dr + c), dot);
    for (int c = 0; c < C; ++c) o[c] = __ldg(pr + c) * (__ldg(dr + c) - dot);
  } else if (act == 2) {
    for (int c = 0; c < C; ++c) {
      const float q = __ldg(pr + c);
      o[c] = __ldg(dr + c) * (q * (1.f - q));
    }
  } else {
    for (int c = 0; c < C; ++c) o[c] = __ldg(dr + c);
  }
}

// Input gradient of a thin dense layer (dx_thin_kernel).  GCS_ERR_UNSUPPORTED, with nothing launched, when the shape
// or alignment is not the kernel's (K > 32, N % 8 != 0, W^T over 48 KB, unaligned dH): the caller then runs
// gcs_linear_bwd_input.
int dense_dx_thin(const float* dH, int64_t ldh, const float* W, int K, int N, float* dX, int64_t lddx, int64_t M,
                  cudaStream_t st) {
  const int K4 = (K + 3) / 4;
  const int64_t smem = static_cast<int64_t>(N) * K4 * 16;
  if (K < 1 || K > 32 || N % 8 != 0 || ldh % 4 != 0 || !aligned16(dH) || smem > 48 * 1024)
    return GCS_ERR_UNSUPPORTED;
  if (M == 0) return GCS_OK;
  const int64_t blocks = ceil_div(M, 256);
  const int64_t cap = 4LL * sm_count();
  const dim3 grid(static_cast<unsigned>(blocks < cap ? blocks : cap));
  const size_t sm = static_cast<size_t>(smem);
  switch (K4) {
    case 1: dx_thin_kernel<1><<<grid, 256, sm, st>>>(dH, ldh, W, K, N, dX, lddx, M); break;
    case 2: dx_thin_kernel<2><<<grid, 256, sm, st>>>(dH, ldh, W, K, N, dX, lddx, M); break;
    case 3: dx_thin_kernel<3><<<grid, 256, sm, st>>>(dH, ldh, W, K, N, dX, lddx, M); break;
    case 4: dx_thin_kernel<4><<<grid, 256, sm, st>>>(dH, ldh, W, K, N, dX, lddx, M); break;
    case 5: dx_thin_kernel<5><<<grid, 256, sm, st>>>(dH, ldh, W, K, N, dX, lddx, M); break;
    case 6: dx_thin_kernel<6><<<grid, 256, sm, st>>>(dH, ldh, W, K, N, dX, lddx, M); break;
    case 7: dx_thin_kernel<7><<<grid, 256, sm, st>>>(dH, ldh, W, K, N, dX, lddx, M); break;
    default: dx_thin_kernel<8><<<grid, 256, sm, st>>>(dH, ldh, W, K, N, dX, lddx, M); break;
  }
  GCS_CHECK_LAUNCH("dx_thin_kernel");
  return GCS_OK;
}

int bn_prelu_bwd_frozen(const float* da, int64_t ldda, const float* h, int64_t ldh, const float* scale, const float* shift,
                        const float* alpha, float* dh, int64_t lddh, int64_t M, int C, cudaStream_t st) {
  if (M == 0) return GCS_OK;
  const int64_t cap = 8LL * sm_count();
  const dim3 grid(static_cast<unsigned>(M < cap ? M : cap));
  const int threads = C < 256 ? ((C + 31) / 32) * 32 : 256;
  bn_prelu_bwd_frozen_kernel<<<grid, threads, 0, st>>>(da, ldda, h, ldh, scale, shift, alpha, dh, lddh, M, C,
                                                       amax_sink().produce);
  GCS_CHECK_LAUNCH("bn_prelu_bwd_frozen_kernel");
  return GCS_OK;
}

}  // namespace gcs

using namespace gcs;

extern "C" int gcs_spmm_edge_grad(const int32_t* rowptr, const int32_t* colidx, const float* values, int64_t n_rows,
                                  const float* dZ, int64_t lddz, int32_t aggregate, const float* X, int64_t ldx,
                                  const float* scale, const float* shift, const float* alpha, const float* Z, int64_t ldz,
                                  const float* ties, int64_t ldt, int32_t H, float* dvalues, int32_t accumulate,
                                  gcs_stream stream) {
  GCS_CHECK_ARG(n_rows >= 0 && H > 0, "gcs_spmm_edge_grad: bad size");
  GCS_CHECK_ARG(aggregate == kEgSum || aggregate == kEgMean || aggregate == kEgMax,
                "gcs_spmm_edge_grad: aggregate must be 0 (sum), 1 (mean) or 2 (max)");
  if (H > 512) return fail(GCS_ERR_UNSUPPORTED, "gcs_spmm_edge_grad: H = %d > 512 is not built", H);
  if (n_rows == 0) return GCS_OK;
  GCS_CHECK_ARG(rowptr && colidx && dZ && X && dvalues && lddz >= H && ldx >= H,
                "gcs_spmm_edge_grad: bad pointer / leading dimension");
  GCS_CHECK_ARG((scale != nullptr) == (shift != nullptr) && (scale != nullptr) == (alpha != nullptr),
                "gcs_spmm_edge_grad: scale/shift/alpha must be all NULL or all set");
  GCS_CHECK_ARG(aggregate != kEgMax || (Z && ties && ldz >= H && ldt >= H),
                "gcs_spmm_edge_grad: max needs the forward output Z and the ties of gcs_spmm_aggregate_bwd");
  GCS_CHECK_ARG(n_rows < INT32_MAX, "gcs_spmm_edge_grad: n_rows exceeds int32 CSR range");
  const unsigned grid = static_cast<unsigned>(ceil_div(n_rows, 8));     // 8 warps (rows) per CTA
  cudaStream_t st = as_stream(stream);
  const int mean = aggregate == kEgMean;
#define GCS_EG(NT, MX)                                                                                               \
  spmm_edge_grad_kernel<NT, MX><<<grid, 256, 0, st>>>(rowptr, colidx, values, n_rows, dZ, lddz, mean, X, ldx, scale, \
                                                      shift, alpha, Z, ldz, ties, ldt, H, dvalues, accumulate)
  const bool mx = aggregate == kEgMax;
  if (H <= 32) { if (mx) GCS_EG(1, true); else GCS_EG(1, false); }
  else if (H <= 64) { if (mx) GCS_EG(2, true); else GCS_EG(2, false); }
  else if (H <= 128) { if (mx) GCS_EG(4, true); else GCS_EG(4, false); }
  else if (H <= 256) { if (mx) GCS_EG(8, true); else GCS_EG(8, false); }
  else { if (mx) GCS_EG(16, true); else GCS_EG(16, false); }
#undef GCS_EG
  GCS_CHECK_LAUNCH("spmm_edge_grad_kernel");
  return GCS_OK;
}

extern "C" int gcs_output_grad(int32_t final_activation, const float* probs, const float* dprobs, int64_t rows, int32_t C,
                               float* dlogits, gcs_stream stream) {
  GCS_CHECK_ARG(final_activation >= 0 && final_activation <= 2,
                "gcs_output_grad: final activation must be 0 (linear), 1 (softmax) or 2 (sigmoid)");
  GCS_CHECK_ARG(rows >= 0 && C > 0, "gcs_output_grad: bad size");
  if (rows == 0) return GCS_OK;
  GCS_CHECK_ARG(probs && dprobs && dlogits, "gcs_output_grad: null pointer");
  output_grad_kernel<<<static_cast<unsigned>(ceil_div(rows, 256)), 256, 0, as_stream(stream)>>>(final_activation, probs, dprobs,
                                                                                                 rows, C, dlogits);
  GCS_CHECK_LAUNCH("output_grad_kernel");
  return GCS_OK;
}
