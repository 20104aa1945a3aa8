// K2 / K8 — Keras BatchNormalization (rank-2, non-fused path) + PReLU, forward and backward.
//
// Upstream semantics restated (SURVEY.md §8 a6/a7; reference instantiates them through
// GeneralGNN at src/scripts/gcn.py:320 and runs them at :334 training / :351 inference):
//   training:  mean = reduce_mean(h, 0); var = reduce_mean((h - mean)^2, 0)   (biased, two-pass)
//              y = h * inv + (beta - mean * inv),  inv = gamma * rsqrt(var + eps)
//              moving <- moving - (moving - batch) * (1 - momentum)
//   inference: the same formula with the moving statistics
//   PReLU:     f(z) = relu(z) - alpha * relu(-z), alpha per channel; df/dz = 1 (z>0), alpha
//              (z<0), 0 (z==0); df/dalpha = min(z, 0)
// The column reductions run ONE pass over h with fp64 accumulators (sum, sum of squares):
// in fp64 E[h^2] - mean^2 reproduces the two-pass variance to fp32 rounding.  Partials are
// written per row-split and combined in a fixed order: deterministic, no atomics.
#include "common.cuh"
#include "dropout.cuh"

namespace gcs {

constexpr int kBnThreads = 256;   // 32 column lanes x 8 row warps

struct BnGrid {
  int vec;         // 4 or 1 columns per lane
  int col_blocks;  // grid.x
  int splits;      // grid.y
  int64_t rows_per_split;
};

static BnGrid bn_grid(int64_t M, int C, bool vec_ok) {
  BnGrid g;
  g.vec = vec_ok ? 4 : 1;
  g.col_blocks = static_cast<int>(ceil_div(C, 32 * g.vec));
  int64_t target = 4LL * sm_count();
  int64_t s = ceil_div(target, g.col_blocks);
  int64_t max_s = ceil_div(M, 32);
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  if (s > 65535) s = 65535;
  g.rows_per_split = ceil_div(M > 0 ? M : 1, s);
  g.splits = static_cast<int>(ceil_div(M > 0 ? M : 1, g.rows_per_split));
  return g;
}

// Upper bound on splits for workspace sizing (alignment-independent).
static int64_t bn_max_splits(int64_t M) {
  int64_t s = 4LL * sm_count();
  int64_t max_s = ceil_div(M > 0 ? M : 1, 32);
  return s < max_s ? s : max_s;
}

// Block-level combine of per-warp fp64 partials: warps 1..7 park their values in shared
// memory, warp 0 adds them in warp order and writes the split's partial.
template <int NV>
__device__ __forceinline__ void block_store_partials(double (&v)[NV], double* __restrict__ dst_col0,
                                                     int64_t col_stride, int ncols_valid, bool lane_valid) {
  __shared__ double sm[7][32][NV];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp > 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) sm[warp - 1][lane][k] = v[k];
  }
  __syncthreads();
  if (warp == 0 && lane_valid) {
#pragma unroll
    for (int w = 0; w < 7; ++w)
#pragma unroll
      for (int k = 0; k < NV; ++k) v[k] += sm[w][lane][k];
#pragma unroll
    for (int k = 0; k < NV; ++k) dst_col0[k] = v[k];
  }
  (void)col_stride; (void)ncols_valid;
}

// Final combine of per-split partials, one WARP per column: lane l adds splits l, l+32, ... in order, then the 32
// lane sums meet in a fixed shuffle tree - deterministic, and ~20x shorter than one thread walking all ~300 splits
// (the three "final" kernels were 40-65 us each, latency-bound: 1.2 ms per train step).
__device__ __forceinline__ double warp_sum_fixed(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;                                             // valid in lane 0
}

// partial layout: ws[(split * C + c) * Q + q], Q quantities per column.
template <int VEC>
__global__ void __launch_bounds__(kBnThreads) bn_stats_partial_kernel(
    const float* __restrict__ h, int64_t ldh, int64_t M, int C, int64_t rows_per_split,
    double* __restrict__ ws) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + lane) * VEC;
  const int64_t rb = blockIdx.y * rows_per_split;
  int64_t re = rb + rows_per_split;
  if (re > M) re = M;
  double acc[2 * VEC];
#pragma unroll
  for (int k = 0; k < 2 * VEC; ++k) acc[k] = 0.0;
  if (c < C) {
    for (int64_t r = rb + warp; r < re; r += 8) {
      float v[VEC];
      if (VEC == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(h + r * ldh + c));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
        v[0] = __ldg(h + r * ldh + c);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        const double d = static_cast<double>(v[k]);
        acc[2 * k] += d;
        acc[2 * k + 1] = fma(d, d, acc[2 * k + 1]);
      }
    }
  }
  block_store_partials<2 * VEC>(acc, ws + (static_cast<int64_t>(blockIdx.y) * C + c) * 2, 0, 0, c < C);
}

__global__ void __launch_bounds__(256) bn_stats_final_kernel(const double* __restrict__ ws, int splits, int C, int64_t M,
                                                             float* __restrict__ mean, float* __restrict__ var) {
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  double s = 0.0, q = 0.0;
  for (int k = lane; k < splits; k += 32) {
    s += ws[(static_cast<int64_t>(k) * C + c) * 2];
    q += ws[(static_cast<int64_t>(k) * C + c) * 2 + 1];
  }
  s = warp_sum_fixed(s);
  q = warp_sum_fixed(q);
  if (lane == 0) {
    const double m = s / static_cast<double>(M);
    double v = q / static_cast<double>(M) - m * m;
    if (v < 0.0) v = 0.0;
    mean[c] = static_cast<float>(m);
    var[c] = static_cast<float>(v);
  }
}

// Statistics out of the dense layer's own epilogue (linear_tc.cu writes, per group of 32 rows and per column, the fp32
// pair {group mean, sum of squared deviations from it}): fold the groups into the same per-split fp64 partials
// {sum h, sum h^2} the pass over h would have produced - sum h = sum n_g*mean_g, sum h^2 = sum (M2_g + n_g*mean_g^2),
// all in fp64, so that the only subtraction of large squares (E[h^2] - mean^2 in bn_stats_finish) happens in fp64.
__global__ void __launch_bounds__(256) bn_stats_from_part_kernel(const float2* __restrict__ part, int64_t groups, int C,
                                                                 int splits, double* __restrict__ ws, int64_t M) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  double acc[2] = {0.0, 0.0};
  if (c < C) {
    for (int64_t g = static_cast<int64_t>(blockIdx.y) * 8 + warp; g < groups; g += 8LL * splits) {
      const float2 v = __ldg(part + g * C + c);
      const double n = static_cast<double>(M - g * 32 < 32 ? M - g * 32 : 32);
      const double mg = static_cast<double>(v.x);
      acc[0] += n * mg;
      acc[1] += static_cast<double>(v.y) + n * mg * mg;
    }
  }
  block_store_partials<2>(acc, ws + (static_cast<int64_t>(blockIdx.y) * C + c) * 2, 0, 0, c < C);
}

// Synchronised BatchNorm: the per-column sums of this rank (+ its row count as the last element) go through the
// all-reduce hook, mean / variance are formed from the global sums.
__global__ void __launch_bounds__(256) bn_stats_sums_kernel(const double* __restrict__ ws, int splits, int C, int64_t M,
                                                            double* __restrict__ sums) {
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  double s = 0.0, q = 0.0;
  for (int k = lane; k < splits; k += 32) {
    s += ws[(static_cast<int64_t>(k) * C + c) * 2];
    q += ws[(static_cast<int64_t>(k) * C + c) * 2 + 1];
  }
  s = warp_sum_fixed(s);
  q = warp_sum_fixed(q);
  if (lane == 0) {
    sums[c] = s;
    sums[C + c] = q;
    if (c == 0) sums[2 * C] = static_cast<double>(M);
  }
}

__global__ void bn_stats_finish_kernel(const double* __restrict__ sums, int C, float* __restrict__ mean,
                                       float* __restrict__ var) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double Mg = sums[2 * C];
  const double m = sums[c] / Mg;
  double v = sums[C + c] / Mg - m * m;
  if (v < 0.0) v = 0.0;
  mean[c] = static_cast<float>(m);
  var[c] = static_cast<float>(v);
}

__global__ void bn_fold_kernel(const float* __restrict__ mean, const float* __restrict__ var,
                               const float* __restrict__ gamma, const float* __restrict__ beta,
                               float eps, float momentum, float* __restrict__ moving_mean,
                               float* __restrict__ moving_var, float* __restrict__ scale,
                               float* __restrict__ shift, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float m = mean[c], v = var[c];
  const float inv = gamma[c] * __frsqrt_rn(v + eps);
  scale[c] = inv;
  shift[c] = beta[c] - m * inv;
  if (moving_mean) {
    const float decay = 1.0f - momentum;
    moving_mean[c] = moving_mean[c] - (moving_mean[c] - m) * decay;
    moving_var[c] = moving_var[c] - (moving_var[c] - v) * decay;
  }
}

// DROP: Keras Dropout between the BatchNorm and the activation, out = prelu(m * scale * bn(h)) (dropout.cuh).
template <int VEC, bool DROP>
__global__ void __launch_bounds__(256) bn_prelu_fwd_kernel(
    const float* __restrict__ h, int64_t ldh, const float* __restrict__ scale,
    const float* __restrict__ shift, const float* __restrict__ alpha, float* __restrict__ out,
    int64_t ldo, int64_t M, int C, float* __restrict__ amax, Dropout d) {
  const int cpr = (C + VEC - 1) / VEC;   // column groups per row
  const int64_t total = M * cpr;
  float mx = 0.f;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = idx / cpr;
    const int c = static_cast<int>(idx - r * cpr) * VEC;
    if (DROP) {
      const unsigned bits = dropout_keep4(d, r, c >> 2) >> (c & 3);
      float v[VEC];
      if (VEC == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(h + r * ldh + c));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
        v[0] = __ldg(h + r * ldh + c);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        const float z = dropout_apply(d, bits, k, fmaf(v[k], __ldg(scale + c + k), __ldg(shift + c + k)));
        v[k] = alpha ? (z > 0.f ? z : __ldg(alpha + c + k) * z) : z;
        mx = fmaxf(mx, fabsf(v[k]));
      }
      if (VEC == 4) *reinterpret_cast<float4*>(out + r * ldo + c) = make_float4(v[0], v[1], v[2], v[3]);
      else out[r * ldo + c] = v[0];
    } else if (VEC == 4) {
      float4 v = __ldg(reinterpret_cast<const float4*>(h + r * ldh + c));
      const float4 sc = __ldg(reinterpret_cast<const float4*>(scale + c));
      const float4 sh = __ldg(reinterpret_cast<const float4*>(shift + c));
      if (alpha) {
        const float4 al = __ldg(reinterpret_cast<const float4*>(alpha + c));
        v.x = bn_prelu(v.x, sc.x, sh.x, al.x); v.y = bn_prelu(v.y, sc.y, sh.y, al.y);
        v.z = bn_prelu(v.z, sc.z, sh.z, al.z); v.w = bn_prelu(v.w, sc.w, sh.w, al.w);
      } else {
        v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y);
        v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
      }
      *reinterpret_cast<float4*>(out + r * ldo + c) = v;
      mx = amax4(mx, v);
    } else {
      const float z = fmaf(__ldg(h + r * ldh + c), __ldg(scale + c), __ldg(shift + c));
      const float o = alpha ? (z > 0.f ? z : __ldg(alpha + c) * z) : z;
      out[r * ldo + c] = o;
      mx = fmaxf(mx, fabsf(o));
    }
  }
  amax_commit(mx, amax);
}

// Backward pass 1: per column S1 = sum dz, S2 = sum dz*xhat, S3 = sum da*min(z,0), with
// z = gamma*xhat + beta, dz = da * slope(z).  DROP: with zd = m*scale*z the block's output is prelu(zd), so
// dz = m*scale*slope(zd)*da and S3 sums da*min(zd,0); m is regenerated from the mask function.
template <int VEC, bool DROP>
__global__ void __launch_bounds__(kBnThreads) bn_bwd_partial_kernel(
    const float* __restrict__ da, int64_t ldda, const float* __restrict__ h, int64_t ldh,
    const float* __restrict__ mean, const float* __restrict__ var, const float* __restrict__ gamma,
    const float* __restrict__ beta, const float* __restrict__ alpha, float eps, int64_t M, int C,
    int64_t rows_per_split, double* __restrict__ ws, Dropout d) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + lane) * VEC;
  const int64_t rb = blockIdx.y * rows_per_split;
  int64_t re = rb + rows_per_split;
  if (re > M) re = M;
  double acc[3 * VEC];
#pragma unroll
  for (int k = 0; k < 3 * VEC; ++k) acc[k] = 0.0;
  if (c < C) {
    float mu[VEC], rs[VEC], ga[VEC], be[VEC], al[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      mu[k] = __ldg(mean + c + k);
      rs[k] = __frsqrt_rn(__ldg(var + c + k) + eps);
      ga[k] = __ldg(gamma + c + k);
      be[k] = __ldg(beta + c + k);
      al[k] = alpha ? __ldg(alpha + c + k) : 1.f;
    }
    // Four rows per step: their contributions are formed and pre-summed in fp32 and folded into the fp64 column
    // accumulators once per step.  One F2F + DADD/DFMA per element made this pass conversion-bound (331 us for
    // 1.06 GB = 3.2 TB/s; the fp64-accumulating statistics pass with a third of the conversions runs at 7.3 TB/s);
    // a four-term fp32 partial sum costs ~1e-7 relative, far inside the 1e-5 budget.
    auto term = [&](float hvk, float gvk, int k, unsigned bits, float& t1, float& t2, float& t3) {
      const float xhat = (hvk - mu[k]) * rs[k];
      float z = fmaf(ga[k], xhat, be[k]);
      if (DROP) z = dropout_apply(d, bits, k, z);
      float dz = gvk;
      t3 = 0.f;
      if (alpha) {
        dz = z > 0.f ? gvk : (z < 0.f ? gvk * al[k] : 0.f);
        t3 = gvk * fminf(z, 0.f);
      }
      if (DROP) dz = dropout_apply(d, bits, k, dz);
      t1 = dz;
      t2 = dz * xhat;
    };
    int64_t r = rb + warp;
    for (; r + 24 < re; r += 32) {
      float hv[4][VEC], gv[4][VEC];
      unsigned bits[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (DROP) bits[u] = dropout_keep4(d, r + 8 * u, c >> 2) >> (c & 3);
        if (VEC == 4) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(h + (r + 8 * u) * ldh + c));
          const float4 g = __ldg(reinterpret_cast<const float4*>(da + (r + 8 * u) * ldda + c));
          hv[u][0] = t.x; hv[u][1] = t.y; hv[u][2] = t.z; hv[u][3] = t.w;
          gv[u][0] = g.x; gv[u][1] = g.y; gv[u][2] = g.z; gv[u][3] = g.w;
        } else {
          hv[u][0] = __ldg(h + (r + 8 * u) * ldh + c);
          gv[u][0] = __ldg(da + (r + 8 * u) * ldda + c);
        }
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        float a1[4], a2[4], a3[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) term(hv[u][k], gv[u][k], k, bits[u], a1[u], a2[u], a3[u]);
        acc[3 * k] += static_cast<double>((a1[0] + a1[1]) + (a1[2] + a1[3]));
        acc[3 * k + 1] += static_cast<double>((a2[0] + a2[1]) + (a2[2] + a2[3]));
        if (alpha) acc[3 * k + 2] += static_cast<double>((a3[0] + a3[1]) + (a3[2] + a3[3]));
      }
    }
    for (; r < re; r += 8) {
      float hv[VEC], gv[VEC];
      const unsigned bits = DROP ? dropout_keep4(d, r, c >> 2) >> (c & 3) : 0u;
      if (VEC == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(h + r * ldh + c));
        const float4 u = __ldg(reinterpret_cast<const float4*>(da + r * ldda + c));
        hv[0] = t.x; hv[1] = t.y; hv[2] = t.z; hv[3] = t.w;
        gv[0] = u.x; gv[1] = u.y; gv[2] = u.z; gv[3] = u.w;
      } else {
        hv[0] = __ldg(h + r * ldh + c);
        gv[0] = __ldg(da + r * ldda + c);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        float t1, t2, t3;
        term(hv[k], gv[k], k, bits, t1, t2, t3);
        acc[3 * k] += static_cast<double>(t1);
        acc[3 * k + 1] += static_cast<double>(t2);
        if (alpha) acc[3 * k + 2] += static_cast<double>(t3);
      }
    }
  }
  block_store_partials<3 * VEC>(acc, ws + (static_cast<int64_t>(blockIdx.y) * C + c) * 3, 0, 0, c < C);
}

// Per column for the apply pass: coef[4c..4c+3] = {S1/M, S2/M, rstd, gamma*rstd}; dgamma/dbeta/dalpha
// are written here.
__global__ void __launch_bounds__(256) bn_bwd_final_kernel(const double* __restrict__ ws, int splits, int C, int64_t M,
                                                           const float* __restrict__ var, const float* __restrict__ gamma,
                                                           float eps, float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                           float* __restrict__ dalpha, float* __restrict__ coef) {
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int k = lane; k < splits; k += 32) {
    const double* p = ws + (static_cast<int64_t>(k) * C + c) * 3;
    s1 += p[0]; s2 += p[1]; s3 += p[2];
  }
  s1 = warp_sum_fixed(s1);
  s2 = warp_sum_fixed(s2);
  s3 = warp_sum_fixed(s3);
  if (lane != 0) return;
  if (dbeta) dbeta[c] = static_cast<float>(s1);
  if (dgamma) dgamma[c] = static_cast<float>(s2);
  if (dalpha) dalpha[c] = static_cast<float>(s3);
  const float rs = __frsqrt_rn(var[c] + eps);
  coef[4 * c] = static_cast<float>(s1 / static_cast<double>(M));
  coef[4 * c + 1] = static_cast<float>(s2 / static_cast<double>(M));
  coef[4 * c + 2] = rs;
  coef[4 * c + 3] = gamma[c] * rs;
}

__global__ void __launch_bounds__(256) bn_bwd_sums_kernel(const double* __restrict__ ws, int splits, int C, int64_t M,
                                                          double* __restrict__ sums) {
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int k = lane; k < splits; k += 32) {
    const double* p = ws + (static_cast<int64_t>(k) * C + c) * 3;
    s1 += p[0]; s2 += p[1]; s3 += p[2];
  }
  s1 = warp_sum_fixed(s1);
  s2 = warp_sum_fixed(s2);
  s3 = warp_sum_fixed(s3);
  if (lane == 0) {
    sums[c] = s1;
    sums[C + c] = s2;
    sums[2 * C + c] = s3;
    if (c == 0) sums[3 * C] = static_cast<double>(M);
  }
}

// From GLOBAL sums: the parameter gradients are divided by the world size because the caller's SUM all-reduce of the
// flat gradient buffer adds the (identical) values of all ranks up again.
__global__ void bn_bwd_finish_kernel(const double* __restrict__ sums, int C, double inv_world, const float* __restrict__ var,
                                     const float* __restrict__ gamma, float eps, float* __restrict__ dgamma,
                                     float* __restrict__ dbeta, float* __restrict__ dalpha, float* __restrict__ coef) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double Mg = sums[3 * C];
  const double s1 = sums[c], s2 = sums[C + c], s3 = sums[2 * C + c];
  if (dbeta) dbeta[c] = static_cast<float>(s1 * inv_world);
  if (dgamma) dgamma[c] = static_cast<float>(s2 * inv_world);
  if (dalpha) dalpha[c] = static_cast<float>(s3 * inv_world);
  const float rs = __frsqrt_rn(var[c] + eps);
  coef[4 * c] = static_cast<float>(s1 / Mg);
  coef[4 * c + 1] = static_cast<float>(s2 / Mg);
  coef[4 * c + 2] = rs;
  coef[4 * c + 3] = gamma[c] * rs;
}

// Backward pass 2: dh = gamma*rstd*(dz - S1/M - xhat*S2/M).  Same thread->column mapping as the
// reduction pass (lane = VEC columns, 8 row warps per block, grid.y row splits), so the per-column
// coefficients stay in registers for the whole row loop.  DROP: dz as in bn_bwd_partial_kernel.
template <int VEC, bool DROP>
__global__ void __launch_bounds__(kBnThreads) bn_bwd_apply_kernel(
    const float* __restrict__ da, int64_t ldda, const float* __restrict__ h, int64_t ldh,
    const float* __restrict__ mean, const float* __restrict__ gamma, const float* __restrict__ beta,
    const float* __restrict__ alpha, const float* __restrict__ coef, float* __restrict__ dh, int64_t lddh,
    int64_t M, int C, int64_t rows_per_split, double* __restrict__ colsum_ws, float* __restrict__ amax, Dropout d) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + lane) * VEC;
  const bool valid = c < C;
  float mx = 0.f;
  const int64_t rb = blockIdx.y * rows_per_split;
  int64_t re = rb + rows_per_split;
  if (re > M) re = M;
  // optional: column sums of dh (= the bias gradient of the dense layer in front of this BatchNorm), folded into
  // this pass instead of a separate read of dh
  double csum[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) csum[k] = 0.0;
  if (valid) {
    float mu[VEC], rs[VEC], ga[VEC], be[VEC], al[VEC], c1[VEC], c2[VEC], gr[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      mu[k] = __ldg(mean + c + k);
      ga[k] = __ldg(gamma + c + k);
      be[k] = __ldg(beta + c + k);
      al[k] = alpha ? __ldg(alpha + c + k) : 1.f;
      c1[k] = __ldg(coef + 4 * (c + k));
      c2[k] = __ldg(coef + 4 * (c + k) + 1);
      rs[k] = __ldg(coef + 4 * (c + k) + 2);
      gr[k] = __ldg(coef + 4 * (c + k) + 3);
    }
    auto out = [&](float hvk, float gvk, int k, unsigned bits) {
      const float xhat = (hvk - mu[k]) * rs[k];
      float z = fmaf(ga[k], xhat, be[k]);
      if (DROP) z = dropout_apply(d, bits, k, z);
      float dz = gvk;
      if (alpha) dz = z > 0.f ? gvk : (z < 0.f ? gvk * al[k] : 0.f);
      if (DROP) dz = dropout_apply(d, bits, k, dz);
      return gr[k] * (dz - c1[k] - xhat * c2[k]);
    };
    int64_t r = rb + warp;
    for (; r + 24 < re; r += 32) {                       // four rows per step: eight 128-bit loads in flight
      float hv[4][VEC], gv[4][VEC], o[4][VEC];
      unsigned bits[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (DROP) bits[u] = dropout_keep4(d, r + 8 * u, c >> 2) >> (c & 3);
        if (VEC == 4) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(h + (r + 8 * u) * ldh + c));
          const float4 g = __ldg(reinterpret_cast<const float4*>(da + (r + 8 * u) * ldda + c));
          hv[u][0] = t.x; hv[u][1] = t.y; hv[u][2] = t.z; hv[u][3] = t.w;
          gv[u][0] = g.x; gv[u][1] = g.y; gv[u][2] = g.z; gv[u][3] = g.w;
        } else {
          hv[u][0] = __ldg(h + (r + 8 * u) * ldh + c);
          gv[u][0] = __ldg(da + (r + 8 * u) * ldda + c);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) { o[u][k] = out(hv[u][k], gv[u][k], k, bits[u]); mx = fmaxf(mx, fabsf(o[u][k])); }
        if (VEC == 4) *reinterpret_cast<float4*>(dh + (r + 8 * u) * lddh + c) = make_float4(o[u][0], o[u][1], o[u][2], o[u][3]);
        else dh[(r + 8 * u) * lddh + c] = o[u][0];
      }
      if (colsum_ws) {                                   // fp32 over the four rows, one fp64 fold
#pragma unroll
        for (int k = 0; k < VEC; ++k) csum[k] += static_cast<double>((o[0][k] + o[1][k]) + (o[2][k] + o[3][k]));
      }
    }
    for (; r < re; r += 8) {
      float hv[VEC], gv[VEC], o[VEC];
      const unsigned bits = DROP ? dropout_keep4(d, r, c >> 2) >> (c & 3) : 0u;
      if (VEC == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(h + r * ldh + c));
        const float4 u = __ldg(reinterpret_cast<const float4*>(da + r * ldda + c));
        hv[0] = t.x; hv[1] = t.y; hv[2] = t.z; hv[3] = t.w;
        gv[0] = u.x; gv[1] = u.y; gv[2] = u.z; gv[3] = u.w;
      } else {
        hv[0] = __ldg(h + r * ldh + c);
        gv[0] = __ldg(da + r * ldda + c);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) { o[k] = out(hv[k], gv[k], k, bits); mx = fmaxf(mx, fabsf(o[k])); }
      if (VEC == 4) *reinterpret_cast<float4*>(dh + r * lddh + c) = make_float4(o[0], o[1], o[2], o[3]);
      else dh[r * lddh + c] = o[0];
      if (colsum_ws) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) csum[k] += static_cast<double>(o[k]);
      }
    }
  }
  amax_commit(mx, amax);
  if (colsum_ws) block_store_partials<VEC>(csum, colsum_ws + static_cast<int64_t>(blockIdx.y) * C + c, 0, 0, valid);
}

__global__ void __launch_bounds__(256) bn_bwd_dbias_final_kernel(const double* __restrict__ ws, int splits, int C,
                                                                 float* __restrict__ dbias) {
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  double s = 0.0;
  for (int k = lane; k < splits; k += 32) s += ws[static_cast<int64_t>(k) * C + c];
  s = warp_sum_fixed(s);
  if (lane == 0) dbias[c] = static_cast<float>(s);
}

}  // namespace gcs

using namespace gcs;

static inline int64_t elementwise_blocks(int64_t work) {
  int64_t b = ceil_div(work, 256);
  const int64_t cap = 16LL * sm_count();
  return b < 1 ? 1 : (b > cap ? cap : b);
}

extern "C" int64_t gcs_bn_workspace_bytes(int64_t M, int32_t C) {
  if (M < 0 || C <= 0) return 0;
  return round_up(bn_max_splits(M) * C * 3 * static_cast<int64_t>(sizeof(double)), 256) +
         round_up(4LL * C * sizeof(float), 256) + round_up((3LL * C + 1) * sizeof(double), 256);   // partials | coef | sync sums
}

// Per-split fp64 partials -> mean / biased variance (through the synchronised-BatchNorm hook when one is installed).
static int bn_stats_finish(const double* ws, int splits, int C, int64_t M, float* mean, float* var, void* workspace,
                           gcs_stream stream) {
  cudaStream_t st = as_stream(stream);
  const SyncHook& hook = sync_hook();
  if (hook.fn) {
    double* sums = reinterpret_cast<double*>(static_cast<char*>(workspace) +
                                             round_up(bn_max_splits(M) * C * 3 * static_cast<int64_t>(sizeof(double)), 256) +
                                             round_up(4LL * C * sizeof(float), 256));
    bn_stats_sums_kernel<<<static_cast<unsigned>(ceil_div(C, 8)), 256, 0, st>>>(ws, splits, C, M, sums);
    GCS_CHECK_LAUNCH("bn_stats_sums_kernel");
    if (hook.fn(sums, 2LL * C + 1, stream, hook.user) != 0) return fail(GCS_ERR_CUDA, "gcs_bn_stats: the all-reduce hook failed");
    bn_stats_finish_kernel<<<static_cast<unsigned>(ceil_div(C, 128)), 128, 0, st>>>(sums, C, mean, var);
    GCS_CHECK_LAUNCH("bn_stats_finish_kernel");
    return GCS_OK;
  }
  bn_stats_final_kernel<<<static_cast<unsigned>(ceil_div(C, 8)), 256, 0, st>>>(ws, splits, C, M, mean, var);
  GCS_CHECK_LAUNCH("bn_stats_final_kernel");
  return GCS_OK;
}

namespace gcs {
// part: [ceil(M/32)][C] float2 written by the dense layer's epilogue (rows >= M excluded there).
int bn_stats_from_partials(const float* part, int64_t M, int C, float* mean, float* var, void* workspace,
                           int64_t workspace_bytes, gcs_stream stream) {
  if (workspace_bytes < gcs_bn_workspace_bytes(M, C)) return fail(GCS_ERR_WORKSPACE, "bn_stats_from_partials: workspace too small");
  const int64_t groups = ceil_div(M, 32);
  int64_t splits = ceil_div(groups, 64);                     // >= 8 groups per warp
  const int64_t cap = bn_max_splits(M) < 64 ? bn_max_splits(M) : 64;
  if (splits > cap) splits = cap;
  if (splits < 1) splits = 1;
  double* ws = static_cast<double*>(workspace);
  dim3 grid(static_cast<unsigned>(ceil_div(C, 32)), static_cast<unsigned>(splits));
  bn_stats_from_part_kernel<<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float2*>(part), groups, C,
                                                                static_cast<int>(splits), ws, M);
  GCS_CHECK_LAUNCH("bn_stats_from_part_kernel");
  return bn_stats_finish(ws, static_cast<int>(splits), C, M, mean, var, workspace, stream);
}
}  // namespace gcs

extern "C" int gcs_bn_stats(const float* h, int64_t ldh, int64_t M, int32_t C, float* mean, float* var,
                            void* workspace, int64_t workspace_bytes, gcs_stream stream) {
  GCS_CHECK_ARG(M > 0 && C > 0, "gcs_bn_stats: needs at least one row (M=%lld, C=%d)", (long long)M, C);
  GCS_CHECK_ARG(h && mean && var && workspace && ldh >= C, "gcs_bn_stats: bad pointer / leading dimension");
  if (workspace_bytes < gcs_bn_workspace_bytes(M, C))
    return fail(GCS_ERR_WORKSPACE, "gcs_bn_stats: workspace %lld < %lld bytes", (long long)workspace_bytes, (long long)gcs_bn_workspace_bytes(M, C));
  GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 7u) == 0, "gcs_bn_stats: workspace must be 8-byte aligned");
  const bool vec = (C % 4 == 0) && (ldh % 4 == 0) && aligned16(h);
  const BnGrid g = bn_grid(M, C, vec);
  cudaStream_t st = as_stream(stream);
  double* ws = static_cast<double*>(workspace);
  dim3 grid(g.col_blocks, g.splits);
  if (vec) bn_stats_partial_kernel<4><<<grid, kBnThreads, 0, st>>>(h, ldh, M, C, g.rows_per_split, ws);
  else bn_stats_partial_kernel<1><<<grid, kBnThreads, 0, st>>>(h, ldh, M, C, g.rows_per_split, ws);
  GCS_CHECK_LAUNCH("bn_stats_partial_kernel");
  return bn_stats_finish(ws, g.splits, C, M, mean, var, workspace, stream);
}

extern "C" int gcs_bn_fold(const float* mean, const float* var, const float* gamma, const float* beta,
                           float eps, float momentum, float* moving_mean, float* moving_var, float* scale,
                           float* shift, int32_t C, gcs_stream stream) {
  GCS_CHECK_ARG(C > 0 && mean && var && gamma && beta && scale && shift, "gcs_bn_fold: bad argument");
  GCS_CHECK_ARG((moving_mean != nullptr) == (moving_var != nullptr), "gcs_bn_fold: moving_mean/moving_var must both be set or both NULL");
  bn_fold_kernel<<<static_cast<unsigned>(ceil_div(C, 128)), 128, 0, as_stream(stream)>>>(mean, var, gamma, beta, eps, momentum, moving_mean, moving_var, scale, shift, C);
  GCS_CHECK_LAUNCH("bn_fold_kernel");
  return GCS_OK;
}

namespace gcs {
// gcs_bn_prelu_fwd with the block's dropout (drop == NULL or threshold 0: none).
int bn_prelu_fwd(const float* h, int64_t ldh, const float* scale, const float* shift, const float* alpha, float* out,
                 int64_t ldo, int64_t M, int32_t C, const Dropout* drop, gcs_stream stream) {
  GCS_CHECK_ARG(M >= 0 && C > 0, "gcs_bn_prelu_fwd: bad size");
  if (M == 0) return GCS_OK;
  GCS_CHECK_ARG(h && scale && shift && out && ldh >= C && ldo >= C, "gcs_bn_prelu_fwd: bad pointer / leading dimension");
  const bool vec = (C % 4 == 0) && (ldh % 4 == 0) && (ldo % 4 == 0) && aligned16(h) && aligned16(out) &&
                   aligned16(scale) && aligned16(shift) && (!alpha || aligned16(alpha));
  cudaStream_t st = as_stream(stream);
  const unsigned b4 = static_cast<unsigned>(elementwise_blocks(M * (C / 4))), b1 = static_cast<unsigned>(elementwise_blocks(M * C));
  float* amax = amax_sink().produce;
  if (drop && drop->threshold) {
    if (vec) bn_prelu_fwd_kernel<4, true><<<b4, 256, 0, st>>>(h, ldh, scale, shift, alpha, out, ldo, M, C, amax, *drop);
    else bn_prelu_fwd_kernel<1, true><<<b1, 256, 0, st>>>(h, ldh, scale, shift, alpha, out, ldo, M, C, amax, *drop);
  } else {
    if (vec) bn_prelu_fwd_kernel<4, false><<<b4, 256, 0, st>>>(h, ldh, scale, shift, alpha, out, ldo, M, C, amax, Dropout{});
    else bn_prelu_fwd_kernel<1, false><<<b1, 256, 0, st>>>(h, ldh, scale, shift, alpha, out, ldo, M, C, amax, Dropout{});
  }
  GCS_CHECK_LAUNCH("bn_prelu_fwd_kernel");
  return GCS_OK;
}
}  // namespace gcs

extern "C" int gcs_bn_prelu_fwd(const float* h, int64_t ldh, const float* scale, const float* shift,
                                const float* alpha, float* out, int64_t ldo, int64_t M, int32_t C,
                                gcs_stream stream) {
  return gcs::bn_prelu_fwd(h, ldh, scale, shift, alpha, out, ldo, M, C, nullptr, stream);
}

namespace gcs {
// gcs_bn_prelu_bwd of a block whose forward applied `drop` (NULL or threshold 0: none).
int bn_prelu_bwd(const float* da, int64_t ldda, const float* h, int64_t ldh, const float* mean, const float* var,
                 const float* gamma, const float* beta, const float* alpha, float eps, float* dh, int64_t lddh,
                 float* dgamma, float* dbeta, float* dalpha, float* dbias, int64_t M, int32_t C, void* workspace,
                 int64_t workspace_bytes, const Dropout* drop, gcs_stream stream) {
  GCS_CHECK_ARG(M > 0 && C > 0, "gcs_bn_prelu_bwd: needs at least one row");
  GCS_CHECK_ARG(da && h && mean && var && gamma && beta && dh && workspace, "gcs_bn_prelu_bwd: null pointer");
  GCS_CHECK_ARG(ldda >= C && ldh >= C && lddh >= C, "gcs_bn_prelu_bwd: leading dimension smaller than C");
  GCS_CHECK_ARG(!dalpha || alpha, "gcs_bn_prelu_bwd: dalpha requested without alpha");
  if (workspace_bytes < gcs_bn_workspace_bytes(M, C))
    return fail(GCS_ERR_WORKSPACE, "gcs_bn_prelu_bwd: workspace %lld < %lld bytes", (long long)workspace_bytes, (long long)gcs_bn_workspace_bytes(M, C));
  GCS_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 7u) == 0, "gcs_bn_prelu_bwd: workspace must be 8-byte aligned");
  const bool vec = (C % 4 == 0) && (ldda % 4 == 0) && (ldh % 4 == 0) && (lddh % 4 == 0) && aligned16(da) &&
                   aligned16(h) && aligned16(dh);
  const BnGrid g = bn_grid(M, C, vec);
  cudaStream_t st = as_stream(stream);
  double* ws = static_cast<double*>(workspace);
  float* coef = reinterpret_cast<float*>(static_cast<char*>(workspace) +
                                         round_up(bn_max_splits(M) * C * 3 * static_cast<int64_t>(sizeof(double)), 256));
  dim3 grid(g.col_blocks, g.splits);
  const bool dr = drop && drop->threshold;
  const Dropout dd = dr ? *drop : Dropout{};
  if (dr) {
    if (vec) bn_bwd_partial_kernel<4, true><<<grid, kBnThreads, 0, st>>>(da, ldda, h, ldh, mean, var, gamma, beta, alpha, eps, M, C, g.rows_per_split, ws, dd);
    else bn_bwd_partial_kernel<1, true><<<grid, kBnThreads, 0, st>>>(da, ldda, h, ldh, mean, var, gamma, beta, alpha, eps, M, C, g.rows_per_split, ws, dd);
  } else {
    if (vec) bn_bwd_partial_kernel<4, false><<<grid, kBnThreads, 0, st>>>(da, ldda, h, ldh, mean, var, gamma, beta, alpha, eps, M, C, g.rows_per_split, ws, dd);
    else bn_bwd_partial_kernel<1, false><<<grid, kBnThreads, 0, st>>>(da, ldda, h, ldh, mean, var, gamma, beta, alpha, eps, M, C, g.rows_per_split, ws, dd);
  }
  GCS_CHECK_LAUNCH("bn_bwd_partial_kernel");
  const SyncHook& hook = sync_hook();
  if (hook.fn) {
    double* sums = reinterpret_cast<double*>(reinterpret_cast<char*>(coef) + round_up(4LL * C * sizeof(float), 256));
    bn_bwd_sums_kernel<<<static_cast<unsigned>(ceil_div(C, 8)), 256, 0, st>>>(ws, g.splits, C, M, sums);
    GCS_CHECK_LAUNCH("bn_bwd_sums_kernel");
    if (hook.fn(sums, 3LL * C + 1, stream, hook.user) != 0) return fail(GCS_ERR_CUDA, "gcs_bn_prelu_bwd: the all-reduce hook failed");
    bn_bwd_finish_kernel<<<static_cast<unsigned>(ceil_div(C, 128)), 128, 0, st>>>(sums, C, 1.0 / hook.world, var, gamma, eps, dgamma, dbeta, dalpha, coef);
    GCS_CHECK_LAUNCH("bn_bwd_finish_kernel");
  } else {
    bn_bwd_final_kernel<<<static_cast<unsigned>(ceil_div(C, 8)), 256, 0, st>>>(ws, g.splits, C, M, var, gamma, eps, dgamma, dbeta, dalpha, coef);
    GCS_CHECK_LAUNCH("bn_bwd_final_kernel");
  }
  double* cws = dbias ? ws : nullptr;          // the reduction partials are consumed: reuse their space
  float* amax = amax_sink().produce;
  if (dr) {
    if (vec) bn_bwd_apply_kernel<4, true><<<grid, kBnThreads, 0, st>>>(da, ldda, h, ldh, mean, gamma, beta, alpha, coef, dh, lddh, M, C, g.rows_per_split, cws, amax, dd);
    else bn_bwd_apply_kernel<1, true><<<grid, kBnThreads, 0, st>>>(da, ldda, h, ldh, mean, gamma, beta, alpha, coef, dh, lddh, M, C, g.rows_per_split, cws, amax, dd);
  } else {
    if (vec) bn_bwd_apply_kernel<4, false><<<grid, kBnThreads, 0, st>>>(da, ldda, h, ldh, mean, gamma, beta, alpha, coef, dh, lddh, M, C, g.rows_per_split, cws, amax, dd);
    else bn_bwd_apply_kernel<1, false><<<grid, kBnThreads, 0, st>>>(da, ldda, h, ldh, mean, gamma, beta, alpha, coef, dh, lddh, M, C, g.rows_per_split, cws, amax, dd);
  }
  GCS_CHECK_LAUNCH("bn_bwd_apply_kernel");
  if (dbias) {
    bn_bwd_dbias_final_kernel<<<static_cast<unsigned>(ceil_div(C, 8)), 256, 0, st>>>(ws, g.splits, C, dbias);
    GCS_CHECK_LAUNCH("bn_bwd_dbias_final_kernel");
  }
  return GCS_OK;
}
}  // namespace gcs

extern "C" int gcs_bn_prelu_bwd(const float* da, int64_t ldda, const float* h, int64_t ldh, const float* mean,
                                const float* var, const float* gamma, const float* beta, const float* alpha,
                                float eps, float* dh, int64_t lddh, float* dgamma, float* dbeta, float* dalpha,
                                float* dbias, int64_t M, int32_t C, void* workspace, int64_t workspace_bytes,
                                gcs_stream stream) {
  return gcs::bn_prelu_bwd(da, ldda, h, ldh, mean, var, gamma, beta, alpha, eps, dh, lddh, dgamma, dbeta, dalpha, dbias,
                           M, C, workspace, workspace_bytes, nullptr, stream);
}

// Test hook (not part of the drop-in surface): the PReLU branch every element takes in the BatchNorm backward above,
// computed with the same float32 expressions (xhat = (h - mean) * rsqrt(var + eps); z = fma(gamma, xhat, beta)):
// out[r, c] = 1 for z > 0, -1 for z < 0, 0 for z == 0.  The parity tests hand it to the float64 oracle so that both
// sides differentiate the same branch of the activation at inputs within rounding of its kink.
namespace gcs {
__global__ void prelu_branch_kernel(const float* __restrict__ h, int64_t ldh, const float* __restrict__ mean,
                                    const float* __restrict__ var, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, float eps, int64_t M, int C, int8_t* __restrict__ out) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= M * C) return;
  const int64_t r = i / C;
  const int c = static_cast<int>(i - r * C);
  const float rs = __frsqrt_rn(__ldg(var + c) + eps);
  const float xhat = (__ldg(h + r * ldh + c) - __ldg(mean + c)) * rs;
  const float z = fmaf(__ldg(gamma + c), xhat, __ldg(beta + c));
  out[i] = z > 0.f ? 1 : (z < 0.f ? -1 : 0);
}
}  // namespace gcs

extern "C" int gcs_debug_prelu_branch(const float* h, int64_t ldh, const float* mean, const float* var, const float* gamma,
                                      const float* beta, float eps, int64_t M, int32_t C, int8_t* out, gcs_stream stream) {
  GCS_CHECK_ARG(h && mean && var && gamma && beta && out && M >= 0 && C > 0 && ldh >= C, "gcs_debug_prelu_branch: bad argument");
  if (M == 0) return GCS_OK;
  const int64_t n = M * C;
  gcs::prelu_branch_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, gcs::as_stream(stream)>>>(h, ldh, mean, var, gamma, beta,
                                                                                                     eps, M, C, out);
  GCS_CHECK_LAUNCH("prelu_branch_kernel");
  return GCS_OK;
}

