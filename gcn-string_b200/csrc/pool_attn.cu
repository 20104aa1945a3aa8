// K4b / K6b — GlobalAttnSumPool (spektral.layers.GlobalAttnSumPool, GeneralGNN(pool='attn_sum')) and its gradient.
//   s_n   = X_n . a                                   a = attn_kernel [W] (Spektral's [W, 1])
//   p_n   = exp(s_n - max_g) / (sum_{m in g} exp(s_m - max_g) + 1e-9)      unsorted_segment_softmax
//   out_g = sum_{n in g} p_n X_n                      (0 for an empty graph)
// Backward with u_g = out_g . dOut_g:
//   ds_n = p_n (X_n . dOut_g - u_g),  dX_n = p_n dOut_g + ds_n a,  da = sum_n ds_n X_n
//
// Both directions are one pass over X.  A thread block owns whole rows of one split of one graph: every thread holds a
// fixed slice of the columns, the row dot products (scores in the forward, X_n . dOut_g in the backward) are summed in
// fp64 - products of two floats are exact there - groups of R rows at a time.  The forward keeps an online softmax (running max, denominator
// and a rescaled [W] accumulator); the backward writes the full dX row and accumulates ds_n X_n in fp64.
// A graph is cut into S splits of equal length, S fixed by (n_rows, n_graphs) alone (one split per kAttnSplitRows rows
// of the average graph): batches of residue graphs run one block per graph, a single long graph (single mode, cfg5)
// spreads over many SMs.  Partial (max, denominator, accumulator) of the splits and the per-split partials of da are
// combined in split order.  No atomics; results are bit-identical run to run.  The running |max| cells of the fp16
// GEMMs (AmaxSink) are neither read nor raised.
#include <math.h>

#include "common.cuh"

namespace gcs {

constexpr int kAttnSplitRows = 512;
constexpr float kSoftmaxEps = 1e-9f;   // Spektral's unsorted_segment_softmax

static int attn_splits(int64_t n_rows, int n_graphs) {
  if (n_graphs <= 0 || n_rows <= 0) return 1;
  const int64_t s = ceil_div(ceil_div(n_rows, n_graphs), kAttnSplitRows);
  return static_cast<int>(s < 1 ? 1 : (s > 65535 ? 65535 : s));
}

// rows per group: keeps the staged rows of a thread at <= 32 floats
template <int VEC, int NV>
__host__ __device__ constexpr int attn_rows() {
  return (32 / (VEC * NV)) > 8 ? 8 : ((32 / (VEC * NV)) < 1 ? 1 : 32 / (VEC * NV));
}

template <int VEC>
__device__ __forceinline__ void load_row(float (&v)[VEC], const float* p) {
  if constexpr (VEC == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
    v[0] = __ldg(p);
  }
}

// the [W] attention kernel: element loads, so that its alignment (it follows the blocks in the flat parameter buffer, at
// any float offset) never decides between the float4 and the scalar path over X
template <int VEC>
__device__ __forceinline__ void load_kernel(float (&v)[VEC], const float* p) {
#pragma unroll
  for (int i = 0; i < VEC; ++i) v[i] = __ldg(p + i);
}

template <int VEC>
__device__ __forceinline__ void store_row(float* p, const float (&v)[VEC]) {
  if constexpr (VEC == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  else p[0] = v[0];
}

// Sum of v[r] over the block, the same value in every thread.  In the warp a reduce-scatter: each halving step
// exchanges half of the values with the lane `off` away (R = 8: 4 + 2 + 1 shuffles, then 2 for the last value), after
// which lane l holds the warp sum of row idx(l); then one thread per row adds the warp sums in warp order.  Every
// partial sum is formed by exactly one lane, so the result is fixed.  red: [2][8][32] and fin: [2][8] doubles, used
// alternately (buf).
template <int R>
__device__ __forceinline__ void block_sum(double (&v)[R], double (*red)[8][32], double (*fin)[8], int buf) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int idx = 0;
  int off = 16;
#pragma unroll
  for (int n = R; n > 1; n >>= 1, off >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int j = 0; j < n / 2; ++j) {
      const double send = hi ? v[j] : v[j + n / 2];
      const double keep = hi ? v[j + n / 2] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
    if (hi) idx += n / 2;
  }
  double t = v[0];
  for (int o = off; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  if ((lane & (32 / R - 1)) == 0) red[buf][idx][warp] = t;
  __syncthreads();
  if (threadIdx.x < R) {
    double a = red[buf][threadIdx.x][0];
    for (int w = 1; w < nw; ++w) a += red[buf][threadIdx.x][w];
    fin[buf][threadIdx.x] = a;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < R; ++r) v[r] = fin[buf][r];
}

__device__ __forceinline__ void split_rows(const int32_t* graph_ptr, int g, int sp, int S, int& r0, int& r1) {
  const int a = __ldg(graph_ptr + g), b = __ldg(graph_ptr + g + 1);
  const int len = b - a;
  const int q = (len + S - 1) / S;
  const int lo = sp * q, hi = lo + q;
  r0 = a + (lo < len ? lo : len);
  r1 = a + (hi < len ? hi : len);
}

// grid (graph, split), block = ceil(W / (VEC*NV)) threads rounded up to a warp.  Thread t owns columns
// (k * blockDim + t) * VEC .. +VEC for k < NV.
template <int VEC, int NV>
__global__ void __launch_bounds__(512, 1) attn_pool_fwd_kernel(
    const float* __restrict__ X, int64_t ldx, const float* __restrict__ a, const int32_t* __restrict__ graph_ptr, int W,
    int S, float* __restrict__ out, int64_t ldo, float* __restrict__ scores, float* __restrict__ gstats,
    float* __restrict__ part_acc, float* __restrict__ part_md) {
  constexpr int R = attn_rows<VEC, NV>();
  __shared__ double red[2][8][32];
  __shared__ double fin[2][8];
  const int g = blockIdx.x, sp = blockIdx.y;
  int r0, r1;
  split_rows(graph_ptr, g, sp, S, r0, r1);
  double av[NV][VEC];
  float acc[NV][VEC];
  bool ok[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int c = (k * blockDim.x + threadIdx.x) * VEC;
    ok[k] = c < W;
    float t[VEC];
    if (ok[k]) load_kernel<VEC>(t, a + c);
#pragma unroll
    for (int v = 0; v < VEC; ++v) { av[k][v] = ok[k] ? static_cast<double>(t[v]) : 0.0; acc[k][v] = 0.f; }
  }
  float m = -INFINITY, den = 0.f;
  int buf = 0;
  for (int r = r0; r < r1; r += R) {
    float x[R][NV][VEC];
    double d[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      d[i] = 0.0;
      const bool row_ok = r + i < r1;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const int c = (k * blockDim.x + threadIdx.x) * VEC;
        if (row_ok && ok[k]) load_row<VEC>(x[i][k], X + static_cast<int64_t>(r + i) * ldx + c);
        else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) x[i][k][v] = 0.f;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
      for (int k = 0; k < NV; ++k)
#pragma unroll
        for (int v = 0; v < VEC; ++v) d[i] = fma(static_cast<double>(x[i][k][v]), av[k][v], d[i]);
    block_sum<R>(d, red, fin, buf);
    buf ^= 1;
    float s[R];
    float mg = m;
#pragma unroll
    for (int i = 0; i < R; ++i) {
      s[i] = static_cast<float>(d[i]);
      if (r + i < r1) {
        mg = fmaxf(mg, s[i]);
        if (scores && threadIdx.x == 0) scores[r + i] = s[i];
      }
    }
    if (mg > m) {                                        // rescale what was accumulated under the old max
      const float f = expf(m - mg);                      // m = -inf: f = 0, and den / acc are 0 anyway
      den *= f;
#pragma unroll
      for (int k = 0; k < NV; ++k)
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[k][v] *= f;
      m = mg;
    }
#pragma unroll
    for (int i = 0; i < R; ++i) {
      if (r + i < r1) {
        const float e = expf(s[i] - m);
        den += e;
#pragma unroll
        for (int k = 0; k < NV; ++k)
#pragma unroll
          for (int v = 0; v < VEC; ++v) acc[k][v] = fmaf(e, x[i][k][v], acc[k][v]);
      }
    }
  }
  if (S == 1) {
    const float inv = 1.f / (den + kSoftmaxEps);         // empty graph: acc = 0 -> out = 0
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (!ok[k]) continue;
      float o[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) o[v] = acc[k][v] * inv;
      store_row<VEC>(out + static_cast<int64_t>(g) * ldo + (k * blockDim.x + threadIdx.x) * VEC, o);
    }
    if (gstats && threadIdx.x == 0) {
      gstats[2 * g] = r1 > r0 ? m : 0.f;
      gstats[2 * g + 1] = den;
    }
  } else {
    const int64_t slot = static_cast<int64_t>(g) * S + sp;
#pragma unroll
    for (int k = 0; k < NV; ++k)
      if (ok[k]) store_row<VEC>(part_acc + slot * W + (k * blockDim.x + threadIdx.x) * VEC, acc[k]);
    if (threadIdx.x == 0) {
      part_md[2 * slot] = m;                             // -inf for an empty split (den = 0)
      part_md[2 * slot + 1] = den;
    }
  }
}

// grid (graph, column tile of 256): the S partials of a graph, in split order.
__global__ void __launch_bounds__(256) attn_pool_combine_kernel(const float* __restrict__ part_acc,
                                                                const float* __restrict__ part_md, int S, int W,
                                                                float* __restrict__ out, int64_t ldo,
                                                                float* __restrict__ gstats) {
  const int g = blockIdx.x;
  const int c = blockIdx.y * 256 + threadIdx.x;
  const float* md = part_md + 2LL * g * S;
  float M = -INFINITY;
  for (int s = 0; s < S; ++s)
    if (md[2 * s + 1] > 0.f) M = fmaxf(M, md[2 * s]);
  float den = 0.f;
  for (int s = 0; s < S; ++s)
    if (md[2 * s + 1] > 0.f) den = fmaf(md[2 * s + 1], expf(md[2 * s] - M), den);
  if (gstats && blockIdx.y == 0 && threadIdx.x == 0) {
    gstats[2 * g] = den > 0.f ? M : 0.f;
    gstats[2 * g + 1] = den;
  }
  if (c >= W) return;
  float acc = 0.f;
  for (int s = 0; s < S; ++s)
    if (md[2 * s + 1] > 0.f) acc = fmaf(part_acc[(static_cast<int64_t>(g) * S + s) * W + c], expf(md[2 * s] - M), acc);
  out[static_cast<int64_t>(g) * ldo + c] = acc / (den + kSoftmaxEps);
}

template <int VEC, int NV>
__global__ void __launch_bounds__(512, 1) attn_pool_bwd_kernel(
    const float* __restrict__ dout, int64_t lddo, const float* __restrict__ X, int64_t ldx, const float* __restrict__ a,
    const int32_t* __restrict__ graph_ptr, int W, int S, const float* __restrict__ out, int64_t ldo,
    const float* __restrict__ scores, const float* __restrict__ gstats, float* __restrict__ dX, int64_t lddx,
    double* __restrict__ part_da) {
  constexpr int R = VEC * NV >= 16 ? 1 : attn_rows<VEC, NV>();   // the fp64 da accumulators need the room
  __shared__ double red[2][8][32];
  __shared__ double fin[2][8];
  const int g = blockIdx.x, sp = blockIdx.y;
  int r0, r1;
  split_rows(graph_ptr, g, sp, S, r0, r1);
  float av[NV][VEC], dov[NV][VEC];
  double da[NV][VEC];
  bool ok[NV];
  double u[1] = {0.0};
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int c = (k * blockDim.x + threadIdx.x) * VEC;
    ok[k] = c < W;
    float o[VEC];
    if (ok[k]) {
      load_kernel<VEC>(av[k], a + c);
      load_row<VEC>(dov[k], dout + static_cast<int64_t>(g) * lddo + c);
      load_row<VEC>(o, out + static_cast<int64_t>(g) * ldo + c);
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      if (!ok[k]) { av[k][v] = 0.f; dov[k][v] = 0.f; o[v] = 0.f; }
      da[k][v] = 0.0;
      u[0] = fma(static_cast<double>(o[v]), static_cast<double>(dov[k][v]), u[0]);
    }
  }
  block_sum<1>(u, red, fin, 0);
  int buf = 1;
  const float M = __ldg(gstats + 2 * g);
  const float inv = 1.f / (__ldg(gstats + 2 * g + 1) + kSoftmaxEps);
  for (int r = r0; r < r1; r += R) {
    float x[R][NV][VEC];
    double d[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      d[i] = 0.0;
      const bool row_ok = r + i < r1;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const int c = (k * blockDim.x + threadIdx.x) * VEC;
        if (row_ok && ok[k]) load_row<VEC>(x[i][k], X + static_cast<int64_t>(r + i) * ldx + c);
        else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) x[i][k][v] = 0.f;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < R; ++i)        // fp64: near a one-hot softmax X_n . dOut - u cancels to far below fp32 rounding
#pragma unroll
      for (int k = 0; k < NV; ++k)
#pragma unroll
        for (int v = 0; v < VEC; ++v) d[i] = fma(static_cast<double>(x[i][k][v]), static_cast<double>(dov[k][v]), d[i]);
    block_sum<R>(d, red, fin, buf);
    buf ^= 1;
#pragma unroll
    for (int i = 0; i < R; ++i) {
      if (r + i >= r1) continue;
      const float p = expf(__ldg(scores + r + i) - M) * inv;
      const double ds = static_cast<double>(p) * (d[i] - u[0]);
      const float dsf = static_cast<float>(ds);
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        if (!ok[k]) continue;
        float o[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          o[v] = fmaf(dsf, av[k][v], p * dov[k][v]);
          da[k][v] = fma(ds, static_cast<double>(x[i][k][v]), da[k][v]);
        }
        store_row<VEC>(dX + static_cast<int64_t>(r + i) * lddx + (k * blockDim.x + threadIdx.x) * VEC, o);
      }
    }
  }
  const int64_t slot = static_cast<int64_t>(g) * S + sp;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    if (!ok[k]) continue;
    const int c = (k * blockDim.x + threadIdx.x) * VEC;
#pragma unroll
    for (int v = 0; v < VEC; ++v) part_da[slot * W + c + v] = da[k][v];
  }
}

// grid (column tile of 32): da[c] = sum over the n_parts partial rows, warp w taking rows w, w+8, ..., the 8 warp sums
// added in warp order (fp64 throughout, rounded once).
__global__ void __launch_bounds__(256) attn_pool_da_reduce_kernel(const double* __restrict__ part, int64_t n_parts, int W,
                                                                  float* __restrict__ da) {
  __shared__ double s[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  double t = 0.0;
  if (c < W)
    for (int64_t r = warp; r < n_parts; r += 8) t += part[r * W + c];
  s[warp][lane] = t;
  __syncthreads();
  if (warp == 0 && c < W) {
    double v = s[0][lane];
    for (int w = 1; w < 8; ++w) v += s[w][lane];
    da[c] = static_cast<float>(v);
  }
}

struct AttnShape {
  int vec, nv, threads;
};

// float4 columns where width, leading dimensions and pointers allow it; NV column slices per thread so that a block
// has at most 512 threads (W <= 8192 on the float4 path, <= 2048 on the scalar one).
static bool attn_shape(int W, bool vec_ok, AttnShape& sh) {
  sh.vec = vec_ok ? 4 : 1;
  const int n = static_cast<int>(ceil_div(W, sh.vec));
  for (int nv = 1; nv <= 4; nv *= 2) {
    const int t = static_cast<int>(round_up(ceil_div(n, nv), 32));
    if (t <= 512) {
      sh.nv = nv;
      sh.threads = t;
      return true;
    }
  }
  return false;
}

template <int VEC>
static void launch_fwd(const AttnShape& sh, dim3 grid, cudaStream_t st, const float* X, int64_t ldx, const float* a,
                       const int32_t* gp, int W, int S, float* out, int64_t ldo, float* scores, float* gstats,
                       float* part_acc, float* part_md) {
  switch (sh.nv) {
    case 1: attn_pool_fwd_kernel<VEC, 1><<<grid, sh.threads, 0, st>>>(X, ldx, a, gp, W, S, out, ldo, scores, gstats, part_acc, part_md); break;
    case 2: attn_pool_fwd_kernel<VEC, 2><<<grid, sh.threads, 0, st>>>(X, ldx, a, gp, W, S, out, ldo, scores, gstats, part_acc, part_md); break;
    default: attn_pool_fwd_kernel<VEC, 4><<<grid, sh.threads, 0, st>>>(X, ldx, a, gp, W, S, out, ldo, scores, gstats, part_acc, part_md); break;
  }
}

template <int VEC>
static void launch_bwd(const AttnShape& sh, dim3 grid, cudaStream_t st, const float* dout, int64_t lddo, const float* X,
                       int64_t ldx, const float* a, const int32_t* gp, int W, int S, const float* out, int64_t ldo,
                       const float* scores, const float* gstats, float* dX, int64_t lddx, double* part) {
  switch (sh.nv) {
    case 1: attn_pool_bwd_kernel<VEC, 1><<<grid, sh.threads, 0, st>>>(dout, lddo, X, ldx, a, gp, W, S, out, ldo, scores, gstats, dX, lddx, part); break;
    case 2: attn_pool_bwd_kernel<VEC, 2><<<grid, sh.threads, 0, st>>>(dout, lddo, X, ldx, a, gp, W, S, out, ldo, scores, gstats, dX, lddx, part); break;
    default: attn_pool_bwd_kernel<VEC, 4><<<grid, sh.threads, 0, st>>>(dout, lddo, X, ldx, a, gp, W, S, out, ldo, scores, gstats, dX, lddx, part); break;
  }
}

static int64_t attn_fwd_part_bytes(int64_t slots, int W) {
  return round_up(slots * W * 4, 256) + round_up(slots * 8, 256);
}

}  // namespace gcs

using namespace gcs;

extern "C" int64_t gcs_attn_pool_workspace_bytes(int64_t n_rows, int32_t n_graphs, int32_t W) {
  if (n_rows < 0 || n_graphs < 0 || W <= 0) return -1;
  const int S = attn_splits(n_rows, n_graphs);
  const int64_t slots = static_cast<int64_t>(n_graphs) * S;
  const int64_t fwd = S > 1 ? attn_fwd_part_bytes(slots, W) : 0;
  const int64_t bwd = round_up(slots * W * 8, 256);
  return fwd > bwd ? fwd : bwd;
}

extern "C" int gcs_attn_sum_pool_fwd(const float* X, int64_t ldx, int64_t n_rows, const float* kernel,
                                     const int32_t* graph_ptr, int32_t n_graphs, int32_t W, float* out, int64_t ldo,
                                     float* scores, float* gstats, void* workspace, int64_t workspace_bytes,
                                     gcs_stream stream) {
  GCS_CHECK_ARG(n_graphs >= 0 && W > 0 && n_rows >= 0 && n_rows < INT32_MAX, "gcs_attn_sum_pool_fwd: bad size");
  if (n_graphs == 0) return GCS_OK;
  GCS_CHECK_ARG(X && kernel && graph_ptr && out && ldx >= W && ldo >= W, "gcs_attn_sum_pool_fwd: bad pointer / leading dimension");
  const int64_t need = gcs_attn_pool_workspace_bytes(n_rows, n_graphs, W);
  GCS_CHECK_ARG(workspace_bytes >= need && (need == 0 || workspace),
                "gcs_attn_sum_pool_fwd: workspace %lld < %lld bytes", (long long)workspace_bytes, (long long)need);
  const bool vec = (W % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && aligned16(X) && aligned16(out);
  AttnShape sh;
  if (!attn_shape(W, vec, sh)) return fail(GCS_ERR_UNSUPPORTED, "gcs_attn_sum_pool_fwd: width %d is too large", W);
  const int S = attn_splits(n_rows, n_graphs);
  const int64_t slots = static_cast<int64_t>(n_graphs) * S;
  float* part_acc = S > 1 ? static_cast<float*>(workspace) : nullptr;
  float* part_md = S > 1 ? reinterpret_cast<float*>(static_cast<char*>(workspace) + round_up(slots * W * 4, 256)) : nullptr;
  cudaStream_t st = as_stream(stream);
  dim3 grid(n_graphs, S);
  if (sh.vec == 4) launch_fwd<4>(sh, grid, st, X, ldx, kernel, graph_ptr, W, S, out, ldo, scores, gstats, part_acc, part_md);
  else launch_fwd<1>(sh, grid, st, X, ldx, kernel, graph_ptr, W, S, out, ldo, scores, gstats, part_acc, part_md);
  GCS_CHECK_LAUNCH("attn_pool_fwd_kernel");
  if (S > 1) {
    attn_pool_combine_kernel<<<dim3(n_graphs, static_cast<unsigned>(ceil_div(W, 256))), 256, 0, st>>>(part_acc, part_md, S, W,
                                                                                                      out, ldo, gstats);
    GCS_CHECK_LAUNCH("attn_pool_combine_kernel");
  }
  return GCS_OK;
}

extern "C" int gcs_attn_sum_pool_bwd(const float* dout, int64_t lddo, const float* X, int64_t ldx, int64_t n_rows,
                                     const float* kernel, const int32_t* graph_ptr, int32_t n_graphs, int32_t W,
                                     const float* out, int64_t ldo, const float* scores, const float* gstats, float* dX,
                                     int64_t lddx, float* dkernel, void* workspace, int64_t workspace_bytes,
                                     gcs_stream stream) {
  GCS_CHECK_ARG(n_graphs >= 0 && W > 0 && n_rows >= 0 && n_rows < INT32_MAX, "gcs_attn_sum_pool_bwd: bad size");
  cudaStream_t st = as_stream(stream);
  if (n_graphs == 0) {
    if (dkernel) GCS_CUDA(cudaMemsetAsync(dkernel, 0, sizeof(float) * W, st));
    return GCS_OK;
  }
  GCS_CHECK_ARG(dout && X && kernel && graph_ptr && out && scores && gstats && dX && dkernel && ldx >= W && ldo >= W &&
                    lddo >= W && lddx >= W,
                "gcs_attn_sum_pool_bwd: bad pointer / leading dimension");
  const int64_t need = gcs_attn_pool_workspace_bytes(n_rows, n_graphs, W);
  GCS_CHECK_ARG(workspace && workspace_bytes >= need, "gcs_attn_sum_pool_bwd: workspace %lld < %lld bytes",
                (long long)workspace_bytes, (long long)need);
  const bool vec = (W % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && (lddo % 4 == 0) && (lddx % 4 == 0) && aligned16(X) &&
                   aligned16(out) && aligned16(dout) && aligned16(dX);
  AttnShape sh;
  if (!attn_shape(W, vec, sh)) return fail(GCS_ERR_UNSUPPORTED, "gcs_attn_sum_pool_bwd: width %d is too large", W);
  const int S = attn_splits(n_rows, n_graphs);
  double* part = static_cast<double*>(workspace);
  dim3 grid(n_graphs, S);
  if (sh.vec == 4) launch_bwd<4>(sh, grid, st, dout, lddo, X, ldx, kernel, graph_ptr, W, S, out, ldo, scores, gstats, dX, lddx, part);
  else launch_bwd<1>(sh, grid, st, dout, lddo, X, ldx, kernel, graph_ptr, W, S, out, ldo, scores, gstats, dX, lddx, part);
  GCS_CHECK_LAUNCH("attn_pool_bwd_kernel");
  attn_pool_da_reduce_kernel<<<static_cast<unsigned>(ceil_div(W, 32)), 256, 0, st>>>(part, static_cast<int64_t>(n_graphs) * S, W,
                                                                                     dkernel);
  GCS_CHECK_LAUNCH("attn_pool_da_reduce_kernel");
  return GCS_OK;
}
