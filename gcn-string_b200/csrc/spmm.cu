// K3 / K7 — sum aggregation  Y = pattern(A) . f(X),  f = fused BatchNorm + PReLU prologue.
//
// Replaces MessagePassing.propagate as GeneralConv.call invokes it (SURVEY.md §8 a4/a5):
//   messages = tf.gather(x, a.indices[:,1])          -> [nnz, H] materialised in TF
//   out      = tf.math.unsorted_segment_sum(messages, a.indices[:,0], N)
// Here the messages are never materialised, BN+PReLU are applied to X on the fly (they are
// a PROLOGUE of the aggregation in GeneralConv: transform -> BN -> PReLU -> aggregate), and
// Y is written straight into its slice of the 'cat' buffer (ldy = concat width).
// Determinism: each output element is owned by one thread which adds its neighbours in
// ascending column order — no atomics, no cross-lane reduction.
//
// Two kernels:
//  * spmm_rb4_kernel  — consumes the RB4 row-block format (built once per batch from the CSR by
//    gcs_spmm_build_rb4); H/4 lanes per block of 4 output rows, 128-bit gathers from global memory
//    (L1/L2 serve the re-reads), 4 union entries in flight per lane.
//  * spmm_rows_kernel — plain CSR, H/4 lanes per row; used when no RB4 structure is supplied or the
//    rows do not share neighbours, and (VEC = 1) for odd widths / unaligned views.
// A shared-memory-staged tile design (per-graph slabs, ghost rows) was built and measured first; it
// loses to both (profiles/r01_spmm_*.md): its four dependent staging phases leave the SM idle and
// its gather is bound by the same 128 B/clk L1/shared pipe.
#include "common.cuh"

namespace gcs {

// ---------------------------------------------------------------------------------------------
// RB4: row-block-of-4 format.  Residue contact maps are banded, so consecutive rows share most of
// their neighbours.  For each block of 4 rows the sorted UNION of its column indices is stored once,
// each entry with a mask of the rows that contain it: ent = (col << 8) | mask.  A neighbour row of X
// is then loaded (and BN+PReLU-transformed) once per block instead of once per row - 2.1x fewer
// gathers and transforms on E. coli-shaped graphs - while every output row still adds its own
// neighbours in ascending column order (bit-identical to the CSR kernels).
// Block height, measured on B200 at cfg2 (forward with prologue / plain gather of the backward):
//   8 rows: union 2.6x smaller, 32 predicated add slots per entry, 77 / 61 registers   356 / 277 us
//   4 rows: union 2.1x smaller, 16 slots per entry, 56 / 47 registers, 4 CTAs per SM    334 / 262 us
//   2 rows: union 1.5x smaller                                                          399 / 272 us
constexpr int kRB = 4;

// RB-way merge of the sorted neighbour lists of one row block; kFill = false counts the union size.
// Order of a block's entries: first the entries that ALL RB rows share (mask = all ones), in ascending column order and
// as many as fill whole groups of four - each of these words carries kRbFullFlag, and a kernel may add such a neighbour
// row once into an accumulator the block shares instead of RB times (in a band of half-width w, 2w - 2 of the 2w + 4
// union columns of a 4-row block are shared by all four rows) - then every other entry in ascending column order.
// Per output row the summation order is therefore: the row's other neighbours ascending, then the shared sum (slab
// kernel), or shared neighbours ascending, then the others (kernels that ignore the flag) - fixed either way.
constexpr uint32_t kRbFullFlag = 1u << 4;
template <int RB, bool kFill>
__global__ void __launch_bounds__(128) rb_build_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                                        int n_rows, int n_blocks, const int32_t* __restrict__ blk_ptr,
                                                        int32_t* __restrict__ count, uint32_t* __restrict__ ent) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_blocks) return;
  constexpr uint32_t kAll = (1u << RB) - 1u;
  // visit(col, mask) for every union entry in ascending column order
  auto merge = [&](auto&& visit) {
    int p[RB], e[RB], cur[RB];
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      const int row = b * RB + r;
      p[r] = row < n_rows ? __ldg(rowptr + row) : 0;
      e[r] = row < n_rows ? __ldg(rowptr + row + 1) : 0;
      cur[r] = p[r] < e[r] ? __ldg(colidx + p[r]) : INT32_MAX;
    }
    while (true) {
      int cmin = cur[0];
#pragma unroll
      for (int r = 1; r < RB; ++r) cmin = min(cmin, cur[r]);
      if (cmin == INT32_MAX) break;
      uint32_t mask = 0;
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        if (cur[r] == cmin) {
          mask |= 1u << r;
          ++p[r];
          cur[r] = p[r] < e[r] ? __ldg(colidx + p[r]) : INT32_MAX;
        }
      }
      visit(cmin, mask);
    }
  };
  int n = 0, n_full = 0, last = 0;
  merge([&](int col, uint32_t mask) { ++n; n_full += mask == kAll ? 1 : 0; last = col; });
  // pad to a multiple of 4 entries with no-ops (mask 0, a column of the block): every block then starts on a 16-byte
  // boundary and the kernels read four entry words per load
  const int padded = (n + 3) & ~3;
  if (!kFill) {
    count[b] = padded;
    return;
  }
  uint32_t* out = ent + __ldg(blk_ptr + b);
  const int lead = n_full & ~3;                      // shared entries that form whole groups of four
  int i_full = 0, i_rest = lead;
  merge([&](int col, uint32_t mask) {
    const uint32_t w = (static_cast<uint32_t>(col) << 8) | mask;
    if (mask == kAll && i_full < lead) out[i_full++] = w | kRbFullFlag;
    else out[i_rest++] = w;
  });
  for (; i_rest < padded; ++i_rest) out[i_rest] = static_cast<uint32_t>(last) << 8;
}

// One row block per `lanes` threads (lanes = H/4, each lane owns 4 columns); a CTA walks a contiguous
// range of row blocks so that neighbouring blocks reuse each other's X rows through L1.
template <bool kTransform>
__global__ void __launch_bounds__(256, 4) spmm_rb4_kernel(
    const int32_t* __restrict__ blk_ptr, const uint32_t* __restrict__ ent, int n_rows, int n_blocks,
    const float* __restrict__ X, int64_t ldx, const float* __restrict__ scale, const float* __restrict__ shift,
    const float* __restrict__ alpha, const float* __restrict__ R, int64_t ldr, float* __restrict__ Y, int64_t ldy,
    int lanes, int slots, int iters, float* __restrict__ amax) {
  const int lane = threadIdx.x % lanes;
  const int slot = threadIdx.x / lanes;
  if (slot >= slots) return;
  const int c = lane * 4;
  float4 sc, sh, al;
  if (kTransform) {
    sc = __ldg(reinterpret_cast<const float4*>(scale + c));
    sh = __ldg(reinterpret_cast<const float4*>(shift + c));
    al = __ldg(reinterpret_cast<const float4*>(alpha + c));
  }
  auto load = [&](uint32_t w) {
    float4 v = __ldg(reinterpret_cast<const float4*>(X + static_cast<int64_t>(w >> 8) * ldx + c));
    if (kTransform) {
      v.x = bn_prelu(v.x, sc.x, sh.x, al.x);
      v.y = bn_prelu(v.y, sc.y, sh.y, al.y);
      v.z = bn_prelu(v.z, sc.z, sh.z, al.z);
      v.w = bn_prelu(v.w, sc.w, sh.w, al.w);
    }
    return v;
  };
  const int b_begin = blockIdx.x * slots * iters;
  float mx = 0.f;
  for (int it = 0; it < iters; ++it) {
    const int b = b_begin + it * slots + slot;
    if (b >= n_blocks) break;
    const int e0 = __ldg(blk_ptr + b), e1 = __ldg(blk_ptr + b + 1);
    float4 acc[kRB];
    // Predicated adds: 4 * kRB issue slots per entry of which about a third do work.  Measured alternatives on B200
    // (8-row blocks): warp-uniform branches per row / per half block 427 us, packed add.f32x2 434 us, predicated 367 us.
    auto scatter = [&](const float4& v, uint32_t m) {
#pragma unroll
      for (int r = 0; r < kRB; ++r) {
        if (m & (1u << r)) { acc[r].x += v.x; acc[r].y += v.y; acc[r].z += v.z; acc[r].w += v.w; }
      }
    };
    int e = e0;
    {
      // leading groups of neighbours that all rows of the block have (kRbFullFlag): one shared sum, 4 adds per
      // neighbour instead of 16 predicated ones; the rows start from it (the order of the list, bit for bit)
      float4 sh = make_float4(0.f, 0.f, 0.f, 0.f);
      for (; e + 4 <= e1; e += 4) {
        const uint32_t w0 = __ldg(ent + e);
        if (!(w0 & kRbFullFlag)) break;
        const uint32_t w1 = __ldg(ent + e + 1), w2 = __ldg(ent + e + 2), w3 = __ldg(ent + e + 3);
        const float4 v0 = load(w0), v1 = load(w1), v2 = load(w2), v3 = load(w3);
        sh.x += v0.x; sh.y += v0.y; sh.z += v0.z; sh.w += v0.w;
        sh.x += v1.x; sh.y += v1.y; sh.z += v1.z; sh.w += v1.w;
        sh.x += v2.x; sh.y += v2.y; sh.z += v2.z; sh.w += v2.w;
        sh.x += v3.x; sh.y += v3.y; sh.z += v3.z; sh.w += v3.w;
      }
#pragma unroll
      for (int r = 0; r < kRB; ++r) acc[r] = sh;
    }
    for (; e + 4 <= e1; e += 4) {
      const uint32_t w0 = __ldg(ent + e), w1 = __ldg(ent + e + 1), w2 = __ldg(ent + e + 2), w3 = __ldg(ent + e + 3);
      const float4 v0 = load(w0), v1 = load(w1), v2 = load(w2), v3 = load(w3);
      scatter(v0, w0); scatter(v1, w1); scatter(v2, w2); scatter(v3, w3);
    }
    for (; e < e1; ++e) {
      const uint32_t w = __ldg(ent + e);
      scatter(load(w), w);
    }
#pragma unroll
    for (int r = 0; r < kRB; ++r) {
      const int row = b * kRB + r;
      if (row < n_rows) {
        if (R) {                                     // Add()([z, out]): the skip operand joins after the aggregation
          const float4 q = __ldg(reinterpret_cast<const float4*>(R + static_cast<int64_t>(row) * ldr + c));
          acc[r].x += q.x; acc[r].y += q.y; acc[r].z += q.z; acc[r].w += q.w;
        }
        *reinterpret_cast<float4*>(Y + static_cast<int64_t>(row) * ldy + c) = acc[r];
        if (amax) mx = amax4(mx, acc[r]);
      }
    }
  }
  amax_commit(mx, amax);
}

// Row-parallel CSR kernel.  VEC = 4: H % 4 == 0 and 16 B-aligned rows, lanes = H/4 threads per
// row.  VEC = 1: any H, lanes = H threads per row.  Rows wider than 256 lanes are split over
// gridDim.y into slices of 256 lanes (256 * VEC columns, a multiple of 4: float4 alignment holds);
// up to that width gridDim.y = 1.  A CTA walks a CONTIGUOUS chunk of rows:
// consecutive rows of a banded matrix share most of their neighbours, which then hit in L1.
// kGeneral adds what GeneralConv itself never asks for (SURVEY.md §8 f3): per-entry weights `values` (CSR order),
// aggregate = mean / max (scatter_mean = unsorted_segment_mean: sum / entry count, 0 for an empty row; scatter_max =
// unsorted_segment_max: the lowest float for an empty row) and a residual R added after the aggregation.
enum { kAggSum = 0, kAggMean = 1, kAggMax = 2 };
template <int VEC, bool kTransform, bool kGeneral>
__global__ void __launch_bounds__(256) spmm_rows_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, int64_t n_rows,
    const float* __restrict__ X, int64_t ldx, const float* __restrict__ scale,
    const float* __restrict__ shift, const float* __restrict__ alpha, float* __restrict__ Y,
    int64_t ldy, int H, int lanes, int rows_per_block, int iters, const float* __restrict__ values,
    const float* __restrict__ R, int64_t ldr, int agg, float* __restrict__ amax) {
  const int lane = threadIdx.x % lanes;
  const int slot = threadIdx.x / lanes;
  const int c = (static_cast<int>(blockIdx.y) * lanes + lane) * VEC;
  if (slot >= rows_per_block || c >= H) return;
  float sc[VEC], sh[VEC], al[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    sc[k] = kTransform ? __ldg(scale + c + k) : 1.f;
    sh[k] = kTransform ? __ldg(shift + c + k) : 0.f;
    al[k] = kTransform ? __ldg(alpha + c + k) : 1.f;
  }
  auto load = [&](int j, float* v) {
    const float* p = X + static_cast<int64_t>(j) * ldx + c;
    if (VEC == 4) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(p));
      v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
      v[0] = __ldg(p);
    }
    if (kTransform) {
#pragma unroll
      for (int k = 0; k < VEC; ++k) v[k] = bn_prelu(v[k], sc[k], sh[k], al[k]);
    }
  };
  float mx = 0.f;
  auto do_row = [&](int64_t r) {
    const int eb = __ldg(rowptr + r), ee = __ldg(rowptr + r + 1);
    float acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = (kGeneral && agg == kAggMax) ? -3.402823466e+38f : 0.f;
    int e = eb;
    if (kGeneral) {
      for (; e < ee; ++e) {
        float v[VEC];
        load(__ldg(colidx + e), v);
        const float w = values ? __ldg(values + e) : 1.f;
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
          const float m = values ? v[k] * w : v[k];
          acc[k] = agg == kAggMax ? fmaxf(acc[k], m) : acc[k] + m;
        }
      }
      if (agg == kAggMean && ee > eb) {
        const float cnt = static_cast<float>(ee - eb);
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[k] = acc[k] / cnt;
      }
      if (R) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[k] += __ldg(R + r * ldr + c + k);
      }
    }
    for (; e + 4 <= ee; e += 4) {
      const int j0 = __ldg(colidx + e), j1 = __ldg(colidx + e + 1);
      const int j2 = __ldg(colidx + e + 2), j3 = __ldg(colidx + e + 3);
      float v0[VEC], v1[VEC], v2[VEC], v3[VEC];
      load(j0, v0); load(j1, v1); load(j2, v2); load(j3, v3);
#pragma unroll
      for (int k = 0; k < VEC; ++k) { acc[k] += v0[k]; acc[k] += v1[k]; acc[k] += v2[k]; acc[k] += v3[k]; }
    }
    for (; e < ee; ++e) {
      float v[VEC];
      load(__ldg(colidx + e), v);
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[k] += v[k];
    }
    float* q = Y + r * ldy + c;
    if (VEC == 4) *reinterpret_cast<float4*>(q) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    else q[0] = acc[0];
#pragma unroll
    for (int k = 0; k < VEC; ++k) mx = fmaxf(mx, fabsf(acc[k]));
  };
  const int64_t chunk = static_cast<int64_t>(rows_per_block) * iters;
  const int64_t rbeg = static_cast<int64_t>(blockIdx.x) * chunk;
  const int64_t rend = rbeg + chunk < n_rows ? rbeg + chunk : n_rows;
  for (int64_t r = rbeg + slot; r < rend; r += rows_per_block) do_row(r);
  amax_commit(mx, amax);
}

// ---------------------------------------------------------------------------------------------
// Backward of the general aggregation (SURVEY.md §8 f3): given dZ = dLoss/dZ for Z = agg_j(w_ij * a[j]), a = f(h),
// dA[j] = dLoss/da[j], gathered over the TRANSPOSED pattern (row j of A^T lists the rows i that have j as a neighbour;
// values_t are the weights in that order):
//   sum : dA[j] = sum_i w_ij * dZ[i]
//   mean: dA[j] = sum_i w_ij * dZ[i] / deg_i            deg_i = entries of row i (scatter_mean divides by the count)
//   max : dA[j, c] = sum_i [w_ij * a[j, c] == Z[i, c]] * w_ij * dZ[i, c] / ties[i, c]
//         (tf.math.unsorted_segment_max's gradient: the maxima of a segment share its gradient equally; ties[i, c] is
//         the number of neighbours of i that attain the maximum, counted by spmm_max_ties_kernel)
// One owner thread per output element, entries in ascending column order: deterministic.  Lanes own VEC adjacent
// columns; rows wider than 256 lanes are split over gridDim.y as in spmm_rows_kernel.
template <int VEC>
__global__ void __launch_bounds__(256) spmm_agg_bwd_kernel(
    const int32_t* __restrict__ rowptr_t, const int32_t* __restrict__ colidx_t, const float* __restrict__ values_t,
    int64_t n_rows, const float* __restrict__ dZ, int64_t lddz, int agg, const int32_t* __restrict__ fwd_rowptr,
    const float* __restrict__ Z, int64_t ldz, const float* __restrict__ ties, int64_t ldt, const float* __restrict__ Hpre,
    int64_t ldh, const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ alpha,
    float* __restrict__ dA, int64_t ldda, int H, int lanes, int rows_per_block) {
  const int lane = threadIdx.x % lanes, slot = threadIdx.x / lanes;
  const int c = (static_cast<int>(blockIdx.y) * lanes + lane) * VEC;
  const int64_t j = static_cast<int64_t>(blockIdx.x) * rows_per_block + slot;
  if (slot >= rows_per_block || j >= n_rows || c >= H) return;
  float own[VEC], acc[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    acc[k] = 0.f;
    own[k] = 0.f;
    if (agg == kAggMax && c + k < H) {
      const float x = __ldg(Hpre + j * ldh + c + k);
      own[k] = scale ? bn_prelu(x, __ldg(scale + c + k), __ldg(shift + c + k), __ldg(alpha + c + k)) : x;
    }
  }
  const int eb = __ldg(rowptr_t + j), ee = __ldg(rowptr_t + j + 1);
  for (int e = eb; e < ee; ++e) {
    const int64_t i = __ldg(colidx_t + e);
    float w = values_t ? __ldg(values_t + e) : 1.f;
    const float wv = w;
    if (agg == kAggMean) w = w / static_cast<float>(__ldg(fwd_rowptr + i + 1) - __ldg(fwd_rowptr + i));
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      if (c + k >= H) continue;
      const float g = __ldg(dZ + i * lddz + c + k);
      if (agg == kAggMax) {
        const float m = values_t ? own[k] * wv : own[k];
        if (m == __ldg(Z + i * ldz + c + k)) acc[k] += (values_t ? g * wv : g) / __ldg(ties + i * ldt + c + k);
      } else {
        acc[k] += values_t || agg == kAggMean ? g * w : g;
      }
    }
  }
#pragma unroll
  for (int k = 0; k < VEC; ++k)
    if (c + k < H) dA[j * ldda + c + k] = acc[k];
}

// ties[i, c] = number of entries (i, j) with w_ij * f(h[j, c]) == Z[i, c]  (forward pattern; >= 1 for a non-empty row)
__global__ void __launch_bounds__(256) spmm_max_ties_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, const float* __restrict__ values, int64_t n_rows,
    const float* __restrict__ Hpre, int64_t ldh, const float* __restrict__ scale, const float* __restrict__ shift,
    const float* __restrict__ alpha, const float* __restrict__ Z, int64_t ldz, float* __restrict__ ties, int64_t ldt, int H,
    int rows_per_block) {
  const int lanes = H < 256 ? H : 256;
  const int lane = threadIdx.x % lanes, slot = threadIdx.x / lanes;
  const int64_t i = static_cast<int64_t>(blockIdx.x) * rows_per_block + slot;
  if (slot >= rows_per_block || i >= n_rows) return;
  const int eb = __ldg(rowptr + i), ee = __ldg(rowptr + i + 1);
  for (int c = lane; c < H; c += lanes) {
    const float z = __ldg(Z + i * ldz + c);
    const float sc = scale ? __ldg(scale + c) : 1.f, sh = scale ? __ldg(shift + c) : 0.f, al = scale ? __ldg(alpha + c) : 1.f;
    int n = 0;
    for (int e = eb; e < ee; ++e) {
      const int64_t j = __ldg(colidx + e);
      const float x = __ldg(Hpre + j * ldh + c);
      const float a = scale ? bn_prelu(x, sc, sh, al) : x;
      n += (values ? a * __ldg(values + e) : a) == z;
    }
    ties[i * ldt + c] = static_cast<float>(n > 0 ? n : 1);
  }
}


}  // namespace gcs

using namespace gcs;

namespace {

struct SpmmArgs {
  const int32_t* rowptr; const int32_t* colidx; const int32_t* blk_ptr; const uint32_t* ent; int64_t n_rows;
  const float* X; int64_t ldx; const float* scale; const float* shift; const float* alpha;
  float* Y; int64_t ldy; int H; cudaStream_t st;
  const float* values = nullptr; const float* R = nullptr; int64_t ldr = 0; int agg = 0;
  bool general() const { return values || agg != kAggSum; }
};

int g_rows_iters = 16;   // tuning knob (gcs_debug_set_param 1)
int g_rb4_iters = 2;     // row blocks per slot per CTA (gcs_debug_set_param 2); sweep on 8-row blocks 1/2/3/4: 372/356/358/367 us fwd, 283/277/287/297 us bwd; on 4-row blocks 2/4/8: 338/334/349, 262/264/293

// Lanes per row and column slices (gridDim.y) of the row kernels for H columns, VEC columns per lane.
struct RowSplit { int lanes; unsigned slices; };
template <int VEC>
RowSplit row_split(int H) {
  const int64_t need = (static_cast<int64_t>(H) + VEC - 1) / VEC;
  return {static_cast<int>(need < 256 ? need : 256), static_cast<unsigned>(ceil_div(need, static_cast<int64_t>(256)))};
}

template <int VEC>
int launch_rows(const SpmmArgs& a) {
  const RowSplit s = row_split<VEC>(a.H);
  const int lanes = s.lanes;
  const int rows_per_block = 256 / lanes;
  const int iters = g_rows_iters;                   // rows_per_block * iters contiguous rows per CTA
  dim3 grid(static_cast<unsigned>(ceil_div(a.n_rows, static_cast<int64_t>(rows_per_block) * iters)), s.slices);
#define GCS_ROWS_LAUNCH(T, G)                                                                                          \
  spmm_rows_kernel<VEC, T, G><<<grid, 256, 0, a.st>>>(a.rowptr, a.colidx, a.n_rows, a.X, a.ldx, a.scale, a.shift,      \
                                                      a.alpha, a.Y, a.ldy, a.H, lanes, rows_per_block, iters, a.values, \
                                                      a.R, a.ldr, a.agg, amax_sink().produce)
  const bool general = a.general() || a.R;
  if (a.scale) { if (general) GCS_ROWS_LAUNCH(true, true); else GCS_ROWS_LAUNCH(true, false); }
  else { if (general) GCS_ROWS_LAUNCH(false, true); else GCS_ROWS_LAUNCH(false, false); }
#undef GCS_ROWS_LAUNCH
  GCS_CHECK_LAUNCH("spmm_rows_kernel");
  return GCS_OK;
}

int launch_rb4(const SpmmArgs& a) {
  const int lanes = a.H / 4;
  const int slots = 256 / lanes;
  const int n_blocks = static_cast<int>(ceil_div(a.n_rows, kRB));
  const int iters = g_rb4_iters;
  dim3 grid(static_cast<unsigned>(ceil_div(n_blocks, static_cast<int64_t>(slots) * iters)));
  if (a.scale)
    spmm_rb4_kernel<true><<<grid, 256, 0, a.st>>>(a.blk_ptr, a.ent, static_cast<int>(a.n_rows), n_blocks, a.X, a.ldx, a.scale, a.shift, a.alpha, a.R, a.ldr, a.Y, a.ldy, lanes, slots, iters, amax_sink().produce);
  else
    spmm_rb4_kernel<false><<<grid, 256, 0, a.st>>>(a.blk_ptr, a.ent, static_cast<int>(a.n_rows), n_blocks, a.X, a.ldx, a.scale, a.shift, a.alpha, a.R, a.ldr, a.Y, a.ldy, lanes, slots, iters, amax_sink().produce);
  GCS_CHECK_LAUNCH("spmm_rb4_kernel");
  return GCS_OK;
}

int g_spmm_mode = 0;   // 0 = auto, 1 = CSR row kernel, 2 = RB4 global-memory kernel whenever supplied (both: never the slab kernel)
}  // namespace

// Test / sweep hook (not part of the drop-in surface).
extern "C" void gcs_debug_set_spmm_mode(int mode) { g_spmm_mode = mode; }
namespace gcs { int spmm_mode() { return g_spmm_mode; } }
namespace gcs { void slab_set_param(int id, int value); void set_thin_wgrad(int v); }
namespace gcs { namespace tc { void set_wgrad_chain(int c); void set_max_chain_k(int k); void set_wgrad_pair(int v); void set_f16_mode(int v); void set_max_chain_k_f16(int k); void set_wgrad_f16(int v); } }
extern "C" void gcs_debug_set_param(int id, int value) {
  if (id == 1 && value > 0) g_rows_iters = value;
  if (id == 2 && value > 0) g_rb4_iters = value;
  if (id == 3) gcs::tc::set_wgrad_chain(value);
  if (id == 5) gcs::tc::set_max_chain_k(value);
  if (id == 4) gcs::tc::set_wgrad_pair(value);
  if (id == 7) gcs::tc::set_f16_mode(value);             // 0 tf32 only, 1 fp16 inside the fused model, 2 fp16 everywhere
  if (id == 8) gcs::tc::set_max_chain_k_f16(value);
  if (id == 9) gcs::tc::set_wgrad_f16(value);                // 0 = weight gradient on the tf32 split only
  if (id == 13) gcs::set_thin_wgrad(value);
  if (id == 10 || id == 11 || id == 12) gcs::slab_set_param(id, value);   // spmm_slab.cu: stages / stage bytes / grid
}

extern "C" int64_t gcs_spmm_rb_workspace_bytes(int64_t n_rows, int32_t rb_height) {
  if (rb_height != 2 && rb_height != 4) return -1;
  return round_up((ceil_div(n_rows > 0 ? n_rows : 1, rb_height) + 1) * static_cast<int64_t>(sizeof(int32_t)), 256);
}
extern "C" int64_t gcs_spmm_rb4_workspace_bytes(int64_t n_rows) { return gcs_spmm_rb_workspace_bytes(n_rows, 4); }

extern "C" int gcs_spmm_build_rb(const int32_t* rowptr, const int32_t* colidx, int64_t n_rows, int64_t nnz, int32_t rb_height,
                                 int32_t* blk_ptr, uint32_t* ent, void* workspace, int64_t workspace_bytes,
                                 gcs_stream stream) {
  GCS_CHECK_ARG(rb_height == 2 || rb_height == 4, "gcs_spmm_build_rb: block height must be 2 or 4");
  GCS_CHECK_ARG(rowptr && blk_ptr && workspace && n_rows >= 0 && nnz >= 0, "gcs_spmm_build_rb: bad argument");
  GCS_CHECK_ARG(nnz == 0 || (colidx && ent), "gcs_spmm_build_rb: null column / entry array");
  GCS_CHECK_ARG(n_rows < (1 << 24), "gcs_spmm_build_rb: the format packs the column index in 24 bits (n_rows < 16 777 216)");
  if (workspace_bytes < gcs_spmm_rb_workspace_bytes(n_rows, rb_height))
    return fail(GCS_ERR_WORKSPACE, "gcs_spmm_build_rb: workspace too small");
  cudaStream_t st = as_stream(stream);
  const int nb = static_cast<int>(ceil_div(n_rows, rb_height));
  int32_t* cnt = static_cast<int32_t*>(workspace);
  if (nb == 0) {
    GCS_CUDA(cudaMemsetAsync(blk_ptr, 0, sizeof(int32_t), st));
    return GCS_OK;
  }
  const unsigned grid = static_cast<unsigned>(ceil_div(nb, 128));
  const int n = static_cast<int>(n_rows);
  if (rb_height == 2) rb_build_kernel<2, false><<<grid, 128, 0, st>>>(rowptr, colidx, n, nb, nullptr, cnt, nullptr);
  else rb_build_kernel<4, false><<<grid, 128, 0, st>>>(rowptr, colidx, n, nb, nullptr, cnt, nullptr);
  GCS_CHECK_LAUNCH("rb_build_kernel<count>");
  GCS_TRY(exclusive_scan_i32(cnt, nb, blk_ptr, st));
  if (rb_height == 2) rb_build_kernel<2, true><<<grid, 128, 0, st>>>(rowptr, colidx, n, nb, blk_ptr, nullptr, ent);
  else rb_build_kernel<4, true><<<grid, 128, 0, st>>>(rowptr, colidx, n, nb, blk_ptr, nullptr, ent);
  GCS_CHECK_LAUNCH("rb_build_kernel<fill>");
  return GCS_OK;
}

extern "C" int gcs_spmm_build_rb4(const int32_t* rowptr, const int32_t* colidx, int64_t n_rows, int64_t nnz,
                                  int32_t* blk_ptr, uint32_t* ent, void* workspace, int64_t workspace_bytes,
                                  gcs_stream stream) {
  return gcs_spmm_build_rb(rowptr, colidx, n_rows, nnz, 4, blk_ptr, ent, workspace, workspace_bytes, stream);
}

extern "C" int gcs_spmm_aggregate(const int32_t* rowptr, const int32_t* colidx, const float* values,
                                  const int32_t* rb4_blk_ptr, const uint32_t* rb4_ent, int64_t n_rows, const float* X,
                                  int64_t ldx, const float* scale, const float* shift, const float* alpha,
                                  const float* residual, int64_t ldr, float* Y, int64_t ldy, int32_t H,
                                  int32_t aggregate, gcs_stream stream) {
  GCS_CHECK_ARG(n_rows >= 0 && H > 0, "gcs_spmm_aggregate: bad size (n_rows=%lld, H=%d)", (long long)n_rows, H);
  GCS_CHECK_ARG(aggregate == kAggSum || aggregate == kAggMean || aggregate == kAggMax,
                "gcs_spmm_aggregate: aggregate must be 0 (sum), 1 (mean) or 2 (max)");
  if (n_rows == 0) return GCS_OK;
  GCS_CHECK_ARG(rowptr && colidx && X && Y, "gcs_spmm_aggregate: null pointer");
  GCS_CHECK_ARG(ldx >= H && ldy >= H, "gcs_spmm_aggregate: leading dimension smaller than H");
  GCS_CHECK_ARG(!residual || ldr >= H, "gcs_spmm_aggregate: residual leading dimension smaller than H");
  GCS_CHECK_ARG((scale != nullptr) == (shift != nullptr) && (scale != nullptr) == (alpha != nullptr),
                "gcs_spmm_aggregate: scale/shift/alpha must be all NULL or all set");
  GCS_CHECK_ARG((rb4_blk_ptr != nullptr) == (rb4_ent != nullptr), "gcs_spmm_aggregate: rb4_blk_ptr and rb4_ent go together");
  GCS_CHECK_ARG(X != Y, "gcs_spmm_aggregate: in-place aggregation is not defined");
  GCS_CHECK_ARG(n_rows < INT32_MAX, "gcs_spmm_aggregate: n_rows exceeds int32 CSR range");
  SpmmArgs a{rowptr, colidx, rb4_blk_ptr, rb4_ent, n_rows, X, ldx, scale, shift, alpha, Y, ldy, H, as_stream(stream)};
  a.values = values; a.R = residual; a.ldr = ldr; a.agg = aggregate;
  const bool vec_ok = (H % 4 == 0) && (ldx % 4 == 0) && (ldy % 4 == 0) && aligned16(X) && aligned16(Y) &&
                      (!scale || (aligned16(scale) && aligned16(shift) && aligned16(alpha)));
  const bool res_ok = !residual || ((ldr % 4 == 0) && aligned16(residual));
  // RB4 whenever the structure is supplied: with the BN+PReLU prologue one transform per block instead of per row
  // (334 vs 463 us at cfg2), and for the plain gather of the backward 262 vs 319 us row by row.  The union entries
  // carry no per-row weight, so weighted / mean / max aggregation runs row by row.
  const bool want_rb4 = g_spmm_mode != 1 && !a.general();
  if (want_rb4 && rb4_blk_ptr && vec_ok && res_ok && H / 4 <= 256 && 256 % (H / 4) == 0) return launch_rb4(a);
  if (vec_ok) return launch_rows<4>(a);
  return launch_rows<1>(a);
}

extern "C" int gcs_spmm_sum(const int32_t* rowptr, const int32_t* colidx, const int32_t* rb4_blk_ptr,
                            const uint32_t* rb4_ent, int64_t n_rows, const float* X, int64_t ldx,
                            const float* scale, const float* shift, const float* alpha, float* Y,
                            int64_t ldy, int32_t H, gcs_stream stream) {
  return gcs_spmm_aggregate(rowptr, colidx, nullptr, rb4_blk_ptr, rb4_ent, n_rows, X, ldx, scale, shift, alpha, nullptr, 0,
                            Y, ldy, H, kAggSum, stream);
}

// Backward of gcs_spmm_aggregate with respect to f(X) (see spmm_agg_bwd_kernel).  (rowptr_t, colidx_t, values_t): the
// TRANSPOSED pattern with its weights in that order; fwd_rowptr: the forward row pointers (mean: entry counts);
// max additionally needs the forward inputs again: (rowptr, colidx, values) forward pattern, X (pre-prologue, with
// scale / shift / alpha as in the forward) and the forward output Z; `ties` [n_rows, H] is scratch.
extern "C" int gcs_spmm_aggregate_bwd(const int32_t* rowptr_t, const int32_t* colidx_t, const float* values_t,
                                      const int32_t* rowptr, const int32_t* colidx, const float* values, int64_t n_rows,
                                      const float* dZ, int64_t lddz, int32_t aggregate, const float* X, int64_t ldx,
                                      const float* scale, const float* shift, const float* alpha, const float* Z, int64_t ldz,
                                      float* ties, int64_t ldt, float* dA, int64_t ldda, int32_t H, gcs_stream stream) {
  GCS_CHECK_ARG(n_rows >= 0 && H > 0, "gcs_spmm_aggregate_bwd: bad size");
  GCS_CHECK_ARG(aggregate == kAggSum || aggregate == kAggMean || aggregate == kAggMax, "gcs_spmm_aggregate_bwd: aggregate must be 0, 1 or 2");
  if (n_rows == 0) return GCS_OK;
  GCS_CHECK_ARG(rowptr_t && colidx_t && dZ && dA && lddz >= H && ldda >= H, "gcs_spmm_aggregate_bwd: bad pointer / leading dimension");
  GCS_CHECK_ARG(aggregate != kAggMean || rowptr, "gcs_spmm_aggregate_bwd: mean needs the forward row pointers");
  GCS_CHECK_ARG(aggregate != kAggMax || (rowptr && colidx && X && Z && ties && ldx >= H && ldz >= H && ldt >= H),
                "gcs_spmm_aggregate_bwd: max needs the forward pattern, X, Z and the ties scratch");
  GCS_CHECK_ARG((scale != nullptr) == (shift != nullptr) && (scale != nullptr) == (alpha != nullptr),
                "gcs_spmm_aggregate_bwd: scale/shift/alpha must be all NULL or all set");
  GCS_CHECK_ARG(n_rows < INT32_MAX, "gcs_spmm_aggregate_bwd: n_rows exceeds int32 CSR range");
  cudaStream_t st = as_stream(stream);
  if (aggregate == kAggMax) {
    const int lanes = H < 256 ? H : 256;
    const int rpb = 256 / lanes;
    spmm_max_ties_kernel<<<static_cast<unsigned>(ceil_div(n_rows, rpb)), 256, 0, st>>>(rowptr, colidx, values, n_rows, X, ldx, scale,
                                                                                      shift, alpha, Z, ldz, ties, ldt, H, rpb);
    GCS_CHECK_LAUNCH("spmm_max_ties_kernel");
  }
  if (H <= 256) {
    const int rpb = 256 / H;
    spmm_agg_bwd_kernel<1><<<static_cast<unsigned>(ceil_div(n_rows, rpb)), 256, 0, st>>>(
        rowptr_t, colidx_t, values_t, n_rows, dZ, lddz, aggregate, rowptr, Z, ldz, ties, ldt, X, ldx, scale, shift, alpha, dA, ldda, H, H, rpb);
  } else {
    const RowSplit s = row_split<4>(H);
    const int rpb = 256 / s.lanes;
    spmm_agg_bwd_kernel<4><<<dim3(static_cast<unsigned>(ceil_div(n_rows, rpb)), s.slices), 256, 0, st>>>(
        rowptr_t, colidx_t, values_t, n_rows, dZ, lddz, aggregate, rowptr, Z, ldz, ties, ldt, X, ldx, scale, shift, alpha, dA, ldda, H, s.lanes, rpb);
  }
  GCS_CHECK_LAUNCH("spmm_agg_bwd_kernel");
  return GCS_OK;
}

