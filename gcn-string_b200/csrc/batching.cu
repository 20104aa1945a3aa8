// K0 — disjoint batching and CSR / segment-offset construction on the device.
//
// Replaces the host collate Spektral's DisjointLoader runs every step for the reference
// (src/scripts/gcn.py:316-317,350,367): np.vstack(x) + sp.block_diag(a) + sp.find +
// tf.sparse.reorder + np.repeat(arange(B), n_nodes)  (SURVEY.md §8 a1).  All outputs are
// integers (or copied floats) and must be bit-exact against oracle/batching_ref.py.
//
// HBM-bound integer/byte work: coalesced copies, one CTA per (graph, chunk).
#include "common.cuh"

namespace gcs {

// ---- scan of the selected graphs' sizes -> graph_ptr / edge_ptr (single CTA) ---------
// B is at most a few thousand; a single 1024-thread CTA does a chunked inclusive scan.
__global__ void __launch_bounds__(1024) batch_offsets_kernel(
    const int64_t* __restrict__ node_off, const int64_t* __restrict__ ds_rowptr,
    const int64_t* __restrict__ graph_ids, int n_graphs, int64_t n_nodes, int64_t nnz,
    int32_t* __restrict__ graph_ptr, int32_t* __restrict__ edge_ptr, int32_t* __restrict__ status) {
  __shared__ int64_t s_n[1024];
  __shared__ int64_t s_e[1024];
  __shared__ int64_t carry_n, carry_e;
  const int t = threadIdx.x;
  if (t == 0) {
    carry_n = 0;
    carry_e = 0;
    graph_ptr[0] = 0;
    edge_ptr[0] = 0;
  }
  __syncthreads();
  for (int base = 0; base < n_graphs; base += 1024) {
    const int j = base + t;
    int64_t n = 0, e = 0;
    if (j < n_graphs) {
      const int64_t g = graph_ids[j];
      const int64_t n0 = node_off[g], n1 = node_off[g + 1];
      n = n1 - n0;
      e = ds_rowptr[n1] - ds_rowptr[n0];
    }
    s_n[t] = n;
    s_e[t] = e;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {  // Hillis-Steele inclusive scan
      int64_t vn = 0, ve = 0;
      if (t >= off) {
        vn = s_n[t - off];
        ve = s_e[t - off];
      }
      __syncthreads();
      s_n[t] += vn;
      s_e[t] += ve;
      __syncthreads();
    }
    if (j < n_graphs) {
      graph_ptr[j + 1] = static_cast<int32_t>(carry_n + s_n[t]);
      edge_ptr[j + 1] = static_cast<int32_t>(carry_e + s_e[t]);
    }
    __syncthreads();
    if (t == 1023) {
      carry_n += s_n[t];
      carry_e += s_e[t];
    }
    __syncthreads();
  }
  if (t == 0 && (carry_n != n_nodes || carry_e != nnz)) atomicExch(status, 1);
}

// ---- fill: one CTA per (graph, chunk) -------------------------------------------------
__global__ void __launch_bounds__(256) batch_fill_kernel(
    const int64_t* __restrict__ node_off, const int64_t* __restrict__ ds_rowptr,
    const int32_t* __restrict__ ds_col, const float* __restrict__ ds_x,
    const float* __restrict__ ds_y, int n_feat, int n_classes,
    const int64_t* __restrict__ graph_ids, const int32_t* __restrict__ graph_ptr,
    const int32_t* __restrict__ edge_ptr, int32_t* __restrict__ rowptr,
    int32_t* __restrict__ colidx, float* __restrict__ x, int64_t* __restrict__ seg_ids,
    float* __restrict__ y, int64_t* __restrict__ coo) {
  const int j = blockIdx.x;
  const int chunk = blockIdx.y, n_chunks = gridDim.y;
  const int tid = chunk * blockDim.x + threadIdx.x;
  const int stride = n_chunks * blockDim.x;
  const int64_t g = graph_ids[j];
  const int64_t n0 = node_off[g];
  const int n = static_cast<int>(node_off[g + 1] - n0);
  const int64_t e0 = ds_rowptr[n0];
  const int ne = static_cast<int>(ds_rowptr[n0 + n] - e0);
  const int r0 = graph_ptr[j];   // first batch row of this graph
  const int eb = edge_ptr[j];    // first batch edge of this graph

  // rowptr + seg ids (+ COO row ids need the row of every edge: done per row below)
  for (int l = tid; l < n; l += stride) {
    const int rs = static_cast<int>(ds_rowptr[n0 + l] - e0);
    rowptr[r0 + l] = eb + rs;
    seg_ids[r0 + l] = j;
    if (coo) {
      const int re = static_cast<int>(ds_rowptr[n0 + l + 1] - e0);
      for (int e = rs; e < re; ++e) coo[2 * static_cast<int64_t>(eb + e)] = r0 + l;
    }
  }
  // column indices: local -> batch-global
  for (int e = tid; e < ne; e += stride) {
    const int c = ds_col[e0 + e] + r0;
    colidx[eb + e] = c;
    if (coo) coo[2 * static_cast<int64_t>(eb + e) + 1] = c;
  }
  // node features (np.vstack): contiguous block copy, float4 when aligned
  const int64_t nx = static_cast<int64_t>(n) * n_feat;
  const float* src = ds_x + n0 * n_feat;
  float* dst = x + static_cast<int64_t>(r0) * n_feat;
  if ((n_feat & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int64_t k = tid; k < nx / 4; k += stride) d4[k] = __ldg(s4 + k);
  } else {
    for (int64_t k = tid; k < nx; k += stride) dst[k] = __ldg(src + k);
  }
  if (y && chunk == 0)
    for (int c = threadIdx.x; c < n_classes; c += blockDim.x)
      y[static_cast<int64_t>(j) * n_classes + c] = ds_y[g * n_classes + c];
  if (j == gridDim.x - 1 && tid == 0) rowptr[r0 + n] = eb + ne;  // rowptr[N] = nnz
}

// rowptr[0] when the batch is empty of graphs is handled by the host wrapper (memset).

// ---- sorted COO (int64 [nnz,2]) -> CSR -------------------------------------------------
__global__ void coo_rowptr_kernel(const int64_t* __restrict__ coo, int64_t nnz, int64_t n_rows,
                                  int32_t* __restrict__ rowptr) {
  // rowptr[r] = first e with row[e] >= r (lower bound over the sorted row column)
  const int64_t r = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (r > n_rows) return;
  int64_t lo = 0, hi = nnz;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (coo[2 * mid] < r) lo = mid + 1; else hi = mid;
  }
  rowptr[r] = static_cast<int32_t>(lo);
}

__global__ void coo_cols_kernel(const int64_t* __restrict__ coo, int64_t nnz, int64_t n_rows,
                                int32_t* __restrict__ colidx, int32_t* __restrict__ status) {
  const int64_t e = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (e >= nnz) return;
  const int64_t r = coo[2 * e], c = coo[2 * e + 1];
  bool bad = r < 0 || r >= n_rows || c < 0 || c >= n_rows;
  if (e > 0) {
    const int64_t pr = coo[2 * e - 2], pc = coo[2 * e - 1];
    bad = bad || pr > r || (pr == r && pc >= c);   // must be strictly row-major ascending
  }
  if (bad) atomicExch(status, 1);
  colidx[e] = static_cast<int32_t>(c);
}

__global__ void segment_ptr_kernel(const int64_t* __restrict__ seg, int64_t n, int n_graphs,
                                   int32_t* __restrict__ graph_ptr, int32_t* __restrict__ status) {
  const int64_t g = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (g <= n_graphs) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (seg[mid] < g) lo = mid + 1; else hi = mid;
    }
    graph_ptr[g] = static_cast<int32_t>(lo);
  }
  // sortedness / range check, grid-stride
  for (int64_t k = g; k < n; k += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t s = seg[k];
    if (s < 0 || s >= n_graphs || (k > 0 && seg[k - 1] > s)) atomicExch(status, 1);
  }
}

// ---- symmetry check: every (r,c) must have (c,r) ---------------------------------------
__global__ void csr_symmetric_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                     int64_t n_rows, int32_t* __restrict__ flag) {
  const int64_t r = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (r >= n_rows) return;
  for (int e = rowptr[r]; e < rowptr[r + 1]; ++e) {
    const int c = colidx[e];
    int lo = rowptr[c], hi = rowptr[c + 1];
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (colidx[mid] < r) lo = mid + 1; else hi = mid;
    }
    if (lo >= rowptr[c + 1] || colidx[lo] != r) {
      *flag = 0;   // benign race: every writer stores 0
      return;
    }
  }
}

__global__ void set_i32_kernel(int32_t* p, int32_t v) { *p = v; }

// ---- transpose (deterministic): count -> scan -> rank-fill ------------------------------
__global__ void tr_count_kernel(const int32_t* __restrict__ colidx, int64_t nnz, int32_t* __restrict__ cnt) {
  const int64_t e = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (e < nnz) atomicAdd(cnt + colidx[e], 1);   // integer atomics: order-independent result
}

// Exclusive scan of cnt[0..n) into out[0..n], chunked single-CTA (n up to a few million int32:
// bandwidth-trivial next to the SpMM it serves).  Per chunk of 16 K elements: 16 per thread, a
// shuffle scan inside each warp, one shuffle scan of the 32 warp totals - two barriers per chunk
// (a shared-memory Hillis-Steele scan with 20 barriers per 8 K chunk took 107 us for the 127 K row
// blocks of a cfg2 batch).
template <typename OutT>
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(const int32_t* __restrict__ cnt, int64_t n,
                                                              OutT* __restrict__ out) {
  __shared__ int32_t warp_tot[32];
  __shared__ int32_t carry_s;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  constexpr int PER = 16;
  OutT carry = 0;                                        // a chunk total fits int32, the running total may not
  for (int64_t base = 0; base < n; base += 1024 * PER) {
    int32_t v[PER];
    int32_t sum = 0;
    const int64_t b = base + static_cast<int64_t>(t) * PER;
    // 128-bit loads / stores where the thread's 16 elements are all there: with scalar accesses every warp instruction
    // touched 32 different sectors (16 K sector requests per chunk through one SM: ~8 us per chunk, 108 us for the 127 K
    // row blocks of a cfg2 batch under ncu)
    const bool vec_in = b + PER <= n && (reinterpret_cast<uintptr_t>(cnt) & 15u) == 0;
    if (vec_in) {
#pragma unroll
      for (int k = 0; k < PER; k += 4) {
        const int4 q = __ldg(reinterpret_cast<const int4*>(cnt + b + k));
        v[k] = q.x; v[k + 1] = q.y; v[k + 2] = q.z; v[k + 3] = q.w;
      }
    } else {
#pragma unroll
      for (int k = 0; k < PER; ++k) v[k] = (b + k < n) ? __ldg(cnt + b + k) : 0;
    }
#pragma unroll
    for (int k = 0; k < PER; ++k) sum += v[k];
    int32_t inc = sum;                                   // inclusive scan of the thread sums inside the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += y;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      int32_t w = warp_tot[lane], winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int32_t y = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += y;
      }
      warp_tot[lane] = winc - w;                         // exclusive offsets of the warps
      if (lane == 31) carry_s = winc;                    // chunk total
    }
    __syncthreads();
    OutT run = carry + static_cast<OutT>(warp_tot[warp] + inc - sum);
    if (sizeof(OutT) == 4 && b + PER <= n && (reinterpret_cast<uintptr_t>(out) & 15u) == 0) {
#pragma unroll
      for (int k = 0; k < PER; k += 4) {
        int4 q;
        q.x = static_cast<int32_t>(run); run += v[k];
        q.y = static_cast<int32_t>(run); run += v[k + 1];
        q.z = static_cast<int32_t>(run); run += v[k + 2];
        q.w = static_cast<int32_t>(run); run += v[k + 3];
        *reinterpret_cast<int4*>(reinterpret_cast<int32_t*>(out) + b + k) = q;
      }
    } else {
#pragma unroll
      for (int k = 0; k < PER; ++k) {
        if (b + k < n) out[b + k] = run;
        run += v[k];
      }
    }
    carry += carry_s;
    __syncthreads();                                     // warp_tot / carry_s are rewritten by the next chunk
  }
  if (t == 0) out[n] = carry;
}

// Entry (r,c) of A lands in row c of A^T.  Slots are claimed with integer cursors and each (short)
// output row is sorted afterwards: the sorted result is unique, hence deterministic.
__global__ void tr_fill_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                               int64_t n_rows, const int32_t* __restrict__ rowptr_t,
                               int32_t* __restrict__ cursor, int32_t* __restrict__ colidx_t) {
  const int64_t r = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (r >= n_rows) return;
  for (int e = rowptr[r]; e < rowptr[r + 1]; ++e) {
    const int c = colidx[e];
    const int slot = atomicAdd(cursor + c, 1);
    colidx_t[rowptr_t[c] + slot] = static_cast<int32_t>(r);
  }
}

__global__ void tr_sort_rows_kernel(const int32_t* __restrict__ rowptr_t, int64_t n_rows,
                                    int32_t* __restrict__ colidx_t) {
  const int64_t r = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (r >= n_rows) return;
  const int b = rowptr_t[r], e = rowptr_t[r + 1];
  for (int i = b + 1; i < e; ++i) {   // insertion sort: rows are short (degree ~12-64)
    const int32_t v = colidx_t[i];
    int k = i - 1;
    while (k >= b && colidx_t[k] > v) {
      colidx_t[k + 1] = colidx_t[k];
      --k;
    }
    colidx_t[k + 1] = v;
  }
}

__global__ void cast_f64_f32_kernel(const double* __restrict__ src, float* __restrict__ dst, int64_t n) {
  for (int64_t k = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; k < n;
       k += static_cast<int64_t>(gridDim.x) * blockDim.x)
    dst[k] = static_cast<float>(src[k]);   // cvt.rn.f32.f64
}

// Whole-graph gather out of a packed dataset (typically in PINNED HOST memory, read over the host link): CTA row j
// copies the contiguous slices of graph ids[j] - features, columns, row pointers (rebased), label - into a packed
// mini-dataset on the device.  Every access is a coalesced run (128-bit for the features), which the row-granular reads
// of batch_fill_kernel are not: the difference between ~5 and ~40 GB/s over PCIe.
__global__ void __launch_bounds__(256) gather_graphs_kernel(
    const int64_t* __restrict__ ids, int b, const int64_t* __restrict__ src_node_off, const int64_t* __restrict__ src_rowptr,
    const int32_t* __restrict__ src_col, const float* __restrict__ src_x, const float* __restrict__ src_y, int n_feat,
    int n_classes, const int64_t* __restrict__ dst_node_off, const int64_t* __restrict__ dst_edge_off,
    int64_t* __restrict__ dst_rowptr, int32_t* __restrict__ dst_col, float* __restrict__ dst_x, float* __restrict__ dst_y) {
  const int j = blockIdx.x;
  const int64_t g = ids[j];
  const int64_t n0 = src_node_off[g], n1 = src_node_off[g + 1];
  const int64_t e0 = src_rowptr[n0], e1 = src_rowptr[n1];
  const int64_t dn0 = dst_node_off[j], de0 = dst_edge_off[j];
  const int64_t tid = static_cast<int64_t>(blockIdx.y) * blockDim.x + threadIdx.x, nth = static_cast<int64_t>(gridDim.y) * blockDim.x;
  const int64_t nx = (n1 - n0) * n_feat;
  const float* sx = src_x + n0 * n_feat;
  float* dx = dst_x + dn0 * n_feat;
  if ((n_feat & 3) == 0 && ((reinterpret_cast<uintptr_t>(sx) | reinterpret_cast<uintptr_t>(dx)) & 15u) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(sx);
    float4* d4 = reinterpret_cast<float4*>(dx);
    for (int64_t i = tid; i < nx / 4; i += nth) d4[i] = s4[i];
  } else {
    for (int64_t i = tid; i < nx; i += nth) dx[i] = sx[i];
  }
  for (int64_t i = tid; i < e1 - e0; i += nth) dst_col[de0 + i] = src_col[e0 + i];
  for (int64_t i = tid; i < n1 - n0; i += nth) dst_rowptr[dn0 + i] = src_rowptr[n0 + i] - e0 + de0;
  if (j == b - 1 && tid == 0) dst_rowptr[dn0 + (n1 - n0)] = de0 + (e1 - e0);
  if (blockIdx.y == 0 && src_y)
    for (int c = threadIdx.x; c < n_classes; c += blockDim.x) dst_y[static_cast<int64_t>(j) * n_classes + c] = src_y[g * n_classes + c];
}

// Node-level labels (np.vstack of the graphs' [n_g, width] label blocks): CTA row j copies the contiguous row block of
// graph ids[j] to batch row graph_ptr[j].  Every access is a coalesced run - 128-bit when width and both addresses allow
// - so the source may sit in pinned host memory as well as in HBM.  Pure copies: deterministic.
__global__ void __launch_bounds__(256) gather_node_rows_kernel(
    const int64_t* __restrict__ ids, const int64_t* __restrict__ src_node_off, const float* __restrict__ src, int width,
    const int32_t* __restrict__ dst_graph_ptr, float* __restrict__ dst) {
  const int j = blockIdx.x;
  const int64_t g = ids[j];
  const int64_t n0 = src_node_off[g];
  const int64_t cnt = (src_node_off[g + 1] - n0) * width;
  const float* s = src + n0 * width;
  float* d = dst + static_cast<int64_t>(dst_graph_ptr[j]) * width;
  const int64_t tid = static_cast<int64_t>(blockIdx.y) * blockDim.x + threadIdx.x, nth = static_cast<int64_t>(gridDim.y) * blockDim.x;
  if ((width & 3) == 0 && ((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d)) & 15u) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(s);
    float4* d4 = reinterpret_cast<float4*>(d);
    for (int64_t i = tid; i < cnt / 4; i += nth) d4[i] = s4[i];
  } else {
    for (int64_t i = tid; i < cnt; i += nth) d[i] = s[i];
  }
}

// out[0..n] = exclusive prefix sums of cnt[0..n) (out[n] = total); shared with spmm.cu.
int exclusive_scan_i64(const int32_t* cnt, int64_t n, int64_t* out, cudaStream_t st) {
  exclusive_scan_kernel<int64_t><<<1, 1024, 0, st>>>(cnt, n, out);
  GCS_CHECK_LAUNCH("exclusive_scan_kernel<int64>");
  return GCS_OK;
}

int exclusive_scan_i32(const int32_t* cnt, int64_t n, int32_t* out, cudaStream_t st) {
  exclusive_scan_kernel<int32_t><<<1, 1024, 0, st>>>(cnt, n, out);
  GCS_CHECK_LAUNCH("exclusive_scan_kernel");
  return GCS_OK;
}

}  // namespace gcs

using namespace gcs;

extern "C" int gcs_batch_disjoint(const int64_t* ds_node_off, const int64_t* ds_rowptr,
                                  const int32_t* ds_col, const float* ds_x, const float* ds_y,
                                  int32_t n_feat, int32_t n_classes, const int64_t* graph_ids,
                                  int32_t n_graphs, int64_t n_nodes, int64_t nnz, int32_t* graph_ptr,
                                  int32_t* edge_ptr, int32_t* rowptr, int32_t* colidx, float* x,
                                  int64_t* seg_ids, float* y, int64_t* coo_indices,
                                  int32_t* status_dev, gcs_stream stream) {
  GCS_CHECK_ARG(ds_node_off && ds_rowptr && ds_col && ds_x && graph_ids, "gcs_batch_disjoint: null dataset pointer");
  GCS_CHECK_ARG(graph_ptr && edge_ptr && rowptr && colidx && x && seg_ids && status_dev, "gcs_batch_disjoint: null output pointer");
  GCS_CHECK_ARG(n_graphs >= 0 && n_nodes >= 0 && nnz >= 0 && n_feat > 0, "gcs_batch_disjoint: negative size");
  GCS_CHECK_ARG(n_nodes < INT32_MAX && nnz < INT32_MAX, "gcs_batch_disjoint: batch exceeds int32 CSR range");
  GCS_CHECK_ARG(!y || ds_y, "gcs_batch_disjoint: y requested but dataset has no labels");
  cudaStream_t st = as_stream(stream);
  batch_offsets_kernel<<<1, 1024, 0, st>>>(ds_node_off, ds_rowptr, graph_ids, n_graphs, n_nodes, nnz,
                                            graph_ptr, edge_ptr, status_dev);
  GCS_CHECK_LAUNCH("batch_offsets_kernel");
  if (n_graphs == 0) {
    GCS_CUDA(cudaMemsetAsync(rowptr, 0, sizeof(int32_t), st));
    return GCS_OK;
  }
  // chunks per graph: enough CTAs to fill the machine ~4x over, at most 16 per graph
  int chunks = static_cast<int>(ceil_div(4LL * sm_count() * 4, n_graphs));
  chunks = chunks < 1 ? 1 : (chunks > 16 ? 16 : chunks);
  dim3 grid(n_graphs, chunks);
  batch_fill_kernel<<<grid, 256, 0, st>>>(ds_node_off, ds_rowptr, ds_col, ds_x, ds_y, n_feat, n_classes,
                                          graph_ids, graph_ptr, edge_ptr, rowptr, colidx, x, seg_ids, y,
                                          coo_indices);
  GCS_CHECK_LAUNCH("batch_fill_kernel");
  return GCS_OK;
}

extern "C" int gcs_gather_graphs(const int64_t* graph_ids, int32_t n_graphs, const int64_t* src_node_off,
                                 const int64_t* src_rowptr, const int32_t* src_col, const float* src_x, const float* src_y,
                                 int32_t n_feat, int32_t n_classes, const int64_t* dst_node_off, const int64_t* dst_edge_off,
                                 int64_t* dst_rowptr, int32_t* dst_col, float* dst_x, float* dst_y, gcs_stream stream) {
  GCS_CHECK_ARG(n_graphs >= 0 && n_feat > 0 && n_classes >= 0, "gcs_gather_graphs: bad size");
  if (n_graphs == 0) return GCS_OK;
  GCS_CHECK_ARG(graph_ids && src_node_off && src_rowptr && src_col && src_x && dst_node_off && dst_edge_off && dst_rowptr &&
                dst_col && dst_x, "gcs_gather_graphs: null pointer");
  GCS_CHECK_ARG(!src_y || dst_y, "gcs_gather_graphs: labels need a destination");
  int chunks = static_cast<int>(ceil_div(8LL * sm_count(), n_graphs));      // >= 8 CTAs per SM in flight on the host link
  chunks = chunks < 1 ? 1 : (chunks > 32 ? 32 : chunks);
  dim3 grid(n_graphs, chunks);
  gather_graphs_kernel<<<grid, 256, 0, as_stream(stream)>>>(graph_ids, n_graphs, src_node_off, src_rowptr, src_col, src_x,
                                                           src_y, n_feat, n_classes, dst_node_off, dst_edge_off, dst_rowptr,
                                                           dst_col, dst_x, dst_y);
  GCS_CHECK_LAUNCH("gather_graphs_kernel");
  return GCS_OK;
}

extern "C" int gcs_gather_node_rows(const int64_t* graph_ids, int32_t n_graphs, const int64_t* src_node_off,
                                    const float* src, int32_t width, const int32_t* dst_graph_ptr, float* dst,
                                    gcs_stream stream) {
  GCS_CHECK_ARG(n_graphs >= 0 && width > 0, "gcs_gather_node_rows: bad size");
  if (n_graphs == 0) return GCS_OK;
  GCS_CHECK_ARG(graph_ids && src_node_off && src && dst_graph_ptr && dst, "gcs_gather_node_rows: null pointer");
  int chunks = static_cast<int>(ceil_div(8LL * sm_count(), n_graphs));      // as gcs_gather_graphs: host-link reads in flight
  chunks = chunks < 1 ? 1 : (chunks > 32 ? 32 : chunks);
  dim3 grid(n_graphs, chunks);
  gather_node_rows_kernel<<<grid, 256, 0, as_stream(stream)>>>(graph_ids, src_node_off, src, width, dst_graph_ptr, dst);
  GCS_CHECK_LAUNCH("gather_node_rows_kernel");
  return GCS_OK;
}

extern "C" int gcs_coo_to_csr(const int64_t* coo_indices, int64_t nnz, int64_t n_rows, int32_t* rowptr,
                              int32_t* colidx, int32_t* status_dev, gcs_stream stream) {
  GCS_CHECK_ARG(rowptr && status_dev && (nnz == 0 || (coo_indices && colidx)), "gcs_coo_to_csr: null pointer");
  GCS_CHECK_ARG(nnz >= 0 && n_rows >= 0 && nnz < INT32_MAX && n_rows < INT32_MAX, "gcs_coo_to_csr: size out of range");
  cudaStream_t st = as_stream(stream);
  coo_rowptr_kernel<<<static_cast<unsigned>(ceil_div(n_rows + 1, 256)), 256, 0, st>>>(coo_indices, nnz, n_rows, rowptr);
  GCS_CHECK_LAUNCH("coo_rowptr_kernel");
  if (nnz > 0) {
    coo_cols_kernel<<<static_cast<unsigned>(ceil_div(nnz, 256)), 256, 0, st>>>(coo_indices, nnz, n_rows, colidx, status_dev);
    GCS_CHECK_LAUNCH("coo_cols_kernel");
  }
  return GCS_OK;
}

extern "C" int gcs_segment_ptr(const int64_t* seg_ids, int64_t n_nodes, int32_t n_graphs,
                               int32_t* graph_ptr, int32_t* status_dev, gcs_stream stream) {
  GCS_CHECK_ARG(graph_ptr && status_dev && (n_nodes == 0 || seg_ids), "gcs_segment_ptr: null pointer");
  GCS_CHECK_ARG(n_nodes >= 0 && n_graphs >= 0 && n_nodes < INT32_MAX, "gcs_segment_ptr: size out of range");
  int64_t threads = n_graphs + 1;
  int64_t want = n_nodes < 1 ? threads : (n_nodes > threads ? n_nodes : threads);
  int64_t blocks = ceil_div(want, 256);
  if (blocks > 8LL * sm_count()) blocks = 8LL * sm_count();
  if (blocks * 256 < threads) blocks = ceil_div(threads, 256);
  segment_ptr_kernel<<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(seg_ids, n_nodes, n_graphs, graph_ptr, status_dev);
  GCS_CHECK_LAUNCH("segment_ptr_kernel");
  return GCS_OK;
}

extern "C" int gcs_csr_is_symmetric(const int32_t* rowptr, const int32_t* colidx, int64_t n_rows,
                                    int32_t* flag_dev, gcs_stream stream) {
  GCS_CHECK_ARG(rowptr && flag_dev && n_rows >= 0, "gcs_csr_is_symmetric: bad argument");
  cudaStream_t st = as_stream(stream);
  set_i32_kernel<<<1, 1, 0, st>>>(flag_dev, 1);
  GCS_CHECK_LAUNCH("set_i32_kernel");
  if (n_rows > 0) {
    csr_symmetric_kernel<<<static_cast<unsigned>(ceil_div(n_rows, 128)), 128, 0, st>>>(rowptr, colidx, n_rows, flag_dev);
    GCS_CHECK_LAUNCH("csr_symmetric_kernel");
  }
  return GCS_OK;
}

extern "C" int gcs_csr_transpose(const int32_t* rowptr, const int32_t* colidx, int64_t n_rows, int64_t nnz,
                                 int32_t* rowptr_t, int32_t* colidx_t, int32_t* workspace, gcs_stream stream) {
  GCS_CHECK_ARG(rowptr && rowptr_t && workspace && n_rows >= 0 && nnz >= 0, "gcs_csr_transpose: bad argument");
  GCS_CHECK_ARG(nnz == 0 || (colidx && colidx_t), "gcs_csr_transpose: null column array");
  cudaStream_t st = as_stream(stream);
  GCS_CUDA(cudaMemsetAsync(workspace, 0, sizeof(int32_t) * (n_rows + 1), st));
  if (nnz > 0) {
    tr_count_kernel<<<static_cast<unsigned>(ceil_div(nnz, 256)), 256, 0, st>>>(colidx, nnz, workspace);
    GCS_CHECK_LAUNCH("tr_count_kernel");
  }
  exclusive_scan_kernel<int32_t><<<1, 1024, 0, st>>>(workspace, n_rows, rowptr_t);
  GCS_CHECK_LAUNCH("exclusive_scan_kernel");
  if (nnz > 0 && n_rows > 0) {
    GCS_CUDA(cudaMemsetAsync(workspace, 0, sizeof(int32_t) * (n_rows + 1), st));
    tr_fill_kernel<<<static_cast<unsigned>(ceil_div(n_rows, 128)), 128, 0, st>>>(rowptr, colidx, n_rows, rowptr_t, workspace, colidx_t);
    GCS_CHECK_LAUNCH("tr_fill_kernel");
    tr_sort_rows_kernel<<<static_cast<unsigned>(ceil_div(n_rows, 128)), 128, 0, st>>>(rowptr_t, n_rows, colidx_t);
    GCS_CHECK_LAUNCH("tr_sort_rows_kernel");
  }
  return GCS_OK;
}

extern "C" int gcs_cast_f64_f32(const double* src, float* dst, int64_t n, gcs_stream stream) {
  GCS_CHECK_ARG(n >= 0 && (n == 0 || (src && dst)), "gcs_cast_f64_f32: bad argument");
  if (n == 0) return GCS_OK;
  int64_t blocks = ceil_div(n, 256);
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  cast_f64_f32_kernel<<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(src, dst, n);
  GCS_CHECK_LAUNCH("cast_f64_f32_kernel");
  return GCS_OK;
}
