/* gcnstring_b200 — C ABI of the B200-native GeneralGNN hot path.
 *
 * This header is the drop-in boundary (SURVEY.md §8b).  The reference
 * (Sum02dean/GCN-STRING) has no native code and no FFI of its own: its hot path is the
 * one-line model `GeneralGNN(dataset.n_labels, activation="softmax")`
 * (src/scripts/gcn.py:320) executed inside un-vendored Spektral/TensorFlow.  Each entry
 * point below therefore cites the reference call site / upstream op group it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; every pointer is a DEVICE pointer unless the
 *     name ends in `_host`.  No torch / DLPack types cross this boundary: the Python
 *     wrapper unwraps `__dlpack__` objects to raw pointers zero-copy.
 *   - every function returns a status (0 = GCS_OK); `gcs_last_error()` returns a
 *     thread-local message for the last non-zero status.  No exceptions cross the ABI.
 *   - the caller owns every buffer, including workspaces (sized by the *_workspace_bytes
 *     queries); the library never allocates device memory and never synchronises: all
 *     work is enqueued on the `stream` argument (a cudaStream_t passed as void*).
 *   - float tensors are row-major fp32 with an explicit leading dimension (`ld*`, in
 *     elements) so that slices of the concat buffer are addressed in place.
 *   - integer graph structure is int32 inside (CSR), int64 where Spektral's loader emits
 *     int64 (`i`, SparseTensor.indices).
 *   - reductions are order-deterministic (no floating-point atomics anywhere).
 */
#ifndef GCNSTRING_B200_H
#define GCNSTRING_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gcs_stream; /* cudaStream_t */

enum gcs_status {
  GCS_OK = 0,
  GCS_ERR_INVALID_ARGUMENT = 1, /* bad shape / null pointer / misaligned */
  GCS_ERR_UNSUPPORTED = 2,      /* configuration outside the native subset */
  GCS_ERR_WORKSPACE = 3,        /* workspace too small */
  GCS_ERR_CUDA = 4,             /* a CUDA runtime call or launch failed */
  GCS_ERR_NCCL = 5              /* NCCL missing or a collective failed */
};

int gcs_version(void);
const char* gcs_last_error(void);
/* SM count of the current device (grid sizing); <0 on error. */
int gcs_device_sm_count(void);

/* Optional synchronised BatchNorm for data-parallel runs (SURVEY.md 8e lists it as the variant in which a G-GPU
 * step equals ONE reference step on the union of the shards).  While a hook is installed (per host thread),
 * gcs_bn_stats and gcs_bn_prelu_bwd - and therefore the model entry points - hand their per-column fp64 sums
 * (sum h, sum h^2 | sum dz, sum dz*xhat, sum da*min(z,0), then the local row count as the last element) to `fn`,
 * which must SUM the `n` doubles at `device_buf` over all ranks, in place, enqueued on `stream`; mean / variance and
 * the gradient coefficients are then formed from the global sums and the global row count.  dgamma / dbeta / dalpha
 * are written as (global sum) / world_size so that the caller's SUM all-reduce of the flat gradient buffer restores
 * them.  fn == NULL removes the hook (the default: replica-local statistics, gradient all-reduce only). */
typedef int (*gcs_allreduce_fn)(double* device_buf, int64_t n, gcs_stream stream, void* user);
int gcs_set_allreduce_hook(gcs_allreduce_fn fn, void* user, int32_t world_size);

/* ---------------------------------------------------------------------------------
 * K0  Disjoint batching on the device.
 * Replaces spektral.data.DisjointLoader.collate as driven by src/scripts/gcn.py:316-317,
 * :350, :367 (np.vstack / sp.block_diag / sp.find / tf.sparse.reorder / np.repeat on the
 * host, every step).  Input is the packed dataset resident in HBM (per-graph CSR with
 * local column indices, see gcn-string_b200/synthetic.py:PackedGraphs); `graph_ids` is
 * this step's slice of the epoch permutation.  n_nodes / nnz are the batch totals the
 * host already knows (sums of per-graph sizes); they are validated on the device and a
 * non-zero value is written to *status_dev on mismatch.
 * Outputs: graph_ptr[B+1], edge_ptr[B+1], rowptr[N+1], colidx[nnz] (global ids), x[N,F],
 * seg_ids[N] (Spektral's `i`, int64), y[B,C] (optional), coo_indices[nnz,2] (optional,
 * SparseTensor.indices in tf.sparse.reorder order).
 * --------------------------------------------------------------------------------- */
int gcs_batch_disjoint(const int64_t* ds_node_off, const int64_t* ds_rowptr, const int32_t* ds_col,
                       const float* ds_x, const float* ds_y, int32_t n_feat, int32_t n_classes,
                       const int64_t* graph_ids, int32_t n_graphs, int64_t n_nodes, int64_t nnz,
                       int32_t* graph_ptr, int32_t* edge_ptr, int32_t* rowptr, int32_t* colidx,
                       float* x, int64_t* seg_ids, float* y, int64_t* coo_indices,
                       int32_t* status_dev, gcs_stream stream);

/* Whole-graph gather for a streaming loader: copies the graphs graph_ids[0..n_graphs) of a packed dataset - typically
 * resident in PINNED HOST memory, read by the kernel over the host link in coalesced runs - into a packed mini-dataset
 * on the device (node_off = dst_node_off, rebased row pointers, graph-local columns, features, labels) that
 * gcs_batch_disjoint then batches with graph ids 0..n_graphs-1.  dst_node_off / dst_edge_off [n_graphs + 1] (device):
 * exclusive prefix sums of the selected graphs' node / entry counts, which the host knows.  src_y / dst_y may be NULL. */
int gcs_gather_graphs(const int64_t* graph_ids, int32_t n_graphs, const int64_t* src_node_off,
                      const int64_t* src_rowptr, const int32_t* src_col, const float* src_x, const float* src_y,
                      int32_t n_feat, int32_t n_classes, const int64_t* dst_node_off, const int64_t* dst_edge_off,
                      int64_t* dst_rowptr, int32_t* dst_col, float* dst_x, float* dst_y, gcs_stream stream);

/* Node-level labels of a disjoint batch.  Replaces Spektral's collate_labels_disjoint(y_list, node_level=True) =
 * np.vstack(y_list): copies the [n_g, width] row block of every graph graph_ids[0..n_graphs) out of a packed node-row
 * array src [sum n, width] (row offsets src_node_off [G + 1], as ds_node_off) to batch rows
 * [dst_graph_ptr[j], dst_graph_ptr[j + 1]) of dst [N, width] - the graph_ptr gcs_batch_disjoint just wrote (which is
 * then called with ds_y = y = NULL).  src / src_node_off may be in HBM or in pinned host memory (read over the host
 * link in coalesced runs, 128-bit when width and alignment allow).  One launch; graphs of 0 rows copy nothing. */
int gcs_gather_node_rows(const int64_t* graph_ids, int32_t n_graphs, const int64_t* src_node_off, const float* src,
                         int32_t width, const int32_t* dst_graph_ptr, float* dst, gcs_stream stream);

/* Row-major-sorted COO (what tf.sparse.reorder returns; Spektral's
 * sp_matrix_to_sp_tensor) -> int32 CSR.  *status_dev != 0 if unsorted/out of range. */
int gcs_coo_to_csr(const int64_t* coo_indices, int64_t nnz, int64_t n_rows, int32_t* rowptr,
                   int32_t* colidx, int32_t* status_dev, gcs_stream stream);
/* graph_ptr[B+1] from the sorted batch index `i` (GlobalSumPool's second input). */
int gcs_segment_ptr(const int64_t* seg_ids, int64_t n_nodes, int32_t n_graphs, int32_t* graph_ptr,
                    int32_t* status_dev, gcs_stream stream);
/* *flag_dev = 1 if pattern(A) == pattern(A)^T (every reference graph is), else 0. */
int gcs_csr_is_symmetric(const int32_t* rowptr, const int32_t* colidx, int64_t n_rows,
                         int32_t* flag_dev, gcs_stream stream);
/* CSR of pattern(A)^T, columns ascending within a row (needed by the backward SpMM for
 * non-symmetric input).  workspace: (n_rows + 1) int32. */
int gcs_csr_transpose(const int32_t* rowptr, const int32_t* colidx, int64_t n_rows, int64_t nnz,
                      int32_t* rowptr_t, int32_t* colidx_t, int32_t* workspace, gcs_stream stream);
/* float64 -> float32 round-to-nearest (Keras autocast of the f64 features the
 * reference's MyDataset produces, gcn.py:128,174). */
int gcs_cast_f64_f32(const double* src, float* dst, int64_t n, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K1/K9  Dense transforms (Keras Dense / K.dot + bias_add inside MLP and GeneralConv).
 *   fwd:        C[M,N]  = A[M,K] . W[K,N] + bias[N]           (bias may be NULL)
 *   bwd_weight: dW[K,N] = A[M,K]^T . dH[M,N];  db[N] = colsum(dH)   (db may be NULL)
 *               workspace: gcs_linear_bwd_weight_workspace_bytes(M,K,N)
 *   bwd_input:  dA[M,K] (+)= dH[M,N] . W[K,N]^T               (accumulate != 0 adds)
 * fwd / bwd_input run on the tensor cores (tcgen05; error-compensated operand splits, fp32-accurate) when the
 * reduction width is a multiple of 32, the output width a multiple of 128 and a workspace
 * of gcs_linear_workspace_bytes(M,K,N) is given (it holds the split weights); otherwise, or
 * with workspace == NULL, on the CUDA cores (exact fp32 FFMA).  These standalone entry points use the 3 x TF32
 * split; inside gcs_model_forward / gcs_model_train_step, where the producer kernels maintain the |max| of every
 * activation / gradient tensor, the same transforms run as 3 x FP16 products (hi + 2^11-scaled lo, power-of-two
 * operand scales) at twice the MMA rate with the same 22-bit operand precision.
 * --------------------------------------------------------------------------------- */
int64_t gcs_linear_workspace_bytes(int64_t M, int32_t K, int32_t N);
int gcs_linear_fwd(const float* A, int64_t lda, const float* W, const float* bias, float* C,
                   int64_t ldc, int64_t M, int32_t K, int32_t N, void* workspace,
                   int64_t workspace_bytes, gcs_stream stream);
int64_t gcs_linear_bwd_weight_workspace_bytes(int64_t M, int32_t K, int32_t N);
int gcs_linear_bwd_weight(const float* A, int64_t lda, const float* dH, int64_t ldh, float* dW,
                          float* db, int64_t M, int32_t K, int32_t N, void* workspace,
                          int64_t workspace_bytes, gcs_stream stream);
int gcs_linear_bwd_input(const float* dH, int64_t ldh, const float* W, float* dA, int64_t lda,
                         int64_t M, int32_t K, int32_t N, int32_t accumulate, void* workspace,
                         int64_t workspace_bytes, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K2/K8  BatchNormalization(momentum, epsilon) + PReLU (Keras defaults; rank-2 input).
 *   bn_stats:   biased batch moments over the M rows (tf.nn.moments), fp64 accumulation.
 *               workspace: gcs_bn_workspace_bytes(M, C)
 *   bn_fold:    scale = gamma * rsqrt(var + eps); shift = beta - mean * scale; if
 *               moving_mean/var != NULL: moving -= (moving - batch) * (1 - momentum).
 *               (inference: pass the moving statistics as mean/var and NULL moving_*)
 *   bn_prelu_fwd: out = prelu(h * scale + shift, alpha)   (alpha NULL -> identity)
 *   bn_prelu_bwd: given da = dLoss/d(out): dgamma, dbeta, dalpha (NULL-able) and
 *               dh = dLoss/dh for training-mode BN.  dbias (NULL-able) receives the column
 *               sums of dh, i.e. the bias gradient of the dense layer that produced h, so
 *               that gcs_linear_bwd_weight can be called with db = NULL (one read of dh
 *               saved).  workspace as bn_stats.
 * --------------------------------------------------------------------------------- */
int64_t gcs_bn_workspace_bytes(int64_t M, int32_t C);
int gcs_bn_stats(const float* h, int64_t ldh, int64_t M, int32_t C, float* mean, float* var,
                 void* workspace, int64_t workspace_bytes, gcs_stream stream);
int gcs_bn_fold(const float* mean, const float* var, const float* gamma, const float* beta,
                float eps, float momentum, float* moving_mean, float* moving_var, float* scale,
                float* shift, int32_t C, gcs_stream stream);
int gcs_bn_prelu_fwd(const float* h, int64_t ldh, const float* scale, const float* shift,
                     const float* alpha, float* out, int64_t ldo, int64_t M, int32_t C,
                     gcs_stream stream);
int gcs_bn_prelu_bwd(const float* da, int64_t ldda, const float* h, int64_t ldh, const float* mean,
                     const float* var, const float* gamma, const float* beta, const float* alpha,
                     float eps, float* dh, int64_t lddh, float* dgamma, float* dbeta,
                     float* dalpha, float* dbias, int64_t M, int32_t C, void* workspace,
                     int64_t workspace_bytes, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K3/K7  Sum aggregation  Y = pattern(A) . f(X)   (MessagePassing.propagate: tf.gather +
 * tf.math.unsorted_segment_sum, the messages never materialised).  f is the fused
 * BatchNorm+PReLU prologue of GeneralConv.call, f(x) = prelu(x*scale + shift, alpha);
 * pass scale = shift = alpha = NULL for f = identity (that is also the backward:
 * dX = pattern(A)^T . dY, called with the transposed CSR).  Every output element has one owner that adds its
 * neighbours in a fixed order (no atomics): ascending column for the CSR row kernels, the order of the row-block list
 * for the row-block kernels - results are reproducible run to run and differ between the two families only by the
 * float32 rounding of a reordered sum (~1e-7).
 * Row-block format (optional): gcs_spmm_build_rb derives, once per batch, the row-block form of the CSR: per block of
 * rb_height (2 or 4) consecutive rows the union of their columns, each entry (col << 8) | mask-of-rows.  Banded
 * residue graphs share most neighbours between consecutive rows, so a neighbour row is gathered once per block instead
 * of once per row.  Order inside a block: first whole groups of four entries that ALL rows of the block have (mask all
 * ones, ascending column, bit 4 of the word set: a kernel may sum them once for the whole block), then every other
 * entry in ascending column order.  Every block is padded to a multiple of 4 entries (mask 0: no-ops) so that it starts
 * on a 16-byte boundary.  rb_blk_ptr needs ceil(n_rows/rb_height)+1 int32 (allocate 3 more: gcs_spmm_sum_graphs copies it in
 * 16-byte units), rb_ent nnz + 3*ceil(n_rows/rb_height) uint32 (upper bound); both 16-byte aligned; workspace
 * gcs_spmm_rb_workspace_bytes(n_rows, rb_height); n_rows < 2^24.  gcs_spmm_build_rb4 = height 4 (the only height the
 * global-memory kernel behind gcs_spmm_sum / gcs_spmm_aggregate reads).  With rb_* == NULL the CSR row kernels run.
 * Any matrix structure is accepted either way.
 * --------------------------------------------------------------------------------- */
int64_t gcs_spmm_rb_workspace_bytes(int64_t n_rows, int32_t rb_height);
int gcs_spmm_build_rb(const int32_t* rowptr, const int32_t* colidx, int64_t n_rows, int64_t nnz, int32_t rb_height,
                      int32_t* rb_blk_ptr, uint32_t* rb_ent, void* workspace, int64_t workspace_bytes,
                      gcs_stream stream);
int64_t gcs_spmm_rb4_workspace_bytes(int64_t n_rows);
int gcs_spmm_build_rb4(const int32_t* rowptr, const int32_t* colidx, int64_t n_rows, int64_t nnz,
                       int32_t* rb4_blk_ptr, uint32_t* rb4_ent, void* workspace, int64_t workspace_bytes,
                       gcs_stream stream);
int gcs_spmm_sum(const int32_t* rowptr, const int32_t* colidx, const int32_t* rb4_blk_ptr,
                 const uint32_t* rb4_ent, int64_t n_rows, const float* X, int64_t ldx,
                 const float* scale, const float* shift, const float* alpha, float* Y, int64_t ldy,
                 int32_t H, gcs_stream stream);

/* The same aggregation for a DISJOINT BATCH (what DisjointLoader emits, gcn.py:316-317): pattern(A) is block-diagonal,
 * graph g owns rows and columns [graph_ptr[g], graph_ptr[g+1]).  One thread block per (graph, 32 feature columns) stages
 * that slice of X in shared memory - every element of X leaves HBM once, the BatchNorm+PReLU prologue is applied once
 * per element - and serves all gathers of the graph from there.  max_graph_nodes = the longest graph of the batch
 * (the loader knows it on the host; 0 = unknown).  Batches whose graphs do not fit a shared-memory slab (or
 * graph_ptr == NULL, or rb_* == NULL) run on the global-memory kernels of gcs_spmm_aggregate.  An entry that leaves its graph's column
 * range is ignored (a caller error).  rb_* / rb_height as above; residual as in gcs_spmm_aggregate.  Results are bit-identical to
 * gcs_spmm_sum on the same row-block list.  Work items are handed to the persistent thread blocks through a ticket counter in
 * device memory that the kernel re-arms itself (up to 64 launches of one device may be in flight at once). */
int64_t gcs_spmm_slab_stage_bytes(void); /* bytes of one shared-memory stage: a graph runs 4 << k columns wide when
                                            n_nodes * (16 << k) + its row-block entries fit; the slab kernel takes a batch
                                            when max_graph_nodes * 16 and (n_rows / n_graphs) * 64 are both <= this */
int gcs_spmm_sum_graphs(const int32_t* graph_ptr, int32_t n_graphs, int32_t max_graph_nodes, const int32_t* rowptr,
                        const int32_t* colidx, const int32_t* rb_blk_ptr, const uint32_t* rb_ent, int32_t rb_height,
                        int64_t n_rows, const float* X, int64_t ldx, const float* scale, const float* shift,
                        const float* alpha, const float* residual, int64_t ldr, float* Y, int64_t ldy, int32_t H,
                        gcs_stream stream);

/* General form (SURVEY.md 8 f3 and the 'sum' skip connection of GeneralGNN.call):
 *   Y = agg_j( w_ij * f(X[j]) ) + residual
 * values   : optional per-entry weights in CSR order (the reference computes `dca` / `proximity` edge attributes,
 *            gcn.py:130-157, behind a `use_edge_data` switch); NULL = pattern only, as GeneralConv does.
 * aggregate: 0 sum (scatter_sum), 1 mean (scatter_mean = unsorted_segment_mean: sum / number of entries of the row,
 *            0 for an empty row), 2 max (scatter_max = unsorted_segment_max: the lowest float for an empty row).
 * residual : optional [n_rows, H] operand added after the aggregation - Keras Add()([z, out]) of
 *            connectivity='sum' - NULL otherwise.
 * The RB4 kernel serves aggregate = 0 without weights (with or without residual); everything else runs row by row.
 * Any H > 0 (as in gcs_spmm_aggregate_bwd): rows wider than one thread block are split into column slices.
 * gcs_spmm_sum(...) == gcs_spmm_aggregate(..., values = NULL, residual = NULL, aggregate = 0). */
int gcs_spmm_aggregate(const int32_t* rowptr, const int32_t* colidx, const float* values,
                       const int32_t* rb4_blk_ptr, const uint32_t* rb4_ent, int64_t n_rows, const float* X,
                       int64_t ldx, const float* scale, const float* shift, const float* alpha,
                       const float* residual, int64_t ldr, float* Y, int64_t ldy, int32_t H,
                       int32_t aggregate, gcs_stream stream);

/* Gradient of gcs_spmm_aggregate with respect to f(X): dA[j] = sum_i w_ij * dZ[i] (sum), / (entries of row i) (mean),
 * or - max - only where w_ij * f(X[j]) attains the maximum Z[i], shared equally between ties (the gradient of
 * tf.math.unsorted_segment_max).  (rowptr_t, colidx_t, values_t): the transposed pattern with the weights in that order
 * (alias the forward arrays for a symmetric matrix with symmetric weights).  mean also reads the forward rowptr; max also
 * reads the forward pattern + weights, X with its prologue, the forward output Z, and uses ties[n_rows, H] as scratch. */
int gcs_spmm_aggregate_bwd(const int32_t* rowptr_t, const int32_t* colidx_t, const float* values_t,
                           const int32_t* rowptr, const int32_t* colidx, const float* values, int64_t n_rows,
                           const float* dZ, int64_t lddz, int32_t aggregate, const float* X, int64_t ldx,
                           const float* scale, const float* shift, const float* alpha, const float* Z, int64_t ldz,
                           float* ties, int64_t ldt, float* dA, int64_t ldda, int32_t H, gcs_stream stream);

/* Gradient of gcs_spmm_aggregate with respect to its per-entry weights (an SDDMM over the forward pattern): for stored
 * entry e = (i, j) of row i, with a = f(X) the transformed rows the aggregation read,
 *   sum : dvalues[e] = sum_c dZ[i, c] * a[j, c]          mean: the same / (entries of row i)
 *   max : the same over the columns where values[e] * a[j, c] attains Z[i, c] only, each divided by the tie count
 *         ties[i, c] that gcs_spmm_aggregate_bwd (aggregate = 2) left in its `ties` scratch - call it first, with the
 *         same forward pattern, X, prologue and Z.
 * Output in forward CSR order (the order of `values`); accumulate != 0 adds to dvalues.  One writer per entry, no
 * atomics: bit-identical from run to run.  H <= 512.  The reference's tf.GradientTape.gradient(pred, a.values) for the
 * edge weights of its `use_edge_data` switch (gcn.py:73-80). */
int gcs_spmm_edge_grad(const int32_t* rowptr, const int32_t* colidx, const float* values, int64_t n_rows,
                       const float* dZ, int64_t lddz, int32_t aggregate, const float* X, int64_t ldx,
                       const float* scale, const float* shift, const float* alpha, const float* Z, int64_t ldz,
                       const float* ties, int64_t ldt, int32_t H, float* dvalues, int32_t accumulate,
                       gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K4/K6  GlobalSumPool = tf.math.segment_sum(X, i) over sorted graph ids, and its
 * gradient dX[n] = dOut[i[n]].
 * --------------------------------------------------------------------------------- */
int gcs_segment_sum_fwd(const float* X, int64_t ldx, const int32_t* graph_ptr, int32_t n_graphs,
                        int32_t W, float* out, int64_t ldo, gcs_stream stream);
int gcs_segment_sum_bwd(const float* dout, int64_t ldo, const int32_t* graph_ptr, int32_t n_graphs,
                        int32_t W, float* dX, int64_t ldx, gcs_stream stream);
/* GlobalAvgPool = tf.math.segment_mean(X, i): the segment sum divided by the graph's row count, 0 for an empty graph;
 * gradient dX[n] = dOut[i[n]] / n_{i[n]}.  Same parameters as gcs_segment_sum_*. */
int gcs_segment_mean_fwd(const float* X, int64_t ldx, const int32_t* graph_ptr, int32_t n_graphs,
                         int32_t W, float* out, int64_t ldo, gcs_stream stream);
int gcs_segment_mean_bwd(const float* dout, int64_t ldo, const int32_t* graph_ptr, int32_t n_graphs,
                         int32_t W, float* dX, int64_t ldx, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K4b/K6b  GlobalAttnSumPool (spektral.layers.pooling.GlobalAttnSumPool) over sorted graph ids.
 *   s_n = X_n . kernel,  p = unsorted_segment_softmax(s, i) = exp(s - max_g) / (sum_g exp(s - max_g) + 1e-9),
 *   out[g] = sum_{n in g} p_n X_n  (0 for an empty graph).  kernel [W] is Spektral's attn_kernel [W, 1].
 * fwd: scores [n_rows] (the s_n) and gstats [2 * n_graphs] ({max_g, sum_g exp(s - max_g)}) are NULL-able; the
 *      backward needs both, together with `out`.
 * bwd: with u_g = out_g . dOut_g:  ds_n = p_n (X_n . dOut_g - u_g),  dX_n = p_n dOut_g + ds_n kernel (written in full),
 *      dkernel = sum_n ds_n X_n (overwritten).
 * One pass over X each; long graphs are split over several thread blocks (fixed by n_rows and n_graphs) whose partials
 * are combined in a fixed order - bit-identical run to run.  W <= 8192 (W <= 2048 when W, a leading dimension or a
 * pointer is not a multiple of 4 floats).  workspace: gcs_attn_pool_workspace_bytes(n_rows, n_graphs, W), 16-byte
 * aligned, for either direction.
 * --------------------------------------------------------------------------------- */
int64_t gcs_attn_pool_workspace_bytes(int64_t n_rows, int32_t n_graphs, int32_t W);
int gcs_attn_sum_pool_fwd(const float* X, int64_t ldx, int64_t n_rows, const float* kernel, const int32_t* graph_ptr,
                          int32_t n_graphs, int32_t W, float* out, int64_t ldo, float* scores, float* gstats,
                          void* workspace, int64_t workspace_bytes, gcs_stream stream);
int gcs_attn_sum_pool_bwd(const float* dout, int64_t lddo, const float* X, int64_t ldx, int64_t n_rows,
                          const float* kernel, const int32_t* graph_ptr, int32_t n_graphs, int32_t W,
                          const float* out, int64_t ldo, const float* scores, const float* gstats, float* dX,
                          int64_t lddx, float* dkernel, void* workspace, int64_t workspace_bytes, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K5  softmax + CategoricalCrossentropy (mean over the batch) + categorical_accuracy
 * (gcn.py:326,335,339).  probs[B,C]; loss_acc[2] = {loss, accuracy}; dlogits (NULL-able)
 * = (probs * sum(y) - y) * grad_scale  (grad_scale = 1/B for the reference's mean loss;
 * 1/global_B under data parallelism).  C <= 64.
 * --------------------------------------------------------------------------------- */
int gcs_softmax_xent(const float* logits, const float* y, int32_t B, int32_t C, float* probs,
                     float* loss_acc, float* dlogits, float grad_scale, gcs_stream stream);
/* The same for any number of rows.  Up to 65 536 rows (B <= 65536) it IS gcs_softmax_xent (one thread block) and
 * needs no workspace; above, a grid-wide kernel runs the same per-row expressions - probs and dlogits are bit-identical
 * to gcs_softmax_xent's - and leaves per-block fp64 loss sums and integer hit counts in the workspace, which a second
 * launch adds in a fixed order (bit-identical run to run).  The choice depends on B alone.  workspace:
 * gcs_softmax_xent_workspace_bytes(B, C) bytes, 8-byte aligned (only read when loss_acc != NULL). */
int64_t gcs_softmax_xent_workspace_bytes(int64_t B, int32_t C);
int gcs_softmax_xent_ws(const float* logits, const float* y, int32_t B, int32_t C, float* probs, float* loss_acc,
                        float* dlogits, float grad_scale, void* workspace, int64_t workspace_bytes, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K5b  sigmoid + BinaryCrossentropy + binary_accuracy: the head of GeneralGNN(C, activation="sigmoid") trained with
 * tf.keras.losses.BinaryCrossentropy() and tf.keras.metrics.binary_accuracy (binary and multi-label targets, graph- or
 * node-level).  Per element l = max(z, 0) - z*y + log1p(exp(-|z|)) (tf.nn.sigmoid_cross_entropy_with_logits);
 *   probs[rows,C] = sigmoid(logits) (NULL-able);
 *   loss_acc[2] = {mean over rows of the mean over the C columns of l, mean of y == (probs > 0.5)} (NULL-able);
 *   dlogits (NULL-able) = (probs - y) * grad_scale / C  (grad_scale = 1/rows for the mean loss; 1/global_rows under
 *   data parallelism).
 * Labels y may be multi-hot or soft, in [0, 1]; y may be NULL when only probs is asked for.  Any C, rows = 0 gives
 * loss_acc = {0, 0}.  A grid-wide elementwise kernel leaves per-block fp64 loss sums and integer hit counts in the
 * workspace and a second launch adds them in a fixed order (bit-identical run to run; the grid depends on rows * C
 * alone).  workspace: gcs_sigmoid_bce_workspace_bytes(rows, C) bytes, 8-byte aligned (only read when loss_acc != NULL;
 * 0 bytes when rows * C <= 1024).
 * --------------------------------------------------------------------------------- */
int64_t gcs_sigmoid_bce_workspace_bytes(int64_t rows, int32_t C);
int gcs_sigmoid_bce(const float* logits, const float* y, int64_t rows, int32_t C, float* probs, float* loss_acc,
                    float* dlogits, float grad_scale, void* workspace, int64_t workspace_bytes, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K5c  Regression losses of a linear head: GeneralGNN(C) (activation=None) trained with tf.keras.losses
 * MeanSquaredError(), MeanAbsoluteError() or Huber(delta), and tf.keras.metrics.mean_absolute_error.  kind: 1 = MSE,
 * 2 = MAE, 3 = Huber (huber_delta finite and > 0; ignored otherwise).  Per element, e = pred - y in float32:
 *   MSE l = e^2, dl = 2e;  MAE l = |e|, dl = sign(e) (sign(0) = 0);
 *   Huber l = 0.5 e^2 if |e| <= delta, else delta |e| - 0.5 delta^2;  dl = e, or delta sign(e).
 *   loss_acc[2] = {mean over rows of the mean over the C columns of l, mean of |e|} (NULL-able);
 *   probs[rows,C] (NULL-able) = pred (the predictions of a linear head are its logits);
 *   dlogits (NULL-able) = dl * grad_scale / C  (grad_scale = 1/rows for the mean loss; 1/global_rows under data
 *   parallelism).
 * y may be NULL when only probs is asked for (a copy, nothing else is computed).  Any C, rows = 0 gives
 * loss_acc = {0, 0}.  A grid-wide elementwise kernel leaves per-block fp64 sums in the workspace and a second launch adds
 * them in a fixed order (bit-identical run to run; the grid depends on rows * C alone).  workspace:
 * gcs_regression_loss_workspace_bytes(rows, C) bytes, 8-byte aligned (only read when loss_acc != NULL; 0 bytes when
 * rows * C <= 1024).
 * --------------------------------------------------------------------------------- */
int64_t gcs_regression_loss_workspace_bytes(int64_t rows, int32_t C);
int gcs_regression_loss(int32_t kind, float huber_delta, const float* pred, const float* y, int64_t rows, int32_t C,
                        float* probs, float* loss_acc, float* dlogits, float grad_scale, void* workspace,
                        int64_t workspace_bytes, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K5d  The three heads above with one weight per row: Keras' loss(y, pred, sample_weight=w) with the default
 * "sum_over_batch_size" reduction, and the sample-weighted metric.  head: 1 = softmax + categorical cross-entropy
 * (C <= 64), 2 = sigmoid + binary cross-entropy, 0 = linear head with the regression loss `kind` (1 = MSE, 2 = MAE,
 * 3 = Huber with huber_delta; kind is ignored for the other heads).  sample_weight [rows] (device, required: the entry
 * points above are the unweighted path) may hold any finite values, 0 included; nothing is validated on the device.
 * With l_r the row loss and m_r the row metric of the unweighted entry point:
 *   loss_acc[0] = sum_r w_r l_r / rows   (divided by the row count, not by sum w);
 *   loss_acc[1] = sum_r w_r m_r / sum_r w_r, 0 when sum w = 0;
 *   dlogits     = w_r * (the unweighted dlogits of row r), so grad_scale keeps its meaning (1/rows, 1/global_rows).
 * probs as the unweighted entry point.  With every weight 1, loss_acc[0], probs and dlogits are bit-identical to the
 * unweighted entry point's, and loss_acc[1] is within one float ulp.  The grid follows the unweighted rule (rows alone
 * for the softmax, rows * C otherwise), so results are bit-identical run to run.  workspace:
 * gcs_weighted_loss_workspace_bytes(head, rows, C) bytes, 8-byte aligned (24 bytes per block of the grid; only read
 * when loss_acc != NULL).
 * --------------------------------------------------------------------------------- */
int64_t gcs_weighted_loss_workspace_bytes(int32_t head, int64_t rows, int32_t C);
int gcs_weighted_loss(int32_t head, int32_t kind, float huber_delta, const float* logits, const float* y,
                      const float* sample_weight, int64_t rows, int32_t C, float* probs, float* loss_acc,
                      float* dlogits, float grad_scale, void* workspace, int64_t workspace_bytes, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K11  Residue contact maps of a batch of chains (SURVEY.md 8 f4).  Replaces
 * GraphMaker.calculate_residue_dist / calculate_dist_matrix / generate_proximity_matrix
 * (src/utilities/gcn_utills.py:161-238): d = sqrt(sum((ca_i - ca_j)^2)) in float32 with NumPy's operation order
 * and no fused multiply-add, adjacency = d < angstroms (the diagonal gives the self-loops), evaluated per chain.
 *   ca[n_residues, 3] float32 (Bio.PDB atom coordinates), chain_ptr[n_chains + 1] int32 residue offsets.
 *   gcs_contact_map_rowptr: rowptr[n_residues + 1] int64 (exclusive scan of the row counts; rowptr[n_residues] = nnz,
 *     which the caller reads back to size `col`); workspace gcs_contact_workspace_bytes(n_residues).
 *   gcs_contact_map_fill:   col[nnz] int32 chain-local column ids, ascending per row; dist[nnz] float32 (NULL-able),
 *     the contact_map values the reference derives its `proximity` edge attribute from (:424-478).
 * K12  Inter-protein pair graphs: GraphMaker.generate_graphs + link_graphs (:240-270, :319-377) followed by the
 * adjacency gcn.py:104-117,184-197 takes from the union graph: nodes of chain pair_a[p] then of chain pair_b[p],
 * both chains' contacts, plus one symmetric edge (bridge_a[q], n_a + bridge_b[q]) per DCA bridge
 * q in [bridge_ptr[p], bridge_ptr[p+1]) (duplicates merged).  Output = the packed dataset layout K0 consumes:
 *   gcs_link_pairs_offsets: node_off[n_pairs + 1] int64; *status_dev bit 0 = a chain id out of range.
 *   gcs_link_pairs with col == NULL: rowptr[n_rows + 1] int64 (n_rows = node_off[n_pairs]); with col != NULL: fills
 *     col[nnz] int32 pair-local ids, ascending per row.  *status_dev bit 1 = a bridge position outside its chain
 *     (networkx would silently add a new node; here it is an error).
 * --------------------------------------------------------------------------------- */
int64_t gcs_contact_workspace_bytes(int64_t n_rows);
int gcs_contact_map_rowptr(const float* ca, const int32_t* chain_ptr, int32_t n_chains, int64_t n_residues,
                           float angstroms, int64_t* rowptr, void* workspace, int64_t workspace_bytes,
                           gcs_stream stream);
int gcs_contact_map_fill(const float* ca, const int32_t* chain_ptr, int32_t n_chains, int64_t n_residues,
                         float angstroms, const int64_t* rowptr, int32_t* col, float* dist, gcs_stream stream);
int gcs_link_pairs_offsets(const int32_t* chain_ptr, int32_t n_chains, const int32_t* pair_a, const int32_t* pair_b,
                           int32_t n_pairs, int64_t* node_off, int32_t* status_dev, void* workspace,
                           int64_t workspace_bytes, gcs_stream stream);
int gcs_link_pairs(const int64_t* chain_rowptr, const int32_t* chain_col, const int32_t* chain_ptr,
                   const int32_t* pair_a, const int32_t* pair_b, int32_t n_pairs, const int32_t* bridge_ptr,
                   const int32_t* bridge_a, const int32_t* bridge_b, const int64_t* node_off, int64_t n_rows,
                   int64_t* rowptr, int32_t* col, int32_t* status_dev, void* workspace, int64_t workspace_bytes,
                   gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * K10  Fused multi-tensor optimizer steps over the flat parameter buffer.
 *   sgd:  w -= lr * (g * grad_scale)          (tf.keras.optimizers.SGD, gcn.py:325,338)
 *   adam: Keras Adam, lr_t = lr*sqrt(1-b2^t)/(1-b1^t), w -= lr_t*m/(sqrt(v)+eps)
 * The _ex forms add Keras' options; with every option off they run the same kernel as the plain entry points.
 *   gcs_sgd_step_ex:  momentum in [0, 1] (slot accum, NULL allowed only for momentum 0, which is plain SGD):
 *                     accum = momentum*accum - lr*g; w += accum, or with nesterov w += momentum*accum - lr*g.
 *   gcs_adam_step_ex: vhat != NULL is amsgrad: vhat = max(vhat, v), w -= lr_t*m/(sqrt(vhat)+eps).
 *   clip (NULL: none) acts on g*grad_scale: GCS_CLIP_VALUE clamps each element to [-clipvalue, clipvalue] (NaN stays
 *   NaN); then GCS_CLIP_NORM (per tensor) or GCS_CLIP_GLOBAL_NORM (all tensors) scales by clipnorm/||g|| where
 *   ||g|| > clipnorm and by exactly 1 otherwise; a non-finite global norm gives NaN everywhere.
 *   The norms come from a chunk table over the buffer: `chunks` is device int64 [n_chunks][4] = {begin, end, lo, hi},
 *   element range [begin, end) of w / g (no chunk crosses a tensor), and [lo, hi) the indices in `partials` of the
 *   chunks of the same tensor.  Row k of a call writes its fp64 sum of squares to partials[chunk_base + k]; the global
 *   norm sums partials[0, n_partials).  A norm-clipped step is two launches (one block per chunk each): the norm pass,
 *   then the update, whose blocks each form their factor from the partials in a fixed order.  No atomics: the step is
 *   bit-identical from run to run.  GCS_CLIP_PARTIALS_READY skips the norm pass when gcs_grad_clip_partials already
 *   wrote this step's partials (tensors that are not one buffer: every tensor's pass first, then every update).
 * --------------------------------------------------------------------------------- */
int gcs_sgd_step(float* w, const float* g, int64_t n, float lr, float grad_scale, gcs_stream stream);
int gcs_adam_step(float* w, const float* g, float* m, float* v, int64_t n, double lr, double beta1,
                  double beta2, double eps, int64_t step, float grad_scale, gcs_stream stream);

enum gcs_clip_mode {
  GCS_CLIP_VALUE = 1,
  GCS_CLIP_NORM = 2,
  GCS_CLIP_GLOBAL_NORM = 4,
  GCS_CLIP_PARTIALS_READY = 8
};
typedef struct gcs_grad_clip {
  int32_t mode;            /* gcs_clip_mode bits; NORM and GLOBAL_NORM exclude each other */
  float clipvalue;         /* >= 0 */
  float clipnorm;          /* >= 0, the threshold of NORM or GLOBAL_NORM */
  int32_t n_chunks;        /* rows of `chunks` this call covers (NORM / GLOBAL_NORM) */
  const int64_t* chunks;   /* device [n_chunks][4] */
  double* partials;        /* device [n_partials] */
  int32_t chunk_base;
  int32_t n_partials;
} gcs_grad_clip;

int gcs_sgd_step_ex(float* w, const float* g, float* accum, int64_t n, float lr, float momentum, int32_t nesterov,
                    float grad_scale, const gcs_grad_clip* clip, gcs_stream stream);
int gcs_adam_step_ex(float* w, const float* g, float* m, float* v, float* vhat, int64_t n, double lr, double beta1,
                     double beta2, double eps, int64_t step, float grad_scale, const gcs_grad_clip* clip,
                     gcs_stream stream);
/* The norm pass alone: partials[chunk_base + k] = sum of squares of clipvalue(g*grad_scale) over row k. */
int gcs_grad_clip_partials(const float* g, int64_t n, float grad_scale, const gcs_grad_clip* clip,
                           gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * C1  Data-parallel collective (SURVEY.md 8b / 8e; the reference is single-process, this is the sharding the north star
 * asks for).  Graphs shard across the GPUs of a node, every rank runs gcs_model_train_step with grad_scale =
 * 1 / global_batch on its shard, then ONE SUM all-reduce of the flat gradient buffer (NCCL over NVLink / NVSwitch) and the
 * fused optimizer step - identical parameters on every rank.  NCCL is bound at run time (dlopen libnccl.so.2).
 *   gcs_comm_unique_id: rank 0 fills 128 bytes (ncclUniqueId) and hands them to the other ranks by any host channel.
 *   gcs_comm_init:      collective; binds to the calling thread's current device.  One communicator per (process, GPU).
 *   gcs_allreduce_grads / gcs_allreduce_f64: in place, enqueued on `stream`; f64 is what a synchronised-BatchNorm
 *                       hook (gcs_set_allreduce_hook) forwards its statistics through.
 * --------------------------------------------------------------------------------- */
typedef struct gcs_comm gcs_comm;
int gcs_comm_unique_id(void* id_host_128_bytes);
int gcs_comm_init(const void* id_host_128_bytes, int32_t rank, int32_t world_size, gcs_comm** comm);
int gcs_comm_destroy(gcs_comm* comm);
int gcs_comm_rank(const gcs_comm* comm);
int gcs_comm_world_size(const gcs_comm* comm);
int gcs_allreduce_grads(gcs_comm* comm, float* grads, int64_t n, gcs_stream stream);
int gcs_allreduce_f64(gcs_comm* comm, double* buf, int64_t n, gcs_stream stream);

/* ---------------------------------------------------------------------------------
 * Whole-model entry points: spektral.models.GeneralGNN.__call__ (gcn.py:334 training,
 * :351 inference) and the GradientTape backward of gcn.py:333-337.
 * --------------------------------------------------------------------------------- */
typedef struct gcs_model_config {
  int32_t in_features;      /* F */
  int32_t output;           /* classes C */
  int32_t hidden;           /* H (default 256) */
  int32_t message_passing;  /* L (default 4) */
  int32_t pre_process;      /* default 2 */
  int32_t post_process;     /* default 2 */
  int32_t connectivity;     /* 0 = None (out = z), 1 = 'cat' (out = concat[z, out]), 2 = 'sum' (out = z + out) */
  int32_t pool;             /* 0 = None (node-level output), 1 = 'sum', 2 = 'avg', 3 = 'attn_sum' (adds the trainable
                               attn_kernel [H*(L+1) or H] after the last post block) */
  int32_t final_activation; /* 0 = linear, 1 = softmax (C <= 64), 2 = sigmoid (any C) */
  float bn_momentum;        /* 0.99 */
  float bn_epsilon;         /* 1e-3 */
  int32_t aggregate;        /* GeneralConv aggregate: 0 = 'sum' (the reference's), 1 = 'mean', 2 = 'max' */
  int32_t loss;             /* loss of the fused train steps: 0 = the head's own (categorical cross-entropy for softmax,
                               binary cross-entropy for sigmoid, MSE for linear); 1 = MSE, 2 = MAE, 3 = Huber, with
                               final_activation = 0 only.  Does not change the parameter or workspace layout. */
  float huber_delta;        /* Huber's delta when loss = 3: finite and > 0 */
} gcs_model_config;

/* Keras Dropout(rate) between the BatchNorm and the activation of every dense block, the last post block included (it
 * acts on the logits), for ONE training-mode call: the `_ex` entry points below take it as their last argument (NULL, or
 * rate 0: no dropout; the entry points without `_ex` are these with NULL).  Inference ignores it.  0 <= rate < 1;
 * anything else, NaN included, is GCS_ERR_INVALID_ARGUMENT.  The keep mask is a function of (seed, step, block, row,
 * column) only (format: csrc/dropout.cuh), so a training-mode gcs_model_forward_ex and the gcs_model_backward_ex that
 * follows it regenerate the same masks when they pass the same struct.  Each training step should pass a new step
 * value.  No extra workspace: the workspace sizes above hold. */
typedef struct gcs_dropout {
  float rate;
  uint32_t _pad;
  uint64_t seed;            /* key of the mask stream */
  uint64_t step;            /* training step (its low 32 bits enter the mask counter) */
} gcs_dropout;

typedef struct gcs_batch {
  int64_t n_nodes;
  int64_t nnz;
  int32_t n_graphs;
  int32_t rb_height;        /* row-block height of rb4_* below: 2 or 4 (0 = 4) */
  const int32_t* rowptr;    /* [N+1]  CSR of pattern(A): row = target, col = source */
  const int32_t* colidx;    /* [nnz] */
  const int32_t* rowptr_t;  /* CSR of pattern(A)^T; may equal rowptr/colidx if symmetric; */
  const int32_t* colidx_t;  /*   only read by the backward */
  const int32_t* graph_ptr; /* [B+1] */
  const float* x;           /* [N, F] */
  int64_t ldx;
  const float* y;           /* [B, C] one-hot ([N, C] node labels when pool == 0); NULL for inference */
  const int64_t* seg_ids;       /* [N] graph id of every node (Spektral's i); needed by the pooled backward */
  const int32_t* rb4_blk_ptr;   /* row-block form of pattern(A) (gcs_spmm_build_rb, height rb_height), or NULL */
  const uint32_t* rb4_ent;
  const int32_t* rb4_blk_ptr_t; /* RB4 form of pattern(A)^T; may alias when symmetric; backward only */
  const uint32_t* rb4_ent_t;
  int32_t max_graph_nodes;      /* longest graph of the batch (host-known), 0 = unknown: selects the shared-memory slab */
  int32_t reserved;             /*   aggregation kernel (gcs_spmm_sum_graphs) when graph_ptr is set */
  const float* values;          /* optional per-entry weights w_ij in CSR order (the `use_edge_data` switch of gcn.py:73-80);
                                   NULL = pattern only, as GeneralConv aggregates */
  const float* values_t;        /* the same weights in the order of (rowptr_t, colidx_t); backward only */
  const float* sample_weight;   /* [rows_post] one loss weight per output row (per graph, or per node when pool == 0),
                                   read by the train steps (gcs_weighted_loss); NULL = unweighted.  The workspace must
                                   then be sized with GCS_WORKSPACE_SAMPLE_WEIGHTS.  gcs_model_forward ignores it. */
} gcs_batch;

/* Number of floats in the flat trainable / state buffers (layout: gcn-string_b200/params.py). */
int64_t gcs_model_num_params(const gcs_model_config* cfg);
int64_t gcs_model_num_state(const gcs_model_config* cfg);
int64_t gcs_model_workspace_bytes(const gcs_model_config* cfg, int64_t n_nodes, int64_t nnz,
                                  int32_t n_graphs, int32_t training);
/* The same with flags: GCS_WORKSPACE_SAMPLE_WEIGHTS sizes the plan for a batch with sample_weight set.  Only the last
 * slot of the plan (the loss partials) grows, so every other offset - gcs_model_logits_offset included - is the
 * unweighted plan's.  flags = 0 is gcs_model_workspace_bytes; unknown bits give -1. */
#define GCS_WORKSPACE_SAMPLE_WEIGHTS 1
int64_t gcs_model_workspace_bytes_ex(const gcs_model_config* cfg, int64_t n_nodes, int64_t nnz, int32_t n_graphs,
                                     int32_t training, int32_t flags);
/* Inference / training-mode forward.  out: [B, C] (or [N, C] when pool == 0), after the final activation.  With
 * training != 0 BatchNorm uses batch statistics and updates `state` in place. */
int gcs_model_forward(const gcs_model_config* cfg, const float* params, float* state,
                      const gcs_batch* batch, int32_t training, float* out, void* workspace,
                      int64_t workspace_bytes, gcs_stream stream);
/* Training-mode forward + backward.  grads: flat, same layout as params (overwritten).
 * loss_acc[2] = {mean categorical cross-entropy over this batch, accuracy}; probs [B,C] ([N,C] when pool == 0: the
 * loss is then the mean over nodes).  grad_scale multiplies dLoss (1/B - 1/N node-level - reproduces the reference; use
 * 1/global_B or 1/global_N when the gradients are then summed across data-parallel ranks).  The loss runs through
 * gcs_softmax_xent_ws; gcs_model_workspace_bytes includes its workspace.  With final_activation = 2 (sigmoid) the loss
 * is binary cross-entropy through gcs_sigmoid_bce instead: probs = sigmoid(logits), loss_acc = {mean binary
 * cross-entropy, binary accuracy}, and grad_scale keeps its meaning (the 1/C of the per-row mean is applied inside).
 * With final_activation = 0 (linear) the loss is the regression loss cfg->loss selects (0 or 1 = MSE, 2 = MAE, 3 =
 * Huber with cfg->huber_delta) through gcs_regression_loss: probs = the predictions (the logits), loss_acc = {mean
 * loss, mean absolute error}, and grad_scale keeps its meaning the same way.  With batch->sample_weight set, every head
 * runs through gcs_weighted_loss instead (loss = sum w l / rows, the weighted mean metric, dlogits scaled per row), and
 * the workspace must be gcs_model_workspace_bytes_ex(..., GCS_WORKSPACE_SAMPLE_WEIGHTS) bytes: with less the call
 * fails with GCS_ERR_WORKSPACE. */
int gcs_model_train_step(const gcs_model_config* cfg, const float* params, float* state,
                         const gcs_batch* batch, float grad_scale, float* grads, float* probs,
                         float* loss_acc, void* workspace, int64_t workspace_bytes,
                         gcs_stream stream);

/* The train step of one data-parallel rank: gcs_model_train_step with grad_scale = 1 / global_batch, plus the SUM
 * all-reduce of `grads` over `comm`, issued on comm_stream in three buckets as the backward finishes trailing ranges of
 * the flat gradient buffer (post-MLP + last GeneralConv layers first), so that the reduction of all but the last bucket
 * overlaps the rest of the backward.  `stream` is made to wait for the reductions before anything enqueued after this
 * call (the optimizer step) runs.  sync_batchnorm != 0: the BatchNorm statistics of this call are all-reduced over
 * `comm` as well (fp64 sums, on `stream`) - the step then equals ONE single-device step on the union of the shards;
 * no hook needs to be installed for that (the library's state is per call). */
int gcs_model_train_step_dp(const gcs_model_config* cfg, const float* params, float* state,
                            const gcs_batch* batch, float grad_scale, float* grads, float* probs,
                            float* loss_acc, void* workspace, int64_t workspace_bytes, gcs_stream stream,
                            gcs_comm* comm, gcs_stream comm_stream, int32_t sync_batchnorm);

/* Split form of the train step, for callers that compute the loss themselves (the
 * GradientTape pattern of gcn.py:333-337): gcs_model_forward(training=1) leaves the
 * logits (pre-softmax BatchNorm output, [B, C]) at byte offset gcs_model_logits_offset()
 * inside the workspace together with the saved activations; gcs_model_backward then takes
 * dLoss/dlogits and fills `grads`.  Same workspace, same batch, nothing in between. */
int64_t gcs_model_logits_offset(const gcs_model_config* cfg, int64_t n_nodes, int32_t n_graphs,
                                int32_t training);
int gcs_model_backward(const gcs_model_config* cfg, const float* params, const gcs_batch* batch,
                       const float* dlogits, float* grads, void* workspace, int64_t workspace_bytes,
                       gcs_stream stream);
/* The four model entry points above with the dropout of the call (gcs_dropout; NULL = none). */
int gcs_model_forward_ex(const gcs_model_config* cfg, const float* params, float* state, const gcs_batch* batch,
                         int32_t training, float* out, void* workspace, int64_t workspace_bytes, gcs_stream stream,
                         const gcs_dropout* dropout);
int gcs_model_train_step_ex(const gcs_model_config* cfg, const float* params, float* state, const gcs_batch* batch,
                            float grad_scale, float* grads, float* probs, float* loss_acc, void* workspace,
                            int64_t workspace_bytes, gcs_stream stream, const gcs_dropout* dropout);
int gcs_model_train_step_dp_ex(const gcs_model_config* cfg, const float* params, float* state, const gcs_batch* batch,
                               float grad_scale, float* grads, float* probs, float* loss_acc, void* workspace,
                               int64_t workspace_bytes, gcs_stream stream, gcs_comm* comm, gcs_stream comm_stream,
                               int32_t sync_batchnorm, const gcs_dropout* dropout);
int gcs_model_backward_ex(const gcs_model_config* cfg, const float* params, const gcs_batch* batch,
                          const float* dlogits, float* grads, void* workspace, int64_t workspace_bytes,
                          gcs_stream stream, const gcs_dropout* dropout);

/* Attributions: gradients with respect to the model's inputs, the saliency pattern of
 *   with tf.GradientTape() as tape: tape.watch(x); pred = model([x, a, i], training=False)
 *   tape.gradient(pred, [x, a.values], output_gradients=...)
 * gcs_model_forward_attr: the inference forward (moving statistics, no dropout, no moving-statistics update) on a
 * training-mode workspace (gcs_model_workspace_bytes(..., training = 1)), every dense block unfused so that the
 * activations stay there for gcs_model_input_grad.  Its `out` equals gcs_model_forward(training = 0) to float32
 * rounding (the plain inference path folds BatchNorm into the GEMM).
 * gcs_model_input_grad: the reverse pass from dlogits [rows_out, C] after either forward, same workspace and batch
 * (with the transposed CSR):
 *   training = 0 (after gcs_model_forward_attr): BatchNorm on the moving statistics; grads must be NULL
 *                (parameter gradients of an inference-mode call are not built: GCS_ERR_UNSUPPORTED);
 *   training = 1 (after gcs_model_forward_ex(training = 1) with the same `dropout`): the parameter gradients into grads
 *                (required) exactly as gcs_model_backward_ex computes them.
 *   dx      [n_nodes, in_features] (ld lddx), optional: dLoss/dx;
 *   dvalues [nnz], optional, only with batch->values: dLoss/d(edge weights) in forward CSR order, the L GeneralConv
 *           layers summed in a fixed order (gcs_spmm_edge_grad).
 * gcs_output_grad: dlogits = J^T dprobs of the head's activation on its output probs [rows, C] - softmax
 * p * (d - p . d), sigmoid d * p (1 - p), linear d - for a gradient of the model output itself (output_gradients). */
int gcs_model_forward_attr(const gcs_model_config* cfg, const float* params, float* state, const gcs_batch* batch,
                           float* out, void* workspace, int64_t workspace_bytes, gcs_stream stream);
int gcs_model_input_grad(const gcs_model_config* cfg, const float* params, const gcs_batch* batch, int32_t training,
                         const float* dlogits, float* dx, int64_t lddx, float* dvalues, float* grads, void* workspace,
                         int64_t workspace_bytes, gcs_stream stream, const gcs_dropout* dropout);
int gcs_output_grad(int32_t final_activation, const float* probs, const float* dprobs, int64_t rows, int32_t C,
                    float* dlogits, gcs_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* GCNSTRING_B200_H */
