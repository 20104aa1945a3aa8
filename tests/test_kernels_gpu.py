"""GPU parity, kernel by kernel, through the C ABI (gcn_string_b200.ops -> ctypes) against
the CPU oracle on the same seeded inputs.  Integer / index outputs must be bit-exact;
floating point within 1e-5 relative (max-abs error over max-abs reference, fp32)."""
import numpy as np
import pytest
import scipy.sparse as sp

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import _lib, ops, synthetic
from oracle import batching_ref, model_ref_np as O1

from conftest import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def host(t):
    return t.detach().cpu().numpy()


def random_csr(rng, n, density, symmetric=False):
    d = rng.random((n, n)) < density
    if symmetric:
        d = d | d.T
    a = sp.csr_matrix(d.astype(np.int64))
    a.sort_indices()
    return a


# ---------------------------------------------------------------- K0 batching (bit-exact)
@pytest.mark.parametrize("n_graphs,n_mean,deg,F", [(8, 60, 8, 12), (33, 40, 6, 5), (1, 30, 4, 3)])
def test_batch_disjoint_matches_scipy_collate(n_graphs, n_mean, deg, F):
    ds = synthetic.make_dataset(n_graphs, seed=5, n_mean=n_mean, deg=deg, n_feat=F)
    store = g.data.DeviceGraphStore(ds)
    rng = np.random.default_rng(1)
    for ids in (np.arange(n_graphs), rng.permutation(n_graphs)[: max(1, n_graphs // 2)]):
        ids = ids.astype(np.int64)
        x, a, seg, y = store.batch(dev(ids), ids, want_coo=True)
        (xr, (idx, _vals, shape), segr), yr = batching_ref.collate([ds.graph(int(k)) for k in ids])
        rowptr, colidx, deg_ = batching_ref.derived_csr(idx, xr.shape[0])
        assert int(a.status.item()) == 0
        assert np.array_equal(host(a.indices), idx) and a.indices.dtype == torch.int64
        assert np.array_equal(host(seg), segr) and seg.dtype == torch.int64
        assert np.array_equal(host(a.rowptr), rowptr) and np.array_equal(host(a.colidx), colidx)
        assert np.array_equal(host(a.graph_ptr), batching_ref.graph_ptr(segr, len(ids)))
        assert np.array_equal(np.diff(host(a.rowptr)), deg_)
        assert np.array_equal(host(x), xr.astype(np.float32)) and np.array_equal(host(y), yr.astype(np.float32))
        assert a.dense_shape == tuple(shape) and a.max_graph_nodes == int(ds.n_nodes[ids].max())


def test_batch_disjoint_ragged_graphs_and_size_check():
    rng = np.random.default_rng(2)
    graphs = []
    for n in (1, 7, 1, 19, 3):                          # single-node graphs, an edgeless graph
        a = random_csr(rng, n, 0.0 if n == 3 else 0.35)
        graphs.append(g.Graph(x=rng.random((n, 4)), a=a, y=np.array([0, 1])))
    packed = synthetic.pack_graphs(graphs)
    store = g.data.DeviceGraphStore(packed)
    ids = np.arange(5, dtype=np.int64)
    x, a, seg, y = store.batch(dev(ids), ids, want_coo=True)
    (xr, (idx, _, _), segr), _ = batching_ref.collate([(gr.x, gr.a, gr.y) for gr in graphs])
    assert np.array_equal(host(a.indices), idx) and np.array_equal(host(seg), segr)
    assert host(a.rowptr)[-1] == idx.shape[0]
    # wrong totals are detected on the device
    lib = _lib.load()
    n, nnz = int(packed.n_nodes.sum()), int(packed.n_edges.sum())
    i32 = dict(dtype=torch.int32, device="cuda")
    bufs = [torch.empty(6, **i32), torch.empty(6, **i32), torch.empty(n + 2, **i32), torch.empty(nnz + 1, **i32)]
    xo = torch.empty(n + 1, 4, device="cuda")
    so = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    flag = torch.zeros(1, **i32)
    st = lib.gcs_batch_disjoint(store.node_off.data_ptr(), store.rowptr.data_ptr(), store.col.data_ptr(),
                                store.x.data_ptr(), store.y.data_ptr(), 4, 2, dev(ids).data_ptr(), 5, n + 1, nnz,
                                *[b.data_ptr() for b in bufs], xo.data_ptr(), so.data_ptr(), None, None,
                                flag.data_ptr(), _lib.stream_ptr())
    assert st == 0 and int(flag.item()) == 1


def test_coo_to_csr_and_segment_ptr_validate():
    rng = np.random.default_rng(3)
    a = random_csr(rng, 50, 0.1)
    r, c, _ = sp.find(a)
    idx = np.stack([r, c], 1).astype(np.int64)
    idx = idx[np.lexsort((idx[:, 1], idx[:, 0]))]
    rowptr, colidx = ops.coo_to_csr(dev(idx), 50)
    assert np.array_equal(host(rowptr), a.indptr) and np.array_equal(host(colidx), a.indices)
    with pytest.raises(ValueError, match="row-major"):
        ops.coo_to_csr(dev(idx[::-1].copy()), 50)
    rp0, ci0 = ops.coo_to_csr(torch.zeros(0, 2, dtype=torch.int64, device="cuda"), 4)   # empty adjacency
    assert host(rp0).tolist() == [0] * 5 and ci0.numel() == 0
    seg = np.repeat(np.arange(6), [3, 0, 4, 1, 0, 2]).astype(np.int64)      # empty segments
    assert host(ops.segment_ptr(dev(seg), 6)).tolist() == [0, 3, 3, 7, 8, 8, 10]
    with pytest.raises(ValueError, match="sorted"):
        ops.segment_ptr(dev(seg[::-1].copy()), 6)


def test_transpose_and_symmetry():
    rng = np.random.default_rng(4)
    a = random_csr(rng, 200, 0.05)
    rp, ci = dev(a.indptr.astype(np.int32)), dev(a.indices.astype(np.int32))
    assert ops.csr_is_symmetric(rp, ci) is False
    rpt, cit = ops.csr_transpose(rp, ci)
    at = sp.csr_matrix(a.T)
    at.sort_indices()
    assert np.array_equal(host(rpt), at.indptr) and np.array_equal(host(cit), at.indices)
    s = random_csr(rng, 200, 0.03, symmetric=True)
    assert ops.csr_is_symmetric(dev(s.indptr.astype(np.int32)), dev(s.indices.astype(np.int32))) is True


def test_cast_f64():
    x = np.random.default_rng(0).standard_normal((37, 5))
    assert np.array_equal(host(ops.cast_f64_f32(dev(x))), x.astype(np.float32))


# ---------------------------------------------------------------- K1/K9 dense
@pytest.mark.parametrize("M,K,N", [(300, 32, 256), (1000, 768, 256), (257, 5, 8), (64, 256, 2), (129, 130, 6),
                                   (4096, 1280, 256)])
def test_linear_forward_and_gradients(M, K, N):
    rng = np.random.default_rng(M + K + N)
    A = rng.standard_normal((M, K)).astype(np.float32)
    W = (rng.standard_normal((K, N)) / np.sqrt(K)).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    dH = rng.standard_normal((M, N)).astype(np.float32)
    A64, W64, dH64 = A.astype(np.float64), W.astype(np.float64), dH.astype(np.float64)
    assert rel_err(host(ops.linear_fwd(dev(A), dev(W), dev(b))), A64 @ W64 + b) < TOL
    dW, db = ops.linear_bwd_weight(dev(A), dev(dH))
    assert rel_err(host(dW), A64.T @ dH64) < TOL and rel_err(host(db), dH64.sum(0)) < TOL
    assert rel_err(host(ops.linear_bwd_input(dev(dH), dev(W))), dH64 @ W64.T) < TOL
    base = rng.standard_normal((M, K)).astype(np.float32)
    acc = ops.linear_bwd_input(dev(dH), dev(W), out=dev(base), accumulate=True)
    assert rel_err(host(acc), base + dH64 @ W64.T) < TOL


@pytest.mark.parametrize("M,K,N", [(1, 256, 128), (255, 128, 256), (256, 512, 512), (257, 384, 128), (511, 2048, 256),
                                   (33000, 1024, 256)])
def test_tensor_core_gemms_forced(M, K, N):
    """The tcgen05 kernels with the FFMA fallback disabled (mode 2 raises when the shape is not eligible): ragged row
    counts around the 256-row CTA-pair tile, reductions chunked at 768, N = 128 / 512, both weight-gradient kernels
    (CTA pair when K % 256 == 0, one CTA otherwise), strided operands, accumulate, run-to-run determinism."""
    lib = _lib.load()
    rng = np.random.default_rng(M * 7 + K + N)
    wideA = rng.standard_normal((M, K + 64)).astype(np.float32)
    A = wideA[:, 32:32 + K]                                  # lda = K + 64, 128-byte aligned start
    W = (rng.standard_normal((K, N)) / np.sqrt(K)).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    dH = rng.standard_normal((M, N)).astype(np.float32)
    A64, W64, dH64 = A.astype(np.float64), W.astype(np.float64), dH.astype(np.float64)
    dA = dev(wideA)[:, 32:32 + K]
    try:
        lib.gcs_debug_set_gemm_mode(2)
        out = torch.zeros(M, N + 128, device="cuda")
        y = ops.linear_fwd(dA, dev(W), dev(b), out=out[:, 128:])          # ldc = N + 128
        assert rel_err(host(y), A64 @ W64 + b) < TOL and float(out[:, :128].abs().max()) == 0.0
        y2 = ops.linear_fwd(dA, dev(W), dev(b))
        assert torch.equal(y2, y.contiguous())                              # deterministic, layout-independent
        dW, _ = ops.linear_bwd_weight(dA, dev(dH), want_db=False)
        assert rel_err(host(dW), A64.T @ dH64) < TOL
        dW2, _ = ops.linear_bwd_weight(dA, dev(dH), want_db=False)
        assert torch.equal(dW, dW2)
        base = rng.standard_normal((M, K)).astype(np.float32)
        acc = ops.linear_bwd_input(dev(dH), dev(W), out=dev(base), accumulate=True)
        assert rel_err(host(acc), base + dH64 @ W64.T) < TOL
        assert rel_err(host(ops.linear_bwd_input(dev(dH), dev(W))), dH64 @ W64.T) < TOL
    finally:
        lib.gcs_debug_set_gemm_mode(0)


@pytest.mark.parametrize("M,K,N", [(1, 256, 128), (255, 128, 256), (257, 384, 128), (511, 2048, 256), (33000, 1280, 256)])
@pytest.mark.parametrize("scaling", ["unit", "tiny", "huge", "spread"])
def test_fp16_split_tensor_core_gemm(M, K, N, scaling):
    """linear_tc_pair_kernel<true> (3 kind::f16 MMAs per product on fp16 hi / 2^11-scaled lo operands, power-of-two
    operand scales from the |max|) through the standalone ops in debug mode 2: fp32-level accuracy against float64 for
    unit-scale operands, for operands far outside fp16's exponent range (gradients ~1e-9, activations ~3e4) and for a
    2^24 spread inside one operand; ragged rows, strided operands, chunked reductions, accumulate, determinism."""
    lib = _lib.load()
    rng = np.random.default_rng(M + K + N + len(scaling))
    a_mag, w_mag = {"unit": (1.0, 1.0), "tiny": (1e-9, 1e-4), "huge": (3e4, 50.0), "spread": (1.0, 1.0)}[scaling]
    wideA = (rng.standard_normal((M, K + 64)) * a_mag).astype(np.float32)
    if scaling == "spread":
        wideA *= np.exp2(-rng.integers(0, 25, wideA.shape)).astype(np.float32)
    A = wideA[:, 32:32 + K]
    W = (rng.standard_normal((K, N)) / np.sqrt(K) * w_mag).astype(np.float32)
    b = (rng.standard_normal(N) * a_mag * w_mag).astype(np.float32)
    dH = (rng.standard_normal((M, N)) * a_mag).astype(np.float32)
    A64, W64, dH64 = A.astype(np.float64), W.astype(np.float64), dH.astype(np.float64)
    dA = dev(wideA)[:, 32:32 + K]
    try:
        lib.gcs_debug_set_param(7, 2)
        lib.gcs_debug_set_gemm_mode(2)
        out = torch.zeros(M, N + 128, device="cuda")
        y = ops.linear_fwd(dA, dev(W), dev(b), out=out[:, 128:])
        assert rel_err(host(y), A64 @ W64 + b) < TOL and float(out[:, :128].abs().max()) == 0.0
        assert torch.equal(ops.linear_fwd(dA, dev(W), dev(b)), y.contiguous())
        base = (rng.standard_normal((M, K)) * a_mag * w_mag).astype(np.float32)
        acc = ops.linear_bwd_input(dev(dH), dev(W), out=dev(base), accumulate=True)
        assert rel_err(host(acc), base + dH64 @ W64.T) < TOL
        if K % 256 == 0:                                                    # weight gradient: the fp16 CTA-pair kernel
            dW, _ = ops.linear_bwd_weight(dA, dev(dH), want_db=False)
            assert rel_err(host(dW), A64.T @ dH64) < TOL
            dW2, _ = ops.linear_bwd_weight(dA, dev(dH), want_db=False)
            assert torch.equal(dW, dW2)
        lib.gcs_debug_set_param(7, 0)                                       # the tf32 kernel on the same operands
        y_tf32 = ops.linear_fwd(dA, dev(W), dev(b))
        assert rel_err(host(y_tf32), A64 @ W64 + b) < TOL
    finally:
        lib.gcs_debug_set_gemm_mode(0)
        lib.gcs_debug_set_param(7, 1)
    # all-zero operand: the scale falls back to 1
    try:
        lib.gcs_debug_set_param(7, 2)
        lib.gcs_debug_set_gemm_mode(2)
        z = ops.linear_fwd(torch.zeros(M, K, device="cuda"), dev(W), dev(b))
        assert rel_err(host(z), np.broadcast_to(b, (M, N))) < TOL
    finally:
        lib.gcs_debug_set_gemm_mode(0)
        lib.gcs_debug_set_param(7, 1)


@pytest.mark.parametrize("M,K,N", [(4096, 32, 256), (9001, 16, 256), (5003, 4, 64), (7000, 28, 200), (33333, 12, 512)])
def test_linear_weight_gradient_thin_first_layer(M, K, N):
    """dW of a thin layer (K <= 32: the first Dense of the pre-processing MLP, F = 16 in the reference's data, 32 in
    BASELINE.json) runs on its own split-row FFMA kernel; against float64, on a strided dH view, and run-to-run
    bit-identical (fixed summation order)."""
    rng = np.random.default_rng(M + K)
    a = rng.standard_normal((M, K)).astype(np.float32)
    wide = rng.standard_normal((M, N + 8)).astype(np.float32)
    dh = dev(wide)[:, 4:4 + N]
    dw, db = ops.linear_bwd_weight(dev(a), dh)
    ref = a.astype(np.float64).T @ wide[:, 4:4 + N].astype(np.float64)
    assert rel_err(host(dw), ref) < TOL
    assert rel_err(host(db), wide[:, 4:4 + N].astype(np.float64).sum(0)) < TOL
    dw2, _ = ops.linear_bwd_weight(dev(a), dh)
    assert torch.equal(dw, dw2)


def test_linear_on_strided_views_of_the_concat_buffer():
    rng = np.random.default_rng(9)
    cat = dev(rng.standard_normal((500, 5 * 64)).astype(np.float32))
    W = (rng.standard_normal((128, 64)) / 11).astype(np.float32)
    view = cat[:, 192:]                                  # trailing 2*H columns, ld = 5*H
    out = ops.linear_fwd(view, dev(W))
    assert rel_err(host(out), host(view).astype(np.float64) @ W) < TOL
    dst = torch.zeros(500, 5 * 64, device="cuda")
    ops.linear_fwd(view, dev(W), out=dst[:, 64:128])
    assert np.array_equal(host(dst[:, 64:128]), host(out)) and float(dst[:, :64].abs().max()) == 0.0


# ---------------------------------------------------------------- K2/K8 BatchNorm + PReLU
@pytest.mark.parametrize("M,C", [(1000, 256), (37, 10), (6, 2), (70000, 64)])
def test_batchnorm_prelu_forward_backward(M, C):
    rng = np.random.default_rng(M + C)
    h = (rng.standard_normal((M, C)) * rng.uniform(0.5, 3, C) + rng.uniform(-5, 5, C)).astype(np.float32)
    gamma = rng.uniform(0.5, 1.5, C).astype(np.float32)
    beta = rng.normal(0, 0.3, C).astype(np.float32)
    alpha = rng.uniform(0.05, 0.4, C).astype(np.float32)
    mm = rng.normal(0, 1, C).astype(np.float32)
    mv = rng.uniform(0.5, 2, C).astype(np.float32)
    da = rng.standard_normal((M, C)).astype(np.float32)
    h64 = h.astype(np.float64)
    mean, var = ops.bn_stats(dev(h))
    mean_r, var_r = h64.mean(0), ((h64 - h64.mean(0)) ** 2).mean(0)
    assert rel_err(host(mean), mean_r) < TOL and rel_err(host(var), var_r) < TOL
    mmd, mvd = dev(mm), dev(mv)
    scale, shift = ops.bn_fold(mean, var, dev(gamma), dev(beta), 1e-3, 0.99, mmd, mvd)
    inv = gamma / np.sqrt(var_r + 1e-3)
    assert rel_err(host(scale), inv) < TOL and rel_err(host(shift), beta - mean_r * inv) < TOL
    assert rel_err(host(mmd), mm - (mm - mean_r) * 0.01) < TOL and rel_err(host(mvd), mv - (mv - var_r) * 0.01) < TOL
    z = h64 * inv + (beta - mean_r * inv)
    out = ops.bn_prelu_fwd(dev(h), scale, shift, dev(alpha))
    assert rel_err(host(out), np.where(z > 0, z, alpha * z)) < TOL
    assert rel_err(host(ops.bn_prelu_fwd(dev(h), scale, shift, None)), z) < TOL
    # backward against the oracle's block backward
    dh, dgamma, dbeta, dalpha = ops.bn_prelu_bwd(dev(da), dev(h), mean, var, dev(gamma), dev(beta), dev(alpha))
    slope = np.where(z > 0, 1.0, np.where(z < 0, alpha, 0.0))
    dz = da * slope
    rstd = 1 / np.sqrt(var_r + 1e-3)
    xhat = (h64 - mean_r) * rstd
    dg_r, db_r = (dz * xhat).sum(0), dz.sum(0)
    dh_r = gamma * rstd * (dz - db_r / M - xhat * dg_r / M)
    near_kink = np.abs(z) < 1e-5                           # fp32 may take the other PReLU branch there
    assert rel_err(host(dgamma), dg_r) < 5 * TOL and rel_err(host(dbeta), db_r) < 5 * TOL
    assert rel_err(host(dalpha), (da * np.minimum(z, 0)).sum(0)) < TOL
    assert rel_err(np.where(near_kink, 0, host(dh)), np.where(near_kink, 0, dh_r)) < 5 * TOL
    # the fused bias gradient: column sums of the dh the kernel wrote (mathematically zero after BatchNorm;
    # the check is against the fp64 sum of the kernel's own fp32 dh, on the scale of sum |dh|)
    dh2, _, _, _, dbias = ops.bn_prelu_bwd(dev(da), dev(h), mean, var, dev(gamma), dev(beta), dev(alpha), want_dbias=True)
    assert torch.equal(dh2, dh)
    want = host(dh).astype(np.float64).sum(0)
    assert np.abs(host(dbias) - want).max() <= 1e-6 * np.abs(host(dh)).sum(0).max()


# ---------------------------------------------------------------- K3/K7 aggregation
def _spmm_ref(a, x):
    return sp.csr_matrix((np.ones(a.nnz), a.indices, a.indptr), shape=a.shape) @ x.astype(np.float64)


@pytest.mark.parametrize("H", [32, 256, 8, 6, 512])
@pytest.mark.parametrize("transform", [False, True])
def test_spmm_row_kernel(H, transform):
    rng = np.random.default_rng(H)
    a = random_csr(rng, 300, 0.04)
    x = rng.standard_normal((300, H)).astype(np.float32)
    rp, ci = dev(a.indptr.astype(np.int32)), dev(a.indices.astype(np.int32))
    if transform:
        sc, sh, al = (rng.uniform(0.5, 1.5, H).astype(np.float32), rng.normal(0, 0.5, H).astype(np.float32),
                      rng.uniform(0.1, 0.4, H).astype(np.float32))
        z = x.astype(np.float64) * sc + sh
        ref = _spmm_ref(a, np.where(z > 0, z, al * z))
        y = ops.spmm_sum(rp, ci, dev(x), dev(sc), dev(sh), dev(al))
    else:
        ref = _spmm_ref(a, x)
        y = ops.spmm_sum(rp, ci, dev(x))
    assert rel_err(host(y), ref) < TOL


REORDER_TOL = 2e-6   # the same float32 sum taken in another (fixed) order


def same_up_to_order(y, ref):
    """The row-block kernels add a row's neighbours in the order of the RB list (neighbours shared by the whole block
    first, then the row's others, each ascending), the CSR row kernel in ascending column order: one owner per element
    and a fixed order in both, equal up to float32 rounding of a reordered sum."""
    return rel_err(host(y), host(ref).astype(np.float64)) < REORDER_TOL


@pytest.mark.parametrize("n_mean,H", [(60, 32), (300, 64), (700, 256), (1400, 32), (90, 1024)])
def test_spmm_rb4_kernel_matches_row_kernel(n_mean, H):
    """Both kernels add neighbours in a fixed order with one owner per element (deterministic); they differ only in
    that order; the RB4 one is also checked against the oracle and its structure against the CSR."""
    lib = _lib.load()
    ds = synthetic.make_dataset(5, seed=n_mean, n_mean=n_mean, deg=10, n_feat=4)
    ids = np.arange(5, dtype=np.int64)
    _, a, _, _ = g.data.DeviceGraphStore(ds).batch(dev(ids), ids)
    rng = np.random.default_rng(0)
    n = a.n_rows
    x = rng.standard_normal((n, H)).astype(np.float32)
    sc, sh, al = (rng.uniform(0.5, 1.5, H).astype(np.float32), rng.normal(0, 0.5, H).astype(np.float32),
                  rng.uniform(0.1, 0.4, H).astype(np.float32))
    wide = torch.zeros(n, 3 * H, device="cuda")           # write into a slice: ldy != H
    try:
        lib.gcs_debug_set_spmm_mode(1)
        y_rows = ops.spmm_sum(a.rowptr, a.colidx, dev(x), dev(sc), dev(sh), dev(al), rb4=a.rb4)   # mode 1 ignores rb4
    finally:
        lib.gcs_debug_set_spmm_mode(0)
    y_rb4 = ops.spmm_sum(a.rowptr, a.colidx, dev(x), dev(sc), dev(sh), dev(al), out=wide[:, H:2 * H], rb4=a.rb4).clone()
    assert same_up_to_order(y_rb4, y_rows)
    assert torch.equal(y_rb4, ops.spmm_sum(a.rowptr, a.colidx, dev(x), dev(sc), dev(sh), dev(al), rb4=a.rb4))
    try:
        lib.gcs_debug_set_spmm_mode(2)                    # RB4 also without the prologue
        y_id = ops.spmm_sum(a.rowptr, a.colidx, dev(x), rb4=a.rb4)
    finally:
        lib.gcs_debug_set_spmm_mode(0)
    # the RB4 structure itself: per block of 4 rows the union of columns with row masks - first whole groups of four
    # columns that all 4 rows have (flag bit 4, ascending), then the rest ascending
    blk_ptr, ent = (host(t) for t in a.rb4)
    ent = ent.view(np.uint32)
    rp, ci = host(a.rowptr), host(a.colidx)
    assert blk_ptr[0] == 0 and blk_ptr.shape[0] == (n + 3) // 4 + 1 and blk_ptr[-1] <= a.nnz + 3 * ((n + 3) // 4)
    assert np.all(blk_ptr % 4 == 0)                       # blocks are padded to 4 entries (mask 0 = no-op)
    for b in (0, 3, (n - 1) // 4):
        rows = range(4 * b, min(4 * b + 4, n))
        want = {}
        for k, r in enumerate(rows):
            for c in ci[rp[r]:rp[r + 1]]:
                want[int(c)] = want.get(int(c), 0) | (1 << k)
        got = ent[blk_ptr[b]:blk_ptr[b + 1]]
        assert all(int(e >> 8) in want for e in got)
        got = got[(got & 15) != 0]
        shared = sorted(c for c in want if want[c] == 15)
        lead = shared[:len(shared) // 4 * 4]
        order = lead + sorted(c for c in want if c not in lead)
        assert [int(e >> 8) for e in got] == order and [int(e & 15) for e in got] == [want[c] for c in order]
        assert [bool(e & 16) for e in got] == [True] * len(lead) + [False] * (len(order) - len(lead))
    assert blk_ptr[-1] < 0.7 * a.nnz                      # banded graphs: well under one entry per edge
    z = x.astype(np.float64) * sc + sh
    csr = sp.csr_matrix((np.ones(a.nnz), ci, rp), shape=(n, n))
    assert rel_err(host(y_rb4), csr @ np.where(z > 0, z, al * z)) < TOL
    assert rel_err(host(y_id), csr @ x.astype(np.float64)) < TOL
    assert float(wide[:, :H].abs().max()) == 0.0 and float(wide[:, 2 * H:].abs().max()) == 0.0
    # slopes above 1 and negative slopes
    al2 = al.copy()
    al2[::3] = 1.7
    al2[1::5] = -0.3
    try:
        lib.gcs_debug_set_spmm_mode(1)
        y_rows2 = ops.spmm_sum(a.rowptr, a.colidx, dev(x), dev(sc), dev(sh), dev(al2))
    finally:
        lib.gcs_debug_set_spmm_mode(0)
    y_rb4_2 = ops.spmm_sum(a.rowptr, a.colidx, dev(x), dev(sc), dev(sh), dev(al2), rb4=a.rb4)
    assert same_up_to_order(y_rb4_2, y_rows2)
    assert rel_err(host(y_rb4_2), csr @ np.where(z > 0, z, al2 * z)) < TOL


def test_spmm_rb4_arbitrary_structure():
    """A non-banded random matrix with a few dense rows, empty rows and a ragged last block."""
    lib = _lib.load()
    rng = np.random.default_rng(7)
    n = 5003
    a = random_csr(rng, n, 0.004).tolil()
    a[3, :] = 1                                          # one row with 5003 neighbours
    a[300, ::2] = 1
    a[40:48, :] = 0                                      # an empty row block
    a = sp.csr_matrix(a)
    a.sort_indices()
    x = dev(rng.standard_normal((n, 64)).astype(np.float32))
    rp, ci = dev(a.indptr.astype(np.int32)), dev(a.indices.astype(np.int32))
    rb4 = ops.build_rb4(rp, ci)
    try:
        lib.gcs_debug_set_spmm_mode(1)
        y_rows = ops.spmm_sum(rp, ci, x)
    finally:
        lib.gcs_debug_set_spmm_mode(0)
    try:
        lib.gcs_debug_set_spmm_mode(2)
        assert same_up_to_order(ops.spmm_sum(rp, ci, x, rb4=rb4), y_rows)
    finally:
        lib.gcs_debug_set_spmm_mode(0)
    assert rel_err(host(y_rows), _spmm_ref(a, host(x))) < TOL


def _block_diag_batch(rng, sizes, density):
    """Disjoint batch of random (non-banded, directed) graphs of the given sizes; some rows empty."""
    mats = []
    for n in sizes:
        d = (rng.random((n, n)) < density).astype(np.int64)
        if n > 3:
            d[rng.integers(0, n)] = 0                     # an empty row
            d[rng.integers(0, n)] = 1                     # a full row
        mats.append(sp.csr_matrix(d))
    a = sp.block_diag(mats, format="csr")
    a.sort_indices()
    gp = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    return a, gp


@pytest.mark.parametrize("stages", [3, 2])
@pytest.mark.parametrize("height", [2, 4])
@pytest.mark.parametrize("H,sizes,slab_bytes", [
    (256, [37, 1, 2, 3, 130, 5, 64, 7, 255], None),       # ragged graphs, blocks straddling graph boundaries
    (48, [301, 17, 90], None),                            # last column group 16 wide
    (20, [9, 33, 4], None),                               # column group of 20 = passes of 16 + 4
    (64, [700, 40, 1300, 5], 32768),                      # small slab: passes of 8 and 4 columns for the long graphs
    (512, [150, 151], None),
])
def test_spmm_slab_kernel_bitwise(stages, height, H, sizes, slab_bytes):
    """The per-graph shared-memory kernel (gcs_spmm_sum_graphs) adds each row's neighbours in the order of the RB list
    (the block's shared neighbours through one shared sum): bit-identical to the global-memory row-block kernel, equal
    to the CSR row kernel up to the rounding of a reordered sum, with and without the prologue and the residual, written
    into a column slice; also against the float64 oracle."""
    lib = _lib.load()
    rng = np.random.default_rng(H + height)
    a, gp = _block_diag_batch(rng, sizes, 0.08)
    n = a.shape[0]
    x = rng.standard_normal((n, H)).astype(np.float32)
    res = rng.standard_normal((n, H)).astype(np.float32)
    sc, sh, al = (rng.uniform(0.5, 1.5, H).astype(np.float32), rng.normal(0, 0.5, H).astype(np.float32),
                  rng.uniform(-0.3, 1.4, H).astype(np.float32))
    rp, ci, gpd = dev(a.indptr.astype(np.int32)), dev(a.indices.astype(np.int32)), dev(gp)
    rb = ops.build_rb(rp, ci, height)
    try:
        lib.gcs_debug_set_spmm_mode(1)
        y_rows = ops.spmm_sum(rp, ci, dev(x), dev(sc), dev(sh), dev(al))
        y_rows_plain = ops.spmm_sum(rp, ci, dev(x))
    finally:
        lib.gcs_debug_set_spmm_mode(0)
    wide = torch.zeros(n, 3 * H, device="cuda")
    try:
        lib.gcs_debug_set_param(10, stages)
        if slab_bytes:
            lib.gcs_debug_set_param(11, slab_bytes)      # small stages: narrow passes; entries that do not fit: direct gather
        y = ops.spmm_sum_graphs(gpd, max(sizes), rp, ci, dev(x), dev(sc), dev(sh), dev(al), out=wide[:, H:2 * H], rb=rb,
                                rb_height=height).clone()
        y_plain = ops.spmm_sum_graphs(gpd, max(sizes), rp, ci, dev(x), rb=rb, rb_height=height)
        y_res = ops.spmm_sum_graphs(gpd, max(sizes), rp, ci, dev(x), dev(sc), dev(sh), dev(al), residual=dev(res), rb=rb,
                                    rb_height=height)
    finally:
        lib.gcs_debug_set_param(11, 0)
        lib.gcs_debug_set_param(10, 2)
    assert same_up_to_order(y, y_rows) and same_up_to_order(y_plain, y_rows_plain)
    assert torch.equal(y_res, y + dev(res))
    if height == 4:                                       # the same list, the same order: the same bits
        try:
            lib.gcs_debug_set_spmm_mode(2)
            assert torch.equal(y, ops.spmm_sum(rp, ci, dev(x), dev(sc), dev(sh), dev(al), rb4=rb))
            assert torch.equal(y_plain, ops.spmm_sum(rp, ci, dev(x), rb4=rb))
        finally:
            lib.gcs_debug_set_spmm_mode(0)
    assert float(wide[:, :H].abs().max()) == 0.0 and float(wide[:, 2 * H:].abs().max()) == 0.0
    z = x.astype(np.float64) * sc + sh
    assert rel_err(host(y), _spmm_ref(a, np.where(z > 0, z, al * z))) < TOL


def test_spmm_graphs_falls_back_without_slab():
    """No graph_ptr / unknown graph lengths / graphs longer than a slab: the global-memory kernels run, same result."""
    lib = _lib.load()
    rng = np.random.default_rng(3)
    a, gp = _block_diag_batch(rng, [60, 500, 31], 0.05)
    x = dev(rng.standard_normal((a.shape[0], 32)).astype(np.float32))
    rp, ci = dev(a.indptr.astype(np.int32)), dev(a.indices.astype(np.int32))
    ref = ops.spmm_sum(rp, ci, x)
    rb2, rb4 = ops.build_rb(rp, ci, 2), ops.build_rb(rp, ci, 4)
    assert same_up_to_order(ops.spmm_sum_graphs(None, 0, rp, ci, x, rb=rb4, rb_height=4), ref)
    assert torch.equal(ops.spmm_sum_graphs(dev(gp), 0, rp, ci, x, rb=rb2, rb_height=2), ref)   # height 2 without a slab: CSR rows
    try:
        lib.gcs_debug_set_param(11, 4096)                # 500 nodes * 16 bytes > 4096
        assert torch.equal(ops.spmm_sum_graphs(dev(gp), 500, rp, ci, x, rb=rb2, rb_height=2), ref)
    finally:
        lib.gcs_debug_set_param(11, 0)


@pytest.mark.parametrize("H", [64, 6, 257, 260, 512, 1028])     # above 256 lanes per row: column slices over gridDim.y
@pytest.mark.parametrize("aggregate", ["sum", "mean", "max"])
@pytest.mark.parametrize("weighted", [False, True])
def test_spmm_aggregate_weights_mean_max_residual(H, aggregate, weighted):
    """gcs_spmm_aggregate against a per-row NumPy restatement of Spektral's scatter_sum / scatter_mean / scatter_max
    (tf.math.unsorted_segment_*: an empty row gives 0 for sum and mean, the lowest float for max), with per-entry
    weights, the fused BatchNorm+PReLU prologue and a residual added after the aggregation."""
    rng = np.random.default_rng(H + len(aggregate))
    n = 400
    a = random_csr(rng, n, 0.03).tolil()
    a[17, :] = 0                                          # empty rows
    a[200:204, :] = 0
    a = sp.csr_matrix(a)
    a.sort_indices()
    x = rng.standard_normal((n, H)).astype(np.float32)
    res = rng.standard_normal((n, H)).astype(np.float32)
    vals = rng.uniform(-1, 2, a.nnz).astype(np.float32) if weighted else None
    sc, sh, al = (rng.uniform(0.5, 1.5, H).astype(np.float32), rng.normal(0, 0.5, H).astype(np.float32),
                  rng.uniform(0.1, 0.4, H).astype(np.float32))
    z = x.astype(np.float64) * sc + sh
    f = np.where(z > 0, z, al * z)
    ref = np.zeros((n, H))
    for r in range(n):
        lo, hi = a.indptr[r], a.indptr[r + 1]
        m = f[a.indices[lo:hi]] * (vals[lo:hi, None].astype(np.float64) if weighted else 1.0)
        if aggregate == "max":
            ref[r] = m.max(0) if hi > lo else np.finfo(np.float32).min
        elif hi > lo:
            ref[r] = m.sum(0) / ((hi - lo) if aggregate == "mean" else 1)
    rp, ci = dev(a.indptr.astype(np.int32)), dev(a.indices.astype(np.int32))
    y = ops.spmm_aggregate(rp, ci, dev(x), dev(sc), dev(sh), dev(al), values=None if vals is None else dev(vals),
                           aggregate=aggregate)
    assert rel_err(host(y), ref) < TOL
    y = ops.spmm_aggregate(rp, ci, dev(x), dev(sc), dev(sh), dev(al), values=None if vals is None else dev(vals),
                           residual=dev(res), aggregate=aggregate)
    ref_r = np.where(ref == np.finfo(np.float32).min, ref, ref + res)
    got = host(y)
    keep = ref != np.finfo(np.float32).min               # lowest float + residual: not a meaningful number
    assert rel_err(got[keep], ref_r[keep]) < TOL
    with pytest.raises(ValueError):
        ops.spmm_aggregate(rp, ci, dev(x), aggregate="median")


def test_spmm_residual_on_the_row_block_kernel():
    """Add()([z, out]): the RB4 kernel with a residual equals the row kernel with a residual bit for bit, and both equal
    aggregate-then-add."""
    lib = _lib.load()
    ds = synthetic.make_dataset(5, seed=3, n_mean=300, deg=10, n_feat=4)
    ids = np.arange(5, dtype=np.int64)
    _, a, _, _ = g.data.DeviceGraphStore(ds).batch(dev(ids), ids)
    rng = np.random.default_rng(0)
    n, H = a.n_rows, 128
    x, res = dev(rng.standard_normal((n, H)).astype(np.float32)), dev(rng.standard_normal((n, 2 * H)).astype(np.float32))
    sc, sh, al = (dev(rng.uniform(0.5, 1.5, H).astype(np.float32)), dev(rng.normal(0, 0.5, H).astype(np.float32)),
                  dev(rng.uniform(0.1, 0.4, H).astype(np.float32)))
    plain = ops.spmm_sum(a.rowptr, a.colidx, x, sc, sh, al, rb4=a.rb4)
    y_rb4 = ops.spmm_aggregate(a.rowptr, a.colidx, x, sc, sh, al, residual=res[:, H:], rb4=a.rb4)
    try:
        lib.gcs_debug_set_spmm_mode(1)
        y_rows = ops.spmm_aggregate(a.rowptr, a.colidx, x, sc, sh, al, residual=res[:, H:], rb4=a.rb4)
    finally:
        lib.gcs_debug_set_spmm_mode(0)
    assert same_up_to_order(y_rb4, y_rows) and torch.equal(y_rb4, plain + res[:, H:])


def test_spmm_is_deterministic_and_handles_empty_rows():
    rng = np.random.default_rng(1)
    a = random_csr(rng, 500, 0.02)
    a[7] = 0
    a.eliminate_zeros()
    x = dev(rng.standard_normal((500, 64)).astype(np.float32))
    rp, ci = dev(a.indptr.astype(np.int32)), dev(a.indices.astype(np.int32))
    y1, y2 = ops.spmm_sum(rp, ci, x), ops.spmm_sum(rp, ci, x)
    assert torch.equal(y1, y2) and float(y1[7].abs().max()) == 0.0
    with pytest.raises(ValueError):
        ops.spmm_sum(rp, ci, x, scale=torch.ones(64, device="cuda"))      # partial prologue


def test_spmm_sum_and_sum_graphs_at_an_odd_width_above_256():
    """H = 258: no 16-byte vectors, so both entry points run the scalar row kernel, one lane per column over two column
    slices; against float64, deterministic, empty rows 0."""
    rng = np.random.default_rng(258)
    H = 258
    a, gp = _block_diag_batch(rng, [60, 1, 130, 17], 0.06)
    n = a.shape[0]
    x = rng.standard_normal((n, H)).astype(np.float32)
    sc, sh, al = (rng.uniform(0.5, 1.5, H).astype(np.float32), rng.normal(0, 0.5, H).astype(np.float32),
                  rng.uniform(-0.3, 1.4, H).astype(np.float32))
    rp, ci = dev(a.indptr.astype(np.int32)), dev(a.indices.astype(np.int32))
    empty = np.diff(a.indptr) == 0
    assert empty.any()
    z = x.astype(np.float64) * sc + sh
    ref = _spmm_ref(a, np.where(z > 0, z, al * z))
    y1 = ops.spmm_sum(rp, ci, dev(x), dev(sc), dev(sh), dev(al))
    assert rel_err(host(y1), ref) < TOL and float(y1[dev(empty)].abs().max()) == 0.0
    assert torch.equal(y1, ops.spmm_sum(rp, ci, dev(x), dev(sc), dev(sh), dev(al)))
    assert rel_err(host(ops.spmm_sum(rp, ci, dev(x))), _spmm_ref(a, x)) < TOL
    rb = ops.build_rb(rp, ci, 4)
    y2 = ops.spmm_sum_graphs(dev(gp), 130, rp, ci, dev(x), dev(sc), dev(sh), dev(al), rb=rb, rb_height=4)
    assert torch.equal(y2, y1)


# ---------------------------------------------------------------- K4/K6 pooling
@pytest.mark.parametrize("W", [1280, 96, 7])
def test_segment_sum_forward_backward(W):
    rng = np.random.default_rng(W)
    sizes = np.array([5, 1, 0, 300, 64, 17])
    gp = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    n = int(gp[-1])
    x = rng.standard_normal((n, W)).astype(np.float32)
    seg = np.repeat(np.arange(len(sizes)), sizes)
    out = ops.segment_sum_fwd(dev(x), dev(gp))
    assert rel_err(host(out), O1.segment_sum(x.astype(np.float64), seg, len(sizes))) < TOL
    assert float(out[2].abs().max()) == 0.0               # empty segment -> zeros (tf.segment_sum)
    dout = rng.standard_normal((len(sizes), W)).astype(np.float32)
    assert np.array_equal(host(ops.segment_sum_bwd(dev(dout), dev(gp), n)), dout[seg])


# ---------------------------------------------------------------- K5 loss, K10 optimizers
@pytest.mark.parametrize("B,C", [(1024, 2), (50, 2), (7, 5), (1, 3)])
def test_softmax_xent(B, C):
    rng = np.random.default_rng(B + C)
    z = (rng.standard_normal((B, C)) * 3).astype(np.float32)
    y = np.eye(C, dtype=np.float32)[rng.integers(0, C, B)]
    probs, loss_acc, dlogits = ops.softmax_xent(dev(z), dev(y), want_grad=True)
    z64 = z.astype(np.float64)
    p = np.exp(z64 - z64.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    loss, _ = O1.xent_from_logits(z64, y.astype(np.float64))
    la = host(loss_acc)
    assert rel_err(host(probs), p) < TOL and abs(la[0] - loss) < TOL * abs(loss)
    assert abs(la[1] - O1.accuracy(p, y)) < 1e-6
    assert rel_err(host(dlogits), (p - y) / B) < TOL
    p_only, none1, none2 = ops.softmax_xent(dev(z))
    assert none1 is None and none2 is None and torch.equal(p_only, probs)


def test_fused_optimizer_steps():
    rng = np.random.default_rng(0)
    n = 100003
    w = rng.standard_normal(n).astype(np.float32)
    gr = rng.standard_normal(n).astype(np.float32)
    wd = dev(w)
    ops.sgd_step(wd, dev(gr), 0.02, 0.5)
    assert rel_err(host(wd), O1.sgd_step(w.astype(np.float64), 0.5 * gr.astype(np.float64), 0.02)) < 1e-6
    wd, m, v = dev(w), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    w64, m64, v64 = w.astype(np.float64), np.zeros(n), np.zeros(n)
    for t in range(1, 4):
        ops.adam_step(wd, dev(gr), m, v, t, 1e-3)
        w64, m64, v64 = O1.adam_step(w64, gr.astype(np.float64), m64, v64, t, 1e-3)
    assert rel_err(host(wd), w64) < 1e-6 and rel_err(host(m), m64) < 1e-6 and rel_err(host(v), v64) < 1e-6


def test_bad_arguments_raise_with_a_message():
    x = torch.zeros(4, 8, device="cuda")
    with pytest.raises(ValueError, match="shape mismatch"):
        ops.linear_fwd(x, torch.zeros(7, 3, device="cuda"))
    with pytest.raises(ValueError, match="float32"):
        ops.linear_fwd(x.double(), torch.zeros(8, 3, device="cuda"))
    lib = _lib.load()
    st = lib.gcs_spmm_sum(None, None, None, None, 5, None, 8, None, None, None, None, 8, 8, _lib.stream_ptr())
    assert st == 1 and b"null pointer" in lib.gcs_last_error()
