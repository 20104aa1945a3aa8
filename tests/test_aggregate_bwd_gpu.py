"""gcs_spmm_aggregate_bwd - the gradient of the weighted / mean / max aggregation (spmm_agg_bwd_kernel and
spmm_max_ties_kernel) - against a float64 NumPy restatement over the COO entries of the forward matrix
(oracle.model_ref_np.aggregate_bwd), and GeneralGNN train steps on directed, weighted graphs against the float64 oracle.

max hands a row's gradient to the entries that attain its maximum, shared equally between ties.  Whether an entry
attains it is decided in float32, so the reference selects by comparing float32 messages with the kernel's own forward
output.  Its messages are the float32 products themselves (rounded once, as on the GPU) or, with the BatchNorm + PReLU
prologue, 'exact' inputs - quarter-integers, power-of-two scales, weights in {-1, -1/2, 0, 1/2, 1, 2} - on which every
forward operation is exact in float32; there the tie counts and the maxima must agree bit for bit."""
import numpy as np
import pytest
import scipy.sparse as sp

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import _lib, ops, synthetic
from gcn_string_b200.data import SparseAdjacency
from gcn_string_b200.params import GNNConfig, block_specs
from oracle import batching_ref, model_ref_np as O1

from conftest import rel_err
from test_model_gpu import assert_grads_close

pytestmark = pytest.mark.gpu
TOL = 1e-5
# VEC = 1 (H <= 256) and VEC = 4 branches of the backward, H % 4 != 0 above 256, rows wider than one CTA's 256 lanes
WIDTHS = [1, 6, 16, 128, 256, 257, 260, 301, 512, 1024, 1028, 2051]
SENTINEL = 12345.0


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def pattern(kind, n, rng, deg=5.0):
    """Row-major sorted COO (rows, cols) of a directed n x n pattern of about ``deg`` entries per row."""
    d = rng.random((n, n)) < deg / n
    if kind == "symmetric":
        d |= d.T
    elif kind == "empty_rows":
        d[rng.choice(n, n // 8, replace=False)] = False
    elif kind == "unreferenced":                          # columns no row refers to: their dA rows must be written as 0
        d[:, rng.choice(n, n // 8, replace=False)] = False
    elif kind == "hub":                                   # one transposed row with an entry from every row
        d[:, n // 3] = True
    rows, cols = np.nonzero(d)
    if kind == "duplicates":                              # every other row repeats one of its entries once or twice
        rep = np.ones(rows.shape[0], dtype=np.int64)
        starts = np.searchsorted(rows, np.arange(0, n, 2))
        starts = starts[(starts < rows.shape[0])]
        rep[starts] += rng.integers(1, 3, starts.shape[0])
        rows, cols = np.repeat(rows, rep), np.repeat(cols, rep)
    return rows.astype(np.int64), cols.astype(np.int64)


def csr(rows, cols, n):
    return np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]).astype(np.int32), cols.astype(np.int32)


def make_inputs(rng, rows, cols, n, H, weights, prologue, exact):
    """x [n, H], per-entry weights (or None), (scale, shift, alpha) (or None), dz [n, H] - all float32."""
    nnz = rows.shape[0]
    if exact:
        x = rng.integers(-8, 9, (n, H)) / 4.0
        key = np.unique(rows * n + cols, return_inverse=True)[1]          # duplicates of an entry share its weight
        w = {"none": None, "positive": rng.choice([0.5, 1.0, 2.0], nnz),
             "signed": rng.choice([-1.0, -0.5, 0.0, 0.5, 1.0, 2.0], nnz)}[weights]
        w = None if w is None else w[key]
        sc, sh = rng.choice([-2.0, -1.0, -0.5, 0.5, 1.0, 2.0], H), rng.integers(-4, 5, H) / 4.0
        al = np.resize([-0.25, 0.25, 1.5], H)
    else:
        x = rng.standard_normal((n, H))
        w = {"none": None, "positive": rng.uniform(0.2, 1.5, nnz), "signed": rng.uniform(-1.5, 1.5, nnz)}[weights]
        if weights == "signed":
            w[rng.random(nnz) < 0.1] = 0.0
        sc, sh = rng.uniform(0.5, 1.5, H), rng.normal(0.0, 0.5, H)
        al = np.resize([-0.3, 0.4, 1.7], H) * rng.uniform(0.8, 1.2, H)   # negative, in (0, 1), above 1
    f32 = lambda a: None if a is None else np.asarray(a, dtype=np.float32)
    pro = (f32(sc), f32(sh), f32(al)) if prologue else None
    return f32(x), f32(w), pro, rng.standard_normal((n, H)).astype(np.float32)


def messages(x, w, pro, cols, exact):
    """The max messages w_ij * f(x[j]) as float64 holding the float32 values the kernels compute."""
    if pro is None:
        m = x[cols] if w is None else x[cols] * w[:, None]                 # float32 products: rounded once, like the GPU
        return m.astype(np.float64)
    assert exact, "with a prologue the messages are only reproducible on exact inputs"
    sc, sh, al = (v.astype(np.float64) for v in pro)
    z = x.astype(np.float64) * sc + sh
    f = np.where(z > 0, z, al * z)
    m = f[cols] if w is None else f[cols] * w[:, None].astype(np.float64)
    assert np.array_equal(m.astype(np.float32).astype(np.float64), m)      # every operation exact in float32
    return m


def placed(a, offset):
    """A device copy of ``a`` [n, H]: contiguous (offset None) or a column slice starting at ``offset`` of a wider
    buffer padded with SENTINEL.  -> (view, buffer)."""
    if offset is None:
        t = dev(a)
        return t, t
    n, H = a.shape
    ld = (H + 8) // 4 * 4 + 4
    buf = torch.full((n, ld), SENTINEL, device="cuda")
    view = buf[:, offset:offset + H]
    view.copy_(dev(a))
    return view, buf


def padding_intact(buf, offset, H):
    if offset is None:
        return True
    b = host(buf)
    return bool(np.all(b[:, :offset] == SENTINEL) and np.all(b[:, offset + H:] == SENTINEL))


def check_bwd(rows, cols, n, H, aggregate, weights="none", prologue=False, exact=False, seed=0, offset=None):
    """One backward call against the float64 restatement; returns the reference tie counts (max) or None."""
    rng = np.random.default_rng(seed)
    x, w, pro, dz = make_inputs(rng, rows, cols, n, H, weights, prologue, exact)
    rp_h, ci_h = csr(rows, cols, n)
    nnz = rows.shape[0]
    # the transposed pattern and the weights in its order, built independently of the library
    at = sp.csr_matrix((np.arange(nnz), ci_h, rp_h), shape=(n, n)).T.tocsr()
    perm = at.data
    rp, ci = dev(rp_h), dev(ci_h)
    rpt, cit = dev(at.indptr.astype(np.int32)), dev(at.indices.astype(np.int32))
    wd, wtd = (None, None) if w is None else (dev(w), dev(w[perm]))
    prod = () if pro is None else tuple(dev(v) for v in pro)
    kw = {} if pro is None else dict(zip(("scale", "shift", "alpha"), prod))
    dzv, dzbuf = placed(dz, offset)
    xv, xbuf = placed(x, offset)
    z = ties_ref = ties = None
    if aggregate == "max":
        msg = messages(x, w, pro, cols, exact)
        z_ref = np.full((n, H), np.finfo(np.float32).min)
        np.maximum.at(z_ref, rows, msg)
        z, zbuf = placed(np.zeros((n, H), np.float32), offset)
        ops.spmm_aggregate(rp, ci, xv, *prod, values=wd, aggregate="max", out=z)
        assert np.array_equal(host(z), z_ref)             # the forward max of float32 messages is exact
        assert padding_intact(zbuf, offset, H)
        sel = msg == host(z).astype(np.float64)[rows]
        ties_ref = np.zeros((n, H))
        np.add.at(ties_ref, rows, sel)
        ties, tbuf = placed(np.full((n, H), -1.0, np.float32), offset)
        ctx = msg
    else:
        ctx = np.bincount(rows, minlength=n).astype(np.float64) if aggregate == "mean" else None
    da, dabuf = placed(np.full((n, H), np.nan, np.float32), offset)
    out = ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dzv, aggregate, values_t=wtd, values=wd, x=xv, z=z, out=da, ties=ties,
                                 **kw)
    assert out.data_ptr() == da.data_ptr()
    ref = O1.aggregate_bwd(rows, cols, dz.astype(np.float64), n, aggregate, None if w is None else w.astype(np.float64),
                           ctx, None if z is None else host(z).astype(np.float64))
    got = host(da)
    assert not np.isnan(got).any()                        # every row written, also those no entry refers to
    assert np.all(got[np.bincount(cols, minlength=n) == 0] == 0.0)
    assert rel_err(got, ref) < TOL, (aggregate, weights, prologue, H)
    for buf in (dzbuf, xbuf, dabuf):
        assert padding_intact(buf, offset, H)
    if ties is not None:
        assert np.array_equal(host(ties), np.maximum(ties_ref, 1.0))   # counted exactly; an empty row counts 1
        assert padding_intact(tbuf, offset, H)
    # deterministic: a second call gives the same bits
    again = ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dzv, aggregate, values_t=wtd, values=wd, x=xv, z=z, **kw)
    assert torch.equal(again, da)
    # the production route: the library's transpose and SparseAdjacency.edge_weight_t()
    rpt2, cit2 = ops.csr_transpose(rp, ci)
    assert np.array_equal(host(rpt2), at.indptr) and np.array_equal(host(cit2), at.indices)
    if w is not None:
        adj = SparseAdjacency(rp, ci, n)
        adj.edge_weight = wd
        wtd2 = adj.edge_weight_t()
        prod_da = ops.spmm_aggregate_bwd(rpt2, cit2, rp, ci, dzv, aggregate, values_t=wtd2, values=wd, x=xv, z=z, **kw)
        if np.unique(rows * n + cols).shape[0] == nnz:    # without duplicates the transposed order is unique
            assert torch.equal(wtd2, wtd) and torch.equal(prod_da, da)
        else:                                             # duplicates of an entry may come in another order
            assert rel_err(host(prod_da), ref) < TOL
    return ties_ref


@pytest.mark.parametrize("aggregate", ["sum", "mean", "max"])
@pytest.mark.parametrize("H", WIDTHS)
def test_aggregate_bwd_widths(H, aggregate):
    """Every width on a directed random pattern, unweighted / positive / signed weights with exact zeros, without and
    with the prologue (slopes negative, in (0, 1) and above 1; for max on exact inputs)."""
    rng = np.random.default_rng(H)
    n = 150
    rows, cols = pattern("directed", n, rng)
    for weights in ("none", "positive", "signed"):
        for prologue in (False, True):
            check_bwd(rows, cols, n, H, aggregate, weights, prologue, exact=aggregate == "max" and prologue, seed=H + 7)


@pytest.mark.parametrize("H", [6, 260])
@pytest.mark.parametrize("kind", ["directed", "symmetric", "empty_rows", "unreferenced", "hub", "duplicates"])
def test_aggregate_bwd_patterns(kind, H):
    """Rows without entries, columns without entries (dA written as 0 over a NaN-filled output), a column every row
    refers to (a transposed row of 3000 entries), and repeated (i, j) entries within a row."""
    rng = np.random.default_rng(len(kind) + H)
    n = 3000 if kind == "hub" else 300
    rows, cols = pattern(kind, n, rng)
    if kind == "hub":
        assert np.bincount(cols).max() == n
    for aggregate in ("sum", "mean", "max"):
        for weights in ("none", "signed"):
            check_bwd(rows, cols, n, H, aggregate, weights, seed=n + H)
        if aggregate == "max":
            check_bwd(rows, cols, n, H, aggregate, "signed", prologue=True, exact=True, seed=n + H)


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("H", [6, 260, 1028])
def test_aggregate_bwd_on_column_slices(H, offset):
    """dz, x, z, ties and dA as column slices of wider buffers whose padding must stay untouched; at offset 1 the rows
    are not 16-byte aligned and the forward runs its scalar kernel."""
    rng = np.random.default_rng(H + offset)
    n = 200
    rows, cols = pattern("duplicates", n, rng)
    for aggregate in ("sum", "mean", "max"):
        check_bwd(rows, cols, n, H, aggregate, "signed", seed=H, offset=offset)
    check_bwd(rows, cols, n, H, "max", "signed", prologue=True, exact=True, seed=H, offset=offset)


@pytest.mark.parametrize("weights", ["none", "signed"])
@pytest.mark.parametrize("prologue", [False, True])
@pytest.mark.parametrize("H", [1, 6, 257, 1028])
def test_aggregate_bwd_max_exact_ties(H, prologue, weights):
    """Exact inputs with many ties: the kernel's tie counts and its forward maxima equal the reference bit for bit, the
    gradient shared between them is within 1e-5.  Repeated entries share their weight, so they tie with themselves."""
    rng = np.random.default_rng(H)
    n = 200
    rows, cols = pattern("duplicates", n, rng, deg=8.0)
    ties = check_bwd(rows, cols, n, H, "max", weights, prologue, exact=True, seed=H)
    nonempty = np.bincount(rows, minlength=n) > 0
    assert (ties[nonempty] >= 2).mean() > 0.1                         # the situation the test is about
    assert (ties >= 3).any()


def test_aggregate_bwd_without_rows_launches_nothing():
    lib = _lib.load()
    rp, ci = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(0, dtype=torch.int32, device="cuda")
    dz = torch.zeros(0, 8, device="cuda")
    before = lib.gcs_debug_launch_count()
    for aggregate in ops.AGGREGATE:
        assert ops.spmm_aggregate_bwd(rp, ci, rp, ci, dz, aggregate, x=dz, z=dz).shape == (0, 8)
    assert lib.gcs_debug_launch_count() == before


def test_aggregate_bwd_bad_arguments_raise_with_a_message():
    rng = np.random.default_rng(0)
    n, H = 20, 8
    rp_h, ci_h = csr(*pattern("directed", n, rng), n)
    rp, ci = dev(rp_h), dev(ci_h)
    rpt, cit = ops.csr_transpose(rp, ci)
    dz, x = torch.ones(n, H, device="cuda"), torch.ones(n, H, device="cuda")
    z = ops.spmm_aggregate(rp, ci, x, aggregate="max")
    ones = torch.ones(H, device="cuda")
    w = torch.ones(ci.shape[0], device="cuda")
    with pytest.raises(ValueError, match="rows"):
        ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dz[1:], "sum")
    with pytest.raises(ValueError, match="x and z must be"):
        ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dz, "max", x=x[:, 1:], z=z)
    with pytest.raises(ValueError, match="dA must be"):
        ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dz, "mean", out=torch.empty(n, H + 1, device="cuda"))
    with pytest.raises(ValueError, match="scale, shift and alpha"):
        ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dz, "max", x=x, z=z, scale=ones, shift=ones)
    with pytest.raises(ValueError, match="needs the forward input x and output z"):
        ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dz, "max", x=x)
    with pytest.raises(ValueError, match="values and values_t go together"):
        ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dz, "sum", values=w)
    with pytest.raises(ValueError, match="aggregate must be one of"):
        ops.spmm_aggregate_bwd(rpt, cit, rp, ci, dz, "median")
    # the C entry point refuses max without Z before it launches anything
    lib = _lib.load()
    before = lib.gcs_debug_launch_count()
    da, ties = torch.empty(n, H, device="cuda"), torch.empty(n, H, device="cuda")
    p = _lib.ptr
    st = lib.gcs_spmm_aggregate_bwd(p(rpt), p(cit), None, p(rp), p(ci), None, n, p(dz), H, 2, p(x), H, None, None, None,
                                    None, H, p(ties), H, p(da), H, H, _lib.stream_ptr())
    assert st == 1 and b"max needs" in lib.gcs_last_error()
    assert lib.gcs_debug_launch_count() == before


# ---------------------------------------------------------------- GeneralGNN train steps
def directed_batch(seed, F, sizes=(30, 1, 45, 12, 60, 7)):
    """A disjoint batch of random DIRECTED graphs with a self-loop on every node (max is then defined on every row):
    the loader's batch and the oracle's collate of the same graphs."""
    rng = np.random.default_rng(seed)
    graphs = []
    for k, n in enumerate(sizes):
        d = rng.random((n, n)) < 0.2
        np.fill_diagonal(d, True)
        graphs.append(g.Graph(x=rng.random((n, F)), a=sp.csr_matrix(d.astype(np.int64)), y=np.eye(2, dtype=np.int64)[k % 2]))
    ref = batching_ref.collate([(gr.x, gr.a, gr.y) for gr in graphs])
    loader = g.DisjointLoader(synthetic.pack_graphs(graphs), batch_size=len(graphs), epochs=1, shuffle=False, want_coo=True)
    return ref, loader


def make_model(cfg, w, s, weighted):
    m = g.GeneralGNN(cfg.output, activation=cfg.activation, hidden=cfg.hidden, message_passing=cfg.message_passing,
                     connectivity=cfg.connectivity, aggregate=cfg.aggregate, use_edge_weights=weighted)
    m.build(cfg.in_features)
    m.load_flat(w, s)
    return m


def unit_slopes(cfg, w):
    """PReLU slopes of 1: no kink the float32 and float64 sides could fall on either side of."""
    for b in block_specs(cfg):
        o, n = b.alpha
        w[o:o + n] = 1.0
    return w


def train_step_vs_oracle(cfg, batch, loader, ew, seed):
    (xr, (idx, _, _), seg), yr = batch
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=seed, perturb=True)
    w = unit_slopes(cfg, w)
    B = yr.shape[0]
    ref = O1.loss_and_grads(cfg, specs, w, s, xr, idx[:, 0], idx[:, 1], seg, yr, B, edge_weight=ew)
    (x, a, i), y = next(loader)
    assert np.array_equal(host(a.indices), idx)           # edge weights are given in this (CSR) entry order
    if ew is not None:
        a.edge_weight = dev(ew)
    model = make_model(cfg, w, s, ew is not None)
    loss_acc, probs = model.train_step_grads([x, a, i], y)
    assert abs(host(loss_acc)[0] - ref["loss"]) < TOL * abs(ref["loss"])
    assert rel_err(host(probs), ref["probs"]) < TOL
    assert rel_err(host(model.state), ref["new_state"]) < TOL
    assert_grads_close(host(model.grads), ref["grads"], cfg, None, tol=2 * TOL)
    return a


@pytest.mark.parametrize("aggregate,weighted", [("sum", True), ("mean", False), ("mean", True), ("max", False),
                                                ("max", True)])
def test_train_step_on_directed_weighted_graphs(aggregate, weighted):
    """The backward reads the transposed pattern, the weights in its order and the forward row counts; on a directed
    pattern with asymmetric weights these all differ from the forward arrays."""
    F = 7
    batch, loader = directed_batch(11, F)
    idx = batch[0][1][0]
    ew = np.random.default_rng(2).uniform(0.2, 1.5, idx.shape[0]).astype(np.float32) if weighted else None
    cfg = GNNConfig(in_features=F, output=2, activation="softmax", hidden=20, message_passing=3, connectivity="cat",
                    aggregate=aggregate)
    a = train_step_vs_oracle(cfg, batch, loader, ew, seed=5)
    assert not a.symmetric


@pytest.mark.parametrize("aggregate", ["sum", "mean"])
def test_train_step_at_hidden_258(small_case, aggregate):
    """A hidden width above 256 that is not a multiple of 4: the aggregations run the scalar row kernel over two column
    slices, the mean backward its 4-column lanes."""
    c = small_case
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=258, message_passing=2, connectivity="cat",
                    aggregate=aggregate)
    batch = ((c["x"], (c["idx"], None, None), c["seg"]), c["y"])
    loader = g.DisjointLoader(c["ds"], batch_size=8, epochs=1, shuffle=False, want_coo=True)
    train_step_vs_oracle(cfg, batch, loader, None, seed=21)


def test_in_place_edge_weight_edit_reaches_the_backward():
    """a.edge_weight.copy_(w2) between two steps on the same adjacency: the second step's gradients are those of a fresh
    adjacency carrying w2 (the weights in transposed order are cached, keyed on the tensor and its in-place version)."""
    F = 5
    (x, a, i), y = next(directed_batch(3, F)[1])
    rng = np.random.default_rng(4)
    w1, w2 = (rng.uniform(0.2, 1.5, a.nnz).astype(np.float32) for _ in range(2))
    cfg = GNNConfig(in_features=F, output=2, activation="softmax", hidden=16, message_passing=2, aggregate="sum")
    w, s = g.init_params(cfg, seed=6, perturb=True)
    model = make_model(cfg, w, s, True)
    a.edge_weight = dev(w1)
    model.train_step_grads([x, a, i], y)
    g1 = model.grads.clone()
    a.edge_weight.copy_(dev(w2))
    model.load_flat(w, s)
    model.train_step_grads([x, a, i], y)
    g_edit = model.grads.clone()
    (x2, a2, i2), y2 = next(directed_batch(3, F)[1])
    a2.edge_weight = dev(w2)
    model.load_flat(w, s)
    model.train_step_grads([x2, a2, i2], y2)
    assert not torch.equal(g_edit, g1)
    assert torch.equal(g_edit, model.grads)
