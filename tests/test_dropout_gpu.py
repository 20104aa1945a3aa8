"""GPU tests of GeneralGNN(dropout=rate): the device mask function against the NumPy restatement bit for bit, the fused
train step against the float64 restatement with the same masks for every pool, connectivity, aggregation, edge
weights, head, sample weights, width and aggregation path, seed and step behaviour, inference, the GradientTape route,
two data-parallel ranks, the dropped fraction and an allocation-free loop."""
import math
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import _lib, synthetic
from gcn_string_b200.params import GNNConfig, block_specs, dropout_seed

from oracle import model_ref_np as O1

import dropout_ref as D

from conftest import rel_err
from test_model_gpu import TOL, gpu_prelu_branches, grad_errors, host

pytestmark = pytest.mark.gpu
LOSS = {"mse": lambda: g.MeanSquaredError()}


def device_mask(seed, step, block, rows, cols, rate):
    out = torch.empty(rows, cols, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().gcs_debug_dropout_keep(seed, step, block, rows, cols, rate, out.data_ptr(), _lib.stream_ptr()))
    return host(out).astype(bool)


@pytest.mark.parametrize("seed,step,block", [(0, 0, 0), (123456789, 7, 3), (2 ** 64 - 1, 2 ** 33 + 5, 9)])
@pytest.mark.parametrize("rows,cols", [(37, 1), (37, 2), (19, 3), (50, 20), (508_428, 256)])
def test_device_mask_equals_numpy_bit_for_bit(seed, step, block, rows, cols):
    for rate in (0.1, 0.5):
        if rows * cols > 10 ** 6 and rate == 0.1:
            continue
        got = device_mask(seed, step, block, rows, cols, rate)
        ref = D.keep_mask(seed, step, block, rows, cols, rate)
        assert np.array_equal(got, ref)
        if rows * cols > 10 ** 6:                              # 7: the dropped fraction of a cfg3-size block
            n = rows * cols
            assert abs((1.0 - got.mean()) - rate) < 6 * math.sqrt(rate * (1 - rate) / n)


def _model(cfg, w, s, rate, seed=0, **kw):
    m = g.GeneralGNN(cfg.output, activation=cfg.activation, hidden=cfg.hidden, message_passing=cfg.message_passing,
                     pre_process=cfg.pre_process, post_process=cfg.post_process, pool=cfg.pool,
                     connectivity=cfg.connectivity, aggregate=cfg.aggregate, dropout=rate, seed=seed, **kw)
    m.build(cfg.in_features)
    m.load_flat(w, s)
    return m


def _labels(head, rows, c, rng):
    if head == "softmax":
        return np.eye(c, dtype=np.float32)[rng.integers(0, c, rows)]
    if head == "sigmoid":
        return (rng.random((rows, c)) > 0.5).astype(np.float32)
    return rng.standard_normal((rows, c)).astype(np.float32)


def step_vs_oracle(cfg, rate, ds, batch_size, head="softmax", weighted=False, ew_kind=None, max_graph_nodes=None,
                   tol=TOL):
    """One fused train step of a dropout model against the float64 restatement with the NumPy masks of that step."""
    from oracle import batching_ref
    graphs = [ds.graph(i) for i in range(batch_size)]
    (xr, (idx, _, _), seg), _ = batching_ref.collate(graphs)
    rows, cols = idx[:, 0], idx[:, 1]
    (x, a, i), _ = next(g.DisjointLoader(ds, batch_size=batch_size, epochs=1, shuffle=False))
    assert np.array_equal(host(a.indices), idx)
    n, B = xr.shape[0], batch_size
    r_out = n if cfg.pool is None else B
    rng = np.random.default_rng(n)
    y = _labels(head, r_out, cfg.output, rng)
    sw = rng.uniform(0.0, 2.0, r_out).astype(np.float32) if weighted else None
    ew = None
    if ew_kind is not None:
        ew = rng.uniform(0.3, 1.5, rows.shape[0]).astype(np.float32)
        a.edge_weight = torch.from_numpy(ew).cuda()
    if max_graph_nodes is not None:
        a.max_graph_nodes = max_graph_nodes
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=21, perturb=True)
    model = _model(cfg, w, s, rate, seed=3, use_edge_weights=ew is not None)
    step = model.dropout_step
    loss = LOSS[head]() if head in LOSS else None
    loss_acc, probs = model.train_step_grads((x, a, i), torch.from_numpy(y).cuda(), loss=loss,
                                             sample_weight=None if sw is None else torch.from_numpy(sw).cuda())
    masks = D.model_masks(specs, cfg, n, r_out, rate, dropout_seed(3, 0), step)
    branches = gpu_prelu_branches(model, cfg, n, B)
    ref = O1.loss_and_grads(cfg, specs, w, s, xr, rows, cols, seg, y, B, masks=masks, rate=rate,
                            loss=head if head in LOSS else None, sample_weight=sw, prelu_branch=branches, edge_weight=ew)
    got = host(loss_acc)
    assert abs(got[0] - ref["loss"]) < tol * max(abs(ref["loss"]), 1e-3), (got[0], ref["loss"])
    assert rel_err(host(model.state), ref["new_state"]) < tol
    if head == "softmax":
        z = ref["logits"]
        e = np.exp(z - z.max(1, keepdims=True))
        assert rel_err(host(probs), e / e.sum(1, keepdims=True)) < tol
    errs = grad_errors(host(model.grads), ref["grads"], cfg)
    bad = {k: v for k, v in errs.items() if v > tol * (2.0 if k == "pool.attn_kernel" else 1.0)}
    assert not bad, f"gradient tensors out of tolerance: {bad}"
    return model, (x, a, i), y


@pytest.fixture(scope="module")
def small_ds():
    return synthetic.make_dataset(8, seed=3, n_mean=60, deg=8, n_feat=12)


@pytest.mark.parametrize("rate", [0.1, 0.5])
@pytest.mark.parametrize("pool", ["sum", "avg", "attn_sum", None])
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_train_step_matches_float64_pools_and_connectivity(small_ds, rate, pool, connectivity):
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=20, message_passing=3, connectivity=connectivity,
                    pool=pool)
    step_vs_oracle(cfg, rate, small_ds, 8)


@pytest.mark.parametrize("aggregate,connectivity", [("sum", "cat"), ("mean", "cat"), ("mean", "sum"), ("max", "cat"),
                                                    ("max", None)])
@pytest.mark.parametrize("weights", [None, "asym"])
@pytest.mark.parametrize("hidden", [8, 256])
def test_train_step_matches_float64_aggregations(small_ds, aggregate, connectivity, weights, hidden):
    """max: dropped zeros tie often; the tie-sharing gradient must split them as the float64 restatement does."""
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=hidden, message_passing=3,
                    connectivity=connectivity, aggregate=aggregate)
    step_vs_oracle(cfg, 0.5, small_ds, 8, ew_kind=weights, tol=2 * TOL)


@pytest.mark.parametrize("head", ["softmax", "sigmoid", "mse"])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("pool", ["sum", None])
def test_train_step_matches_float64_heads(small_ds, head, weighted, pool):
    act = head if head in ("softmax", "sigmoid") else None
    cfg = GNNConfig(in_features=12, output=3, activation=act, hidden=20, message_passing=2, pool=pool)
    step_vs_oracle(cfg, 0.3, small_ds, 8, head=head, weighted=weighted)


def test_train_step_matches_float64_on_the_global_memory_and_oversized_paths():
    ds = synthetic.make_dataset(6, seed=5, n_mean=300, deg=12, n_feat=16)
    cfg = GNNConfig(in_features=16, output=2, activation="softmax", hidden=64, message_passing=2)
    step_vs_oracle(cfg, 0.5, ds, 6, max_graph_nodes=0)                  # no slab: the global-memory row-block kernel
    big = synthetic.make_dataset(2, seed=6, n_mean=5000, deg=32, n_feat=16)
    step_vs_oracle(cfg, 0.5, big, 2, tol=2 * TOL)                        # cfg5-shape graphs: the slab kernel's oversized path


def test_train_step_matches_float64_on_a_cfg2_size_batch():
    ds = synthetic.make_dataset(64, seed=7, n_mean=500, deg=12, n_feat=32)
    cfg = GNNConfig(in_features=32, output=2, activation="softmax", hidden=256, message_passing=4)
    step_vs_oracle(cfg, 0.1, ds, 64, tol=2 * TOL)


def _plain_step(rate, step=None, seed=3):
    ds = synthetic.make_dataset(6, seed=11, n_mean=90, deg=10, n_feat=8)
    (x, a, i), y = next(g.DisjointLoader(ds, batch_size=6, epochs=1, shuffle=False))
    cfg = GNNConfig(in_features=8, output=2, activation="softmax", hidden=64, message_passing=2)
    w, s = g.init_params(cfg, seed=5, perturb=True)
    m = _model(cfg, w, s, rate, seed=seed)
    if step is not None:
        m.dropout_step = step
    la, probs = m.train_step_grads((x, a, i), y)
    return m, la.clone(), probs.clone(), (x, a, i), y


def test_seed_and_step_behaviour():
    m1, la1, p1, _, _ = _plain_step(0.5, step=4)
    m2, la2, p2, _, _ = _plain_step(0.5, step=4)
    assert torch.equal(la1, la2) and torch.equal(p1, p2) and torch.equal(m1.grads, m2.grads)
    m3, la3, _, _, _ = _plain_step(0.5, step=5)
    assert not torch.equal(m1.grads, m3.grads)
    assert not np.array_equal(device_mask(7, 4, 0, 100, 64, 0.5), device_mask(7, 5, 0, 100, 64, 0.5))
    tiny = 1e-12                                                   # threshold 0, scale 1.0f: the dropout=0 bits
    m0, la0, p0, _, _ = _plain_step(0.0)
    mt, lat, pt, _, _ = _plain_step(tiny)
    assert torch.equal(la0, lat) and torch.equal(p0, pt) and torch.equal(m0.grads, mt.grads) and torch.equal(m0.state, mt.state)


def test_inference_is_the_identity():
    m, _, _, inputs, _ = _plain_step(0.5)
    plain = _model(m.cfg, host(m.params), host(m.state), 0.0)
    assert torch.equal(m(inputs, training=False), plain(inputs, training=False))


def test_tape_route_equals_the_fused_step():
    fused, la, probs, inputs, y = _plain_step(0.5, step=2)
    w, s = g.init_params(fused.cfg, seed=5, perturb=True)
    taped = _model(fused.cfg, w, s, 0.5, seed=3)
    taped.dropout_step = 2
    with g.GradientTape() as tape:
        pred = taped(inputs, training=True)
        loss = g.CategoricalCrossentropy()(y, pred)
    tape.gradient(loss, taped.trainable_variables)
    assert taped.dropout_step == 3
    assert torch.equal(probs, pred) and torch.equal(fused.grads, taped.grads) and torch.equal(fused.state, taped.state)


@pytest.mark.parametrize("sync_bn", [False, True])
def test_two_data_parallel_ranks_draw_different_masks_and_keep_identical_parameters(sync_bn):
    """Two ranks as two host threads on this GPU (NCCL cannot run two ranks on one device): each trains its shard with
    its rank's mask key (what DataParallelTrainer sets), the gradients are summed, and one optimizer step runs on each.
    The masks differ; the parameters stay bit-identical step after step, also with synchronised BatchNorm."""
    ds = synthetic.make_dataset(8, seed=3, n_mean=60, deg=8, n_feat=12)
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=32, message_passing=2)
    w, s = g.init_params(cfg, seed=1, perturb=True)
    models = [_model(cfg, w, s, 0.4, seed=7) for _ in range(2)]
    opts = [g.optimizers.SGD(learning_rate=0.05) for _ in range(2)]
    for r, m in enumerate(models):
        m.dropout_rank = r
    assert dropout_seed(7, 0) != dropout_seed(7, 1)
    assert not np.array_equal(device_mask(dropout_seed(7, 0), 0, 0, 40, 32, 0.4),
                              device_mask(dropout_seed(7, 1), 0, 0, 40, 32, 0.4))
    shards = [(0, 5), (5, 8)]
    barrier = threading.Barrier(2)
    pending = [None, None]

    def view(model, ptr, n):
        off = ptr - model._ws.data_ptr()
        return model._ws[off:off + 8 * n].view(torch.float64)

    def worker(r, errors):
        try:
            torch.cuda.set_device(0)
            stream = torch.cuda.Stream()
            with torch.cuda.stream(stream):
                lo, hi = shards[r]
                ids = np.arange(lo, hi, dtype=np.int64)
                x, a, seg, y = g.data.DeviceGraphStore(ds).batch(torch.from_numpy(ids).cuda(), ids)

                def allreduce(ptr, n, _stream):
                    stream.synchronize()
                    pending[r] = (ptr, n)
                    barrier.wait()
                    total = view(models[r], *pending[r]) + view(models[1 - r], *pending[1 - r])
                    stream.synchronize()
                    barrier.wait()
                    view(models[r], *pending[r]).copy_(total)

                if sync_bn:
                    _lib.set_allreduce_hook(allreduce, 2)
                try:
                    models[r].train_step_grads([x, a, seg], y, grad_scale=1.0 / 8)
                finally:
                    if sync_bn:
                        _lib.set_allreduce_hook(None)
                stream.synchronize()
        except Exception as e:
            errors.append(e)
            barrier.abort()

    for _ in range(4):
        errors = []
        threads = [threading.Thread(target=worker, args=(r, errors)) for r in range(2)]
        [t.start() for t in threads]
        [t.join(120) for t in threads]
        assert not errors, errors
        total = models[0].grads + models[1].grads                  # the flat gradient all-reduce
        for m, opt in zip(models, opts):
            m.grads.copy_(total)
            opt.apply_flat(m.params, m.grads)
        torch.cuda.synchronize()
        assert torch.equal(models[0].params, models[1].params)
        if sync_bn:
            assert torch.equal(models[0].state, models[1].state)
    assert models[0].dropout_step == models[1].dropout_step == 4


def test_running_loop_with_dropout_allocates_nothing():
    ds = synthetic.make_dataset(96, seed=3, n_mean=120, deg=10, n_feat=16)
    model = g.GeneralGNN(2, activation="softmax", hidden=64, message_passing=2, seed=0, dropout=0.3)
    model.build(16)
    loader = g.DisjointLoader(ds, batch_size=24, epochs=None, shuffle=False)
    opt = g.optimizers.SGD(learning_rate=0.01)

    def step():
        (x, a, i), y = next(loader)
        model.train_step_grads((x, a, i), y)
        opt.apply_flat(model.params, model.grads)
    for _ in range(16):
        step()
    torch.cuda.synchronize()
    before = torch.cuda.memory_stats().get("num_device_alloc", 0)
    for _ in range(24):
        step()
    torch.cuda.synchronize()
    assert torch.cuda.memory_stats().get("num_device_alloc", 0) == before
