"""GPU tests of node-level training: the node-label gather of every store path, the grid-wide cross-entropy against
float64 and the single-block kernel, the GeneralGNN(pool=None) train step / inference / GradientTape route / evaluate()
against the float64 restatement, and the data-parallel step scaled by nodes."""
import os
import socket

import numpy as np
import pytest
import scipy.sparse as sp

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import _lib, ops, synthetic
from gcn_string_b200.data import Graph
from gcn_string_b200.distributed import balanced_shard
from gcn_string_b200.params import GNNConfig, block_specs
from oracle import batching_ref, model_ref_np as O1, model_ref_torch as O2

from conftest import rel_err
from test_model_gpu import TOL, gpu_prelu_branches, grad_errors, host, make_model

pytestmark = pytest.mark.gpu
THRESHOLD = 65536            # rows up to which gcs_softmax_xent_ws runs the single-block kernel


# ---------------------------------------------------------------- node-label gather
def _node_dataset(c, seed=0):
    """Graphs of 0, 1 and up to 40 nodes with random [n, c] labels (no two rows alike)."""
    rng = np.random.default_rng(seed)
    sizes = [5, 0, 1, 17, 1, 0, 40, 3, 9, 1, 22, 6, 0, 13]
    graphs = []
    for n in sizes:
        a = sp.random(n, n, density=0.2, random_state=int(rng.integers(1 << 30)), format="csr") if n else sp.csr_matrix((0, 0))
        a = ((a + a.T + sp.eye(n)) > 0).astype(np.float32)
        graphs.append(Graph(x=rng.random((n, 6)).astype(np.float32), a=a, y=rng.standard_normal((n, c)).astype(np.float32)))
    return graphs


STORES = {"device": dict(), "host_slices": dict(device_resident=False), "host_staged": dict(device_resident=False),
          "device_gather": dict(device_resident=False, device_gather=True), "zero_copy": dict(device_resident=False, zero_copy=True)}


@pytest.mark.parametrize("store", list(STORES))
@pytest.mark.parametrize("c", [1, 2, 3, 64])
def test_node_labels_of_shuffled_batches_equal_vstack(store, c):
    graphs = _node_dataset(c, seed=c)
    shuffle = store != "host_slices"                       # consecutive ids take the sliced-upload path
    loader = g.DisjointLoader(graphs, node_level=True, batch_size=5, epochs=2, shuffle=shuffle, **STORES[store])
    np.random.seed(100 + c)                                # the loader shuffles with the global NumPy RNG
    replay = np.random.RandomState(100 + c)
    order = np.arange(len(graphs))
    seen = 0
    for epoch in range(2):
        if shuffle:
            replay.shuffle(order)
        for b0 in range(0, len(graphs), 5):
            ids = order[b0:b0 + 5].copy()
            (x, a, i), y = next(loader)
            ref_y = np.vstack([graphs[k].y for k in ids])
            assert tuple(y.shape) == ref_y.shape and y.dtype == torch.float32 and y.is_cuda
            assert np.array_equal(host(y), ref_y)                        # bit for bit
            assert np.array_equal(host(x), np.vstack([graphs[k].x for k in ids]))
            assert a.global_batch_nodes == ref_y.shape[0] and a.global_batch_graphs == len(ids)
            seen += 1
    assert seen == 2 * len(loader)


@pytest.mark.parametrize("world", [2, 3])
def test_rank_shards_balanced_by_nnz_carry_their_node_labels(world):
    graphs = _node_dataset(2, seed=5)
    packed = synthetic.pack_graphs(graphs, node_level=True)
    cost = packed.n_edges + 4 * packed.n_nodes
    per_rank = []
    for r in range(world):
        loader = g.DisjointLoader(packed, node_level=True, batch_size=9, epochs=1, shuffle=False, rank=r,
                                  world_size=world, balance="nnz")
        out = []
        for b0 in range(0, len(graphs), 9):
            ids = np.arange(b0, min(b0 + 9, len(graphs)))
            if ids.shape[0] < world:
                continue
            mine = balanced_shard(ids, cost[ids], r, world)
            (x, a, i), y = next(loader)
            assert np.array_equal(host(y), np.vstack([graphs[k].y for k in mine]))
            out.append((a.global_batch_nodes, int(y.shape[0]), int(packed.n_nodes[ids].sum())))
        per_rank.append(out)
    for step in zip(*per_rank):
        assert len({s[0] for s in step}) == 1                                # the same on every rank
        assert step[0][0] == sum(s[1] for s in step) == step[0][2]           # = the sum over the ranks' shards


# ---------------------------------------------------------------- loss over many rows
def _loss_case(rows, c, seed):
    rng = np.random.default_rng(seed)
    z = (3 * rng.standard_normal((rows, c))).astype(np.float32)
    y = np.zeros((rows, c), np.float32)
    y[np.arange(rows), rng.integers(0, c, rows)] = 1.0
    soft = rng.random(rows) < 0.1
    y[soft] = rng.random((int(soft.sum()), c)).astype(np.float32)          # soft labels, sum != 1
    y[rng.random(rows) < 0.05] = 0.0                                        # rows without a label
    return z, y


def _single_block(logits, y, grad_scale):
    lib = _lib.load()
    b, c = logits.shape
    probs, dl = torch.empty_like(logits), torch.empty_like(logits)
    la = torch.empty(2, device="cuda")
    _lib.check(lib.gcs_softmax_xent(logits.data_ptr(), y.data_ptr(), b, c, probs.data_ptr(), la.data_ptr(), dl.data_ptr(),
                                    grad_scale, _lib.stream_ptr()), "gcs_softmax_xent")
    return probs, la, dl


@pytest.mark.parametrize("rows,c", [(THRESHOLD, 2), (THRESHOLD + 1, 2), (THRESHOLD + 1, 64), (508_428, 2), (508_428, 1),
                                    (508_428, 64), (2_100_001, 2)])
def test_grid_cross_entropy_against_float64_and_the_single_block_kernel(rows, c):
    z, y = _loss_case(rows, c, seed=rows % 1000 + c)
    zt, yt = torch.from_numpy(z).cuda(), torch.from_numpy(y).cuda()
    probs, la, dl = ops.softmax_xent(zt, yt, want_grad=True)
    z64, y64 = z.astype(np.float64), y.astype(np.float64)
    m = z64.max(1, keepdims=True)
    lse = np.log(np.exp(z64 - m).sum(1, keepdims=True)) + m
    loss = float((lse[:, 0] * y64.sum(1) - (y64 * z64).sum(1)).mean())
    acc = float((np.argmax(y, 1) == np.argmax(z, 1)).mean())
    got = host(la)
    assert abs(got[0] - loss) <= 1e-6 * max(1.0, abs(loss)), (got[0], loss)
    assert abs(got[1] - acc) <= 1e-6, (got[1], acc)
    p64 = np.exp(z64 - lse)
    assert np.abs(host(probs) - p64).max() < 1e-6
    assert rel_err(host(dl), (p64 * y64.sum(1, keepdims=True) - y64) / rows) < 1e-5
    # probs / dlogits bit-identical to the single-block kernel; reruns bit-identical
    p1, la1, dl1 = _single_block(zt, yt, 1.0 / rows)
    assert torch.equal(probs, p1) and torch.equal(dl, dl1)
    assert abs(float(la1[0]) - got[0]) <= 1e-6 * max(1.0, abs(loss)) and abs(float(la1[1]) - got[1]) <= 1e-6
    again = ops.softmax_xent(zt, yt, want_grad=True)
    assert torch.equal(again[0], probs) and torch.equal(again[1], la) and torch.equal(again[2], dl)
    if rows <= THRESHOLD:
        assert torch.equal(la, la1)                                         # the single-block kernel itself ran


def test_grid_cross_entropy_probabilities_only_and_argument_errors():
    z, _ = _loss_case(THRESHOLD + 7, 5, seed=3)
    zt = torch.from_numpy(z).cuda()
    probs, la, dl = ops.softmax_xent(zt)
    assert la is None and dl is None
    assert torch.equal(probs, _single_block(zt, torch.zeros_like(zt), 0.0)[0])
    lib = _lib.load()
    la = torch.empty(2, device="cuda")
    st = lib.gcs_softmax_xent_ws(zt.data_ptr(), zt.data_ptr(), zt.shape[0], 5, None, la.data_ptr(), None, 1.0, None, 0,
                                 _lib.stream_ptr())
    assert st == 3                                                          # GCS_ERR_WORKSPACE
    assert lib.gcs_softmax_xent_ws(zt.data_ptr(), None, zt.shape[0], 65, zt.data_ptr(), None, None, 1.0, None, 0,
                                   _lib.stream_ptr()) == 1                 # C > 64


# ---------------------------------------------------------------- whole model against the float64 restatement
def _parity(cfg, w, s, inputs, y, args, tol=TOL):
    model = make_model(cfg, w, s)
    loss_acc, probs = model.train_step_grads(inputs, y)
    n = int(inputs[0].shape[0])
    branches = gpu_prelu_branches(model, cfg, n, int(inputs[1].graph_ptr.shape[0]) - 1)
    ref = O1.loss_and_grads(*args, prelu_branch=branches)
    o2 = O2.loss_and_grads(*args)["grads"]
    got = host(loss_acc)
    assert probs.shape == (n, cfg.output)
    assert abs(got[0] - ref["loss"]) < tol * abs(ref["loss"])
    assert abs(got[1] - ref["metric"]) < 1e-6
    assert rel_err(host(probs), ref["probs"]) < tol
    assert rel_err(host(model.state), ref["new_state"]) < tol
    e_gpu = grad_errors(host(model.grads), ref["grads"], cfg)
    e_o2 = grad_errors(o2, ref["grads"], cfg)
    bad = {k: (v, e_o2[k]) for k, v in e_gpu.items() if v > max(tol, 4 * e_o2[k])}
    assert not bad, f"gradient tensors out of tolerance (gpu err, fp32-cpu err): {bad}"
    # deterministic rerun, then inference on the moving statistics
    g1, p1, la1 = model.grads.clone(), probs.clone(), loss_acc.clone()
    model.load_flat(w, s)
    la2, p2 = model.train_step_grads(inputs, y)
    assert torch.equal(g1, model.grads) and torch.equal(p1, p2) and torch.equal(la1, la2)
    model.load_flat(w, s)
    p_inf, _ = O1.forward(cfg, args[1], w, s, args[4], args[5], args[6], None, None, training=False)
    # on the moving statistics of perturbed parameters the default architecture's node logits reach |z| ~ 100, where the
    # float32 rounding of the logits alone moves the probabilities by ~1e-4: the bound is 1e-5 or 4x the error of the
    # float32 CPU restatement (O2), like the gradients above
    with torch.no_grad():
        z32 = O2.forward(cfg, O2.unpack(args[1], w, s, requires_grad=False), torch.tensor(np.asarray(args[4], np.float32)),
                         torch.tensor(np.asarray(args[5], np.int64)), torch.tensor(np.asarray(args[6], np.int64)), None, 0,
                         False)
    e_o2_inf = rel_err(torch.softmax(z32, 1).numpy(), p_inf)
    err_inf = rel_err(host(model(list(inputs), training=False)), p_inf)
    assert err_inf < max(tol, 4 * e_o2_inf), (err_inf, e_o2_inf)
    return model


def _small_node_ds():
    # the graphs of the session's small_case (same generator arguments), labelled per node
    return synthetic.make_dataset(8, seed=3, n_mean=60, deg=8, n_feat=12, node_level=True)


@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
@pytest.mark.parametrize("hidden", [16, 128])
def test_train_step_and_inference_match_float64(small_case, connectivity, hidden):
    c = small_case
    ds = _small_node_ds()
    assert np.array_equal(ds.x, c["ds"].x)
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=hidden, message_passing=3,
                    connectivity=connectivity, pool=None)
    w, s = g.init_params(cfg, seed=41, perturb=True)
    (x, a, i), y = next(g.DisjointLoader(ds, node_level=True, batch_size=8, epochs=1, shuffle=False))
    assert np.array_equal(host(y), ds.y)
    args = (cfg, block_specs(cfg), w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], None, ds.y, None)
    _parity(cfg, w, s, (x, a, i), y, args)


def _collated(ds, ids):
    """x, COO indices and y (np.vstack of the node labels) of the graphs ``ids``, collated on the host."""
    (xr, (idx, _, _), _), yr = batching_ref.collate([ds.graph(k) for k in ids])
    return xr, idx, yr


def test_default_architecture_train_step():
    ds = synthetic.make_dataset(8, seed=0, n_mean=500, deg=12, n_feat=32, node_level=True)
    xr, idx, _ = _collated(ds, range(8))
    cfg = GNNConfig(in_features=32, output=2, activation="softmax", pool=None)
    w, s = g.init_params(cfg, seed=4, perturb=True)
    (x, a, i), y = next(g.DisjointLoader(ds, node_level=True, batch_size=8, epochs=1, shuffle=False))
    _parity(cfg, w, s, (x, a, i), y, (cfg, block_specs(cfg), w, s, xr, idx[:, 0], idx[:, 1], None, ds.y, None))


@pytest.fixture(scope="module")
def big_batch():
    """One batch of > 65 536 nodes: the grid-wide loss kernel runs inside the fused step."""
    ds = synthetic.make_dataset(720, seed=2, n_mean=100, deg=8, n_feat=8, node_level=True)
    assert int(ds.node_off[-1]) > 70_000
    xr, idx, _ = _collated(ds, range(720))
    return ds, xr, idx


def test_train_step_above_the_loss_threshold(big_batch):
    ds, xr, idx = big_batch
    cfg = GNNConfig(in_features=8, output=2, activation="softmax", hidden=32, message_passing=2, pool=None)
    w, s = g.init_params(cfg, seed=6, perturb=True)
    (x, a, i), y = next(g.DisjointLoader(ds, node_level=True, batch_size=720, epochs=1, shuffle=False))
    assert x.shape[0] > THRESHOLD
    _parity(cfg, w, s, (x, a, i), y, (cfg, block_specs(cfg), w, s, xr, idx[:, 0], idx[:, 1], None, ds.y, None))


@pytest.mark.parametrize("big", [False, True])
def test_gradient_tape_route_equals_fused_step(big, big_batch):
    ds = big_batch[0] if big else synthetic.make_dataset(6, seed=11, n_mean=90, deg=10, n_feat=8, node_level=True)
    (x, a, i), y = next(g.DisjointLoader(ds, node_level=True, batch_size=ds.n_graphs, epochs=1, shuffle=False))
    assert (x.shape[0] > THRESHOLD) == big
    models = []
    for _ in range(2):
        m = g.GeneralGNN(2, activation="softmax", hidden=64, message_passing=2, seed=0, pool=None)
        m.build(8)
        w, s = g.init_params(m.cfg, seed=5, perturb=True)
        m.load_flat(w, s)
        models.append(m)
    fused, taped = models
    loss_acc, probs = fused.train_step_grads((x, a, i), y)
    with g.GradientTape() as tape:
        pred = taped((x, a, i), training=True)
        loss = g.CategoricalCrossentropy()(y, pred)
    tape.gradient(loss, taped.trainable_variables)
    assert torch.equal(probs, pred) and torch.equal(loss_acc[0], loss)
    assert torch.equal(fused.grads, taped.grads) and torch.equal(fused.state, taped.state)


def test_evaluate_weights_batches_by_nodes(small_case):
    from gcn_string_b200.evaluate import evaluate
    ds = _small_node_ds()
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=16, message_passing=3, pool=None)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=43, perturb=True)
    model = make_model(cfg, w, s)
    loader = g.DisjointLoader(ds, node_level=True, batch_size=3, epochs=None, shuffle=False)
    (loss, acc), preds = evaluate(model, loader)
    losses, accs, sizes, probs_ref = [], [], [], []
    for b0 in range(0, 8, 3):
        ids = list(range(b0, min(b0 + 3, 8)))
        xr, idx, yr = _collated(ds, ids)
        yr = yr.astype(np.float64)
        probs, cache = O1.forward(cfg, specs, w, s, xr, idx[:, 0], idx[:, 1], None, None, training=False)
        probs_ref.append(probs)
        losses.append(O1.xent_from_logits(cache["logits"], yr)[0])
        accs.append(O1.accuracy(probs, yr))
        sizes.append(yr.shape[0])
    assert len(set(sizes)) > 1                                   # the node weights differ from the graph counts' ratio
    ref_loss = np.average(losses, weights=sizes)
    assert abs(loss - ref_loss) < TOL * abs(ref_loss)
    assert abs(acc - np.average(accs, weights=sizes)) < 1e-6
    assert rel_err(np.concatenate([host(p) for p in preds]), np.concatenate(probs_ref)) < TOL


# ---------------------------------------------------------------- data parallel
def _dp_child(rank, world, port, queue):
    import torch.distributed as dist
    from gcn_string_b200.distributed import DataParallelTrainer
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
        n_graphs = 12 * world + 1                                # unequal shards
        ds = synthetic.make_dataset(n_graphs, seed=11, n_mean=200, deg=10, n_feat=16, node_level=True)

        def model():
            m = g.GeneralGNN(2, activation="softmax", hidden=64, message_passing=2, seed=0, pool=None)
            m.build(16)
            return m

        m = model()
        w0 = m.params.clone()
        loader = g.DisjointLoader(ds, node_level=True, batch_size=n_graphs, epochs=1, shuffle=False, symmetric=True,
                                  rank=rank, world_size=world, balance="nnz")
        (x, a, i), y = next(loader)
        trainer = DataParallelTrainer(m, g.optimizers.SGD(learning_rate=0.02), native_comm=True, sync_bn=True)
        trainer.train_step((x, a, i), y)
        torch.cuda.synchronize()
        gathered = [torch.empty_like(m.params) for _ in range(world)]
        dist.all_gather(gathered, m.params)
        same = all(torch.equal(gathered[0], t) for t in gathered[1:])
        diff = None
        if rank == 0:                                            # one single-GPU step on the union batch
            u = model()
            (xu, au, iu), yu = next(g.DisjointLoader(ds, node_level=True, batch_size=n_graphs, epochs=1, shuffle=False,
                                                     symmetric=True))
            u.train_step_grads((xu, au, iu), yu)
            expect = w0 - 0.02 * u.grads
            diff = float((m.params - expect).abs().max() / (u.grads.abs().max() * 0.02))
        dist.barrier()
        dist.destroy_process_group()
        queue.put((rank, same, diff, None))
    except Exception as e:                                    # reported to the parent
        queue.put((rank, False, None, repr(e)))


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_data_parallel_node_level_step_equals_one_step_on_the_union():
    """native_comm + sync_bn, shards of unequal node counts: every rank's parameters are bit-identical, and equal one
    single-GPU step on the union batch (gradient scaled by 1 / global_batch_nodes)."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    world = 2
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    queue = ctx.Queue()
    procs = [ctx.Process(target=_dp_child, args=(r, world, port, queue)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        results = sorted(queue.get(timeout=300) for _ in range(world))
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
                p.join()
    assert all(r[3] is None for r in results), results
    assert all(r[1] for r in results)
    assert results[0][2] < 1e-5, results[0][2]
