"""GPU tests of GeneralGNN(pool='avg' | 'attn_sum'): the segment-mean and attention-pooling kernels against float64,
the fused train step, inference, the GradientTape route and the data-parallel step against the oracle."""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import ops, synthetic
from gcn_string_b200.params import GNNConfig, block_specs, pool_kernel_slice
from oracle import batching_ref, model_ref_np as O1, model_ref_torch as O2

from conftest import rel_err
from test_model_gpu import TOL, _Sparse, gpu_prelu_branches, grad_errors, host, make_model

pytestmark = pytest.mark.gpu
POOLS = ["avg", "attn_sum"]


def _graph_ptr(sizes):
    return torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int32, device="cuda")


def _rows(sizes, W, seed, ld_pad=0, col_off=0):
    """x [N, W] as a view with leading dimension W + ld_pad starting at column col_off, and its float64 copy."""
    n = int(np.sum(sizes))
    rng = np.random.default_rng(seed)
    full = rng.standard_normal((n, W + ld_pad)).astype(np.float32)
    buf = torch.from_numpy(full).cuda()
    x = buf[:, col_off:col_off + W]
    return x, full[:, col_off:col_off + W].astype(np.float64)


# ---------------------------------------------------------------- kernels against float64
@pytest.mark.parametrize("W,ld_pad,col_off", [(1280, 8, 4), (96, 3, 1), (96, 0, 0), (7, 2, 1)])
def test_segment_mean_kernels(W, ld_pad, col_off):
    sizes = [0, 1, 37, 500, 3, 0, 1200, 2]
    x, x64 = _rows(sizes, W, 1, ld_pad, col_off)
    gp = _graph_ptr(sizes)
    seg = np.repeat(np.arange(len(sizes)), sizes)
    out = ops.segment_mean_fwd(x, gp)
    assert rel_err(host(out), O1.segment_mean(x64, seg, len(sizes))) < 1e-6
    assert np.array_equal(host(out)[[0, 5]], np.zeros((2, W), dtype=np.float32))
    dout = torch.randn(len(sizes), W, device="cuda")
    dx = ops.segment_mean_bwd(dout, gp, x.shape[0])
    cnt = np.maximum(np.bincount(seg, minlength=len(sizes)), 1)[:, None]
    assert rel_err(host(dx), (host(dout).astype(np.float64) / cnt)[seg]) < 1e-6


def _attn_check(sizes, W, seed, scale, ld_pad=0, col_off=0, tol=1e-5):
    x, x64 = _rows(sizes, W, seed, ld_pad, col_off)
    rng = np.random.default_rng(seed + 1)
    lim = np.sqrt(6.0 / (W + 1))
    a = (scale * rng.uniform(-lim, lim, W)).astype(np.float32)
    kern = torch.zeros(W + 1, device="cuda")[1:]          # at any float offset, like pool.attn_kernel in the model
    kern.copy_(torch.from_numpy(a))
    gp = _graph_ptr(sizes)
    B = len(sizes)
    seg = np.repeat(np.arange(B), sizes)
    out, scores, gstats = ops.attn_sum_pool_fwd(x, kern, gp)
    ref, ctx = O1.attn_sum_pool(x64, a.astype(np.float64), seg, B)
    e_out = rel_err(host(out), ref)
    assert e_out < tol, e_out
    assert rel_err(host(scores), ctx["scores"]) < 1e-6
    for b in np.flatnonzero(np.asarray(sizes) == 0):
        assert not host(out)[b].any()
    dout = torch.from_numpy(rng.standard_normal((B, W)).astype(np.float32)).cuda()
    dx, dk = ops.attn_sum_pool_bwd(dout, x, kern, gp, out, scores, gstats)
    # the backward as a function of its inputs: float64 arithmetic on the scores and the output the forward returned
    # (near a one-hot softmax X_n . dOut - out . dOut cancels, and the float32 rounding of `out` is the forward's error)
    s64 = host(scores).astype(np.float64)
    mx = np.full(B, -np.inf)
    np.maximum.at(mx, seg, s64)
    e = np.exp(s64 - mx[seg])
    den = np.zeros(B)
    np.add.at(den, seg, e)
    gctx = dict(p=e / (den[seg] + 1e-9), out=host(out).astype(np.float64))
    dx_ref, dk_ref = O1.attn_sum_pool_bwd(x64, a.astype(np.float64), seg, host(dout).astype(np.float64), gctx)
    e_dx, e_dk = rel_err(host(dx), dx_ref), rel_err(host(dk), dk_ref)
    assert e_dx < tol and e_dk < 2 * tol, (e_dx, e_dk)
    # bit-identical run to run
    out2, scores2, gstats2 = ops.attn_sum_pool_fwd(x, kern, gp)
    dx2, dk2 = ops.attn_sum_pool_bwd(dout, x, kern, gp, out2, scores2, gstats2)
    assert torch.equal(out, out2) and torch.equal(gstats, gstats2) and torch.equal(dx, dx2) and torch.equal(dk, dk2)
    # peakedness of the softmax the case exercised: largest weight of the longest graph
    gi = int(np.argmax(sizes))
    return float(ctx["p"][seg == gi].max())


@pytest.mark.parametrize("W,ld_pad,col_off", [(1280, 8, 4), (1280, 1, 1), (96, 0, 0), (96, 3, 1), (7, 2, 1)])
def test_attn_sum_pool_kernels_ragged_graphs(W, ld_pad, col_off):
    """Graph sizes 0 and 1 among longer ones; float4 and scalar paths (a misaligned strided view forces the latter);
    kernels scaled from a near-uniform to a near-one-hot softmax."""
    sizes = [0, 1, 37, 500, 3, 0, 1200, 2]
    peaks = [_attn_check(sizes, W, 3, scale, ld_pad, col_off) for scale in (1e-3, 1.0, 30.0)]
    assert peaks[0] < 2.0 / 1200 and peaks[-1] > 0.5


@pytest.mark.parametrize("sizes", [[120_000], [100_000, 0, 7, 1, 2500]])
def test_attn_sum_pool_kernels_long_graph_split(sizes):
    """A graph of >= 100 k rows (single mode, cfg5-like) is cut into splits whose partials are combined in order."""
    for scale in (1e-2, 1.0, 30.0):
        _attn_check(sizes, 96, 5, scale)
    _attn_check(sizes, 1280 if len(sizes) == 1 else 260, 6, 1.0)


def test_attn_sum_pool_rejects_bad_arguments():
    x = torch.randn(10, 8, device="cuda")
    gp = _graph_ptr([4, 6])
    with pytest.raises(ValueError):
        ops.attn_sum_pool_fwd(x, torch.randn(7, device="cuda"), gp)
    with pytest.raises(NotImplementedError):
        ops.attn_sum_pool_fwd(torch.randn(3, 9000, device="cuda"), torch.randn(9000, device="cuda"), _graph_ptr([3]))


# ---------------------------------------------------------------- whole model against the oracle
def _model_parity(cfg, w, s, inputs, y, args, n_nodes, n_graphs, tol=TOL, with_o2=True):
    model = make_model(cfg, w, s)
    loss_acc, probs = model.train_step_grads(inputs, y)
    branches = gpu_prelu_branches(model, cfg, n_nodes, n_graphs)
    ref = O1.loss_and_grads(*args, prelu_branch=branches)
    o2 = O2.loss_and_grads(*args)["grads"] if with_o2 else None
    assert abs(host(loss_acc)[0] - ref["loss"]) < tol * abs(ref["loss"])
    assert rel_err(host(probs), ref["probs"]) < tol
    assert rel_err(host(model.state), ref["new_state"]) < tol
    # every tensor to 1e-5 (or 4x the float32 CPU restatement's own error), pool.attn_kernel to 2e-5: its gradient
    # sum_n p_n (X_n . dOut - u) X_n nearly cancels, and u = out . dOut is formed from the float32 pooled output, whose
    # rounding the cancellation amplifies (autograd's u = sum_m p_m X_m . dOut shares its rounding with X_n . dOut)
    e_gpu = grad_errors(host(model.grads), ref["grads"], cfg)
    e_o2 = grad_errors(o2, ref["grads"], cfg) if o2 is not None else {}
    bad = {k: (v, e_o2.get(k)) for k, v in e_gpu.items()
           if v > max(tol * (2.0 if k == "pool.attn_kernel" else 1.0), 4 * e_o2.get(k, 0.0))}
    assert not bad, f"gradient tensors out of tolerance (gpu err, fp32-cpu err): {bad}"
    assert ("pool.attn_kernel" in e_gpu) == (pool_kernel_slice(cfg) is not None)
    return model


@pytest.mark.parametrize("pool", POOLS)
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
@pytest.mark.parametrize("hidden", [16, 128])
def test_train_step_and_inference_match_oracle(small_case, pool, connectivity, hidden):
    """Loss, probabilities, BatchNorm state and every gradient tensor (pool.attn_kernel included) of the fused train
    step, then inference, against the float64 oracle; hidden = 128 runs the fp16-split tensor-core GEMMs."""
    c = small_case
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=hidden, message_passing=3,
                    connectivity=connectivity, pool=pool)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=41, perturb=True)
    args = (cfg, specs, w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], c["y"], 8)
    (x, a, i), y = next(g.DisjointLoader(c["ds"], batch_size=8, epochs=1, shuffle=False))
    model = _model_parity(cfg, w, s, (x, a, i), y, args, c["x"].shape[0], 8)
    g1 = model.grads.clone()
    model.load_flat(w, s)
    model.train_step_grads([x, a, i], y)
    assert torch.equal(g1, model.grads)                       # deterministic
    model.load_flat(w, s)
    p_inf, _ = O1.forward(cfg, specs, w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], 8, False)
    assert rel_err(host(model([x, a, i], training=False)), p_inf) < TOL


@pytest.mark.parametrize("pool", POOLS)
@pytest.mark.parametrize("n_graphs,seed", [(8, 0), (32, 1)])
def test_default_architecture_train_step(pool, n_graphs, seed):
    """Hidden 256, 4 GeneralConv layers, F = 32 on 8 and on 32 (BASELINE cfg1) E. coli-shaped graphs."""
    ds = synthetic.make_dataset(n_graphs, seed=seed, n_mean=500, deg=12, n_feat=32)
    (xr, (idx, _, _), seg), yr = batching_ref.collate([ds.graph(k) for k in range(n_graphs)])
    cfg = GNNConfig(in_features=32, output=2, activation="softmax", pool=pool)
    w, s = g.init_params(cfg, seed=4, perturb=True)
    args = (cfg, block_specs(cfg), w, s, xr, idx[:, 0], idx[:, 1], seg, yr, n_graphs)
    (x, a, i), y = next(g.DisjointLoader(ds, batch_size=n_graphs, epochs=1, shuffle=False))
    _model_parity(cfg, w, s, (x, a, i), y, args, xr.shape[0], n_graphs)


@pytest.mark.parametrize("pool", POOLS)
def test_gradient_tape_route_equals_fused_step(pool):
    ds = synthetic.make_dataset(6, seed=11, n_mean=90, deg=10, n_feat=16)
    (x, a, i), y = next(g.DisjointLoader(ds, batch_size=6, epochs=1, shuffle=False))
    models = []
    for _ in range(2):
        m = g.GeneralGNN(2, activation="softmax", hidden=128, message_passing=3, seed=0, pool=pool)
        m.build(16)
        w, s = g.init_params(m.cfg, seed=5, perturb=True)
        m.load_flat(w, s)
        models.append(m)
    fused, taped = models
    loss_acc, probs = fused.train_step_grads((x, a, i), y)
    with g.GradientTape() as tape:
        pred = taped((x, a, i), training=True)
        loss = g.CategoricalCrossentropy()(y, pred)
    grads = tape.gradient(loss, taped.trainable_variables)
    assert torch.equal(probs, pred)
    assert torch.equal(fused.grads, taped.grads) and torch.equal(fused.state, taped.state)
    names = [v.name for v in taped.trainable_variables]
    if pool == "attn_sum":
        assert names[-1] == "pool.attn_kernel" and tuple(grads[-1].shape) == (taped.cfg.cat_width, 1)
        assert float(grads[-1].abs().max()) > 0
    else:
        assert "pool.attn_kernel" not in names


@pytest.mark.parametrize("pool", POOLS)
def test_single_mode_layers_and_evaluate(small_case, pool):
    from gcn_string_b200.evaluate import evaluate
    c = small_case
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=16, message_passing=3, pool=pool)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=43, perturb=True)
    model = make_model(cfg, w, s)
    n = c["x"].shape[0]
    rows, cols = c["idx"][:, 0], c["idx"][:, 1]
    xs = torch.from_numpy(c["x"].astype(np.float32)).cuda()
    a = _Sparse(c["idx"], n)
    one = model([xs, a])                                                   # [x, a]: one graph of all nodes
    ref1, _ = O1.forward(cfg, specs, w, s, c["x"].astype(np.float32), rows, cols, np.zeros(n, dtype=np.int64), 1, False)
    assert one.shape == (1, 2) and rel_err(host(one), ref1) < TOL
    # the pooling layers on their own, disjoint ([x, i]) and single ([x]) mode
    i = torch.from_numpy(c["seg"]).cuda()
    x64 = c["x"].astype(np.float32).astype(np.float64)
    if pool == "avg":
        layer = g.GlobalAvgPool()
        assert rel_err(host(layer([xs, i])), O1.segment_mean(x64, c["seg"], 8)) < 1e-6
        assert rel_err(host(layer([xs])), x64.mean(0, keepdims=True)) < 1e-6
    else:
        layer = g.GlobalAttnSumPool(seed=3)
        out = layer([xs, i])
        k = host(layer.attn_kernel).astype(np.float64)[:, 0]
        assert layer.attn_kernel.shape == (12, 1)
        assert rel_err(host(out), O1.attn_sum_pool(x64, k, c["seg"], 8)[0]) < TOL
        assert rel_err(host(layer(xs)), O1.attn_sum_pool(x64, k, np.zeros(n, dtype=np.int64), 1)[0]) < TOL
    # evaluate(): inference over batches of 3, 3, 2 graphs
    loader = g.DisjointLoader(c["ds"], batch_size=3, epochs=None, shuffle=False)
    (loss, acc), preds = evaluate(model, loader)
    losses, sizes, probs_ref = [], [], []
    for b0 in range(0, 8, 3):
        ids = list(range(b0, min(b0 + 3, 8)))
        (xr, (idx, _, _), seg), yr = batching_ref.collate([c["ds"].graph(k) for k in ids])
        probs, cache = O1.forward(cfg, specs, w, s, xr, idx[:, 0], idx[:, 1], seg, len(ids), training=False)
        probs_ref.append(probs)
        losses.append(O1.xent_from_logits(cache["logits"], yr.astype(np.float64))[0])
        sizes.append(len(ids))
    assert abs(loss - np.average(losses, weights=sizes)) < TOL * abs(np.average(losses, weights=sizes))
    assert rel_err(np.concatenate([host(p) for p in preds]), np.concatenate(probs_ref)) < TOL


# ---------------------------------------------------------------- data parallel
def _dp_child(rank, world, port, queue):
    import torch.distributed as dist
    from gcn_string_b200.distributed import DataParallelTrainer
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
        ds = synthetic.make_dataset(12 * world, seed=11, n_mean=200, deg=10, n_feat=16)

        def model_and_batch(r, w):
            m = g.GeneralGNN(2, activation="softmax", hidden=64, message_passing=2, seed=0, pool="attn_sum")
            m.build(16)
            loader = g.DisjointLoader(ds, batch_size=12 * world, epochs=1, shuffle=False, symmetric=True, rank=r,
                                      world_size=w, balance="nnz" if w > 1 else None)
            return m, next(loader)

        model, ((x, a, i), y) = model_and_batch(rank, world)
        trainer = DataParallelTrainer(model, g.optimizers.SGD(learning_rate=0.02), native_comm=True)
        trainer.train_step((x, a, i), y)
        torch.cuda.synchronize()
        gathered = [torch.empty_like(model.params) for _ in range(world)]
        dist.all_gather(gathered, model.params)
        same = all(torch.equal(gathered[0], t) for t in gathered[1:])
        diff = None
        if rank == 0:
            w0 = None
            total = None
            for r in range(world):
                m, ((xr, ar, ir), yr) = model_and_batch(r, world)
                w0 = m.params.clone()
                m.train_step_grads((xr, ar, ir), yr, grad_scale=1.0 / (12 * world))
                total = m.grads.clone() if total is None else total + m.grads
            expect = w0 - 0.02 * total
            diff = float((model.params - expect).abs().max() / expect.abs().max())
        dist.barrier()
        dist.destroy_process_group()
        queue.put((rank, same, diff, None))
    except Exception as e:                                    # reported to the parent
        queue.put((rank, False, None, repr(e)))


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_data_parallel_step_with_attention_pooling():
    """pool.attn_kernel lies after the last block: its gradient must be inside the all-reduce buckets of
    gcs_model_train_step_dp.  Parameters are bit-identical on every rank and equal what rank 0 computes alone."""
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
