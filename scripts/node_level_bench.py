"""Cost of node-level training (GeneralGNN(pool=None), y [N, C] from DisjointLoader(node_level=True)) against the default
graph-level step (pool='sum') on one GPU, at the cfg3 per-GPU train-step shape (1024 synthetic E. coli-shaped graphs of
~500 residues, ~508 k nodes, F 32, hidden 256, 4 GeneralConv layers, 'cat').

    python scripts/node_level_bench.py [--steps 20] [--warmup 5] [--reps 3] [--out FILE]

Reports, as one JSON line (also written to --out):
  * ms per train step (train_step_grads + SGD) from CUDA events on one fixed batch per kind, graph-level and
    node-level alternated in one process after warm-up, median over --reps rounds;
  * the loss kernels alone at N = 508 k rows, C = 2: the single-block gcs_softmax_xent against gcs_softmax_xent_ws
    (which runs the grid kernel above 65 536 rows), CUDA events over --kernel-iters calls each;
  * driver allocations (cudaMalloc calls counted by PyTorch's caching allocator) inside a timed loop of --loop-steps
    node-level steps that draw shuffled batches from the loader (batching + node-label gather + train step + SGD);
  * the GPU's name, power limit and maximum SM clock, read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_MEAN, DEG, N_FEAT, HIDDEN, LAYERS, CLASSES = 500, 12, 32, 256, 4, 2


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def time_calls(torch, fn, n):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-iters", type=int, default=50)
    ap.add_argument("--loop-steps", type=int, default=12)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("node_level_bench needs a CUDA device")
    info = gpu_info()
    lib = _lib.load()
    gl = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=DEG, n_feat=N_FEAT)
    nl = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=DEG, n_feat=N_FEAT, node_level=True)
    batch = {"graph": next(g.DisjointLoader(gl, batch_size=args.graphs, epochs=1, shuffle=False, symmetric=True)),
             "node": next(g.DisjointLoader(nl, batch_size=args.graphs, epochs=1, shuffle=False, node_level=True,
                                           symmetric=True))}
    (x, a, i), _ = batch["node"]
    n_nodes = int(x.shape[0])
    opt = g.optimizers.SGD(learning_rate=1e-4)
    models = {}
    for kind, pool in (("graph", "sum"), ("node", None)):
        m = g.GeneralGNN(CLASSES, activation="softmax", hidden=HIDDEN, message_passing=LAYERS, pool=pool, seed=0)
        m.build(N_FEAT)
        models[kind] = m

    def step(kind):
        inputs, y = batch[kind]
        m = models[kind]
        m.train_step_grads(inputs, y)
        opt.apply_flat(m.params, m.grads)

    for kind in models:
        for _ in range(args.warmup):
            step(kind)
    torch.cuda.synchronize()
    per_step = {k: [] for k in models}
    for _ in range(args.reps):
        for kind in models:
            per_step[kind].append(time_calls(torch, lambda: step(kind), args.steps))
    ms = {k: float(np.median(v)) for k, v in per_step.items()}

    # the loss kernels alone: [N, 2] logits of the node-level step's size
    logits = torch.randn(n_nodes, CLASSES, device="cuda") * 3
    y = torch.nn.functional.one_hot(torch.randint(0, CLASSES, (n_nodes,), device="cuda"), CLASSES).float()
    probs, dl = torch.empty_like(logits), torch.empty_like(logits)
    loss_acc = torch.empty(2, device="cuda")
    ws_bytes = int(lib.gcs_softmax_xent_workspace_bytes(n_nodes, CLASSES))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device="cuda")
    gs = 1.0 / n_nodes
    p = lambda t: t.data_ptr()                                    # noqa: E731
    single = lambda: lib.gcs_softmax_xent(p(logits), p(y), n_nodes, CLASSES, p(probs), p(loss_acc), p(dl), gs,  # noqa: E731
                                          _lib.stream_ptr())
    grid = lambda: lib.gcs_softmax_xent_ws(p(logits), p(y), n_nodes, CLASSES, p(probs), p(loss_acc), p(dl), gs,  # noqa: E731
                                           p(ws), ws_bytes, _lib.stream_ptr())
    kernel_ms = {"single_block": time_calls(torch, single, args.kernel_iters),
                 "grid": time_calls(torch, grid, args.kernel_iters)}

    # driver allocations inside a running node-level loop (shuffled batches from the loader)
    big = synthetic.tile_dataset(nl, 2 * args.graphs)
    loader = g.DisjointLoader(big, batch_size=args.graphs, epochs=None, shuffle=True, node_level=True, symmetric=True)
    m = models["node"]

    def loop_step():
        inputs, yb = next(loader)
        m.train_step_grads(inputs, yb)
        opt.apply_flat(m.params, m.grads)

    for _ in range(args.warmup):
        loop_step()
    torch.cuda.synchronize()
    before = torch.cuda.memory_stats().get("num_device_alloc", 0)
    loop_ms = time_calls(torch, loop_step, args.loop_steps)
    allocs = torch.cuda.memory_stats().get("num_device_alloc", 0) - before

    line = {
        "gpu": info, "shape": {"graphs": args.graphs, "nodes": n_nodes, "nnz": int(a.nnz), "hidden": HIDDEN,
                               "layers": LAYERS, "features": N_FEAT, "classes": CLASSES},
        "ms_per_step": {"graph_level_sum": ms["graph"], "node_level": ms["node"]},
        "ms_per_step_all_rounds": {"graph_level_sum": per_step["graph"], "node_level": per_step["node"]},
        "node_minus_graph_ms": ms["node"] - ms["graph"],
        "loss_kernel_ms": kernel_ms, "loss_single_over_grid": kernel_ms["single_block"] / kernel_ms["grid"],
        "node_loop_ms_per_step": loop_ms, "node_loop_steps": args.loop_steps + 1,
        "driver_allocations_in_node_loop": int(allocs),
        "notes": ("ms_per_step: CUDA events over --steps train steps (train_step_grads + SGD) on one fixed batch per kind, "
                  "median of --reps rounds with the kinds alternated; loss_kernel_ms: CUDA events over --kernel-iters "
                  "calls at N rows x 2 classes (probs, loss, accuracy, dlogits); node loop: loader (shuffled, device "
                  "store) + train step + SGD, cudaMalloc calls counted by torch.cuda.memory_stats()['num_device_alloc']"),
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
