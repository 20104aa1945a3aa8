"""Cost of sample weights on one GPU.

    python scripts/sample_weight_bench.py [--steps 20] [--warmup 5] [--reps 3] [--out FILE]

Reports, as one JSON line (also written to --out):
  * the weighted loss kernel alone (gcs_weighted_loss, loss_acc and dlogits requested) against the head's unweighted
    entry point at [508 428, 2] and [508 428, 16], for the softmax, sigmoid and MSE heads; CUDA events over
    --kernel-iters calls each;
  * ms per train step (train_step_grads + SGD) at the cfg3 per-GPU shape (1024 synthetic E. coli-shaped graphs, ~508 k
    nodes, F 32, hidden 256, 4 GeneralConv layers, 'cat', softmax C = 2): graph-level (pool='sum') unweighted against
    fractional per-graph weights, and node-level (pool=None, ~508 k output rows) unweighted against a 50 % mask; the
    four alternated in one process, median and spread (max - min) over --reps rounds;
  * the GPU's name, power limit and maximum SM clock, read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from regression_head_bench import DEG as N_DEG, HIDDEN, LAYERS, N_FEAT, N_MEAN, gpu_info, time_calls  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-iters", type=int, default=100)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("sample_weight_bench needs a CUDA device")
    info = gpu_info()
    lib = _lib.load()
    p = lambda t: t.data_ptr() if t is not None else None       # noqa: E731
    st = _lib.stream_ptr

    kernels = []
    for rows, c in ((508_428, 2), (508_428, 16)):
        z = torch.randn(rows, c, device="cuda")
        w = (torch.rand(rows, device="cuda") < 0.5).float()
        dl, probs = torch.empty_like(z), torch.empty_like(z)
        la = torch.empty(2, device="cuda")
        gs = 1.0 / rows
        rec = {"rows": rows, "C": c}
        for name, head, kind, y, plain, plain_ws in (
                ("softmax", 1, 0, torch.nn.functional.one_hot(torch.randint(0, c, (rows,), device="cuda"), c).float(),
                 lambda y, ws, n: lib.gcs_softmax_xent_ws(p(z), p(y), rows, c, p(probs), p(la), p(dl), gs, p(ws), n, st()),
                 lib.gcs_softmax_xent_workspace_bytes),
                ("sigmoid", 2, 0, (torch.rand(rows, c, device="cuda") > 0.5).float(),
                 lambda y, ws, n: lib.gcs_sigmoid_bce(p(z), p(y), rows, c, p(probs), p(la), p(dl), gs, p(ws), n, st()),
                 lib.gcs_sigmoid_bce_workspace_bytes),
                ("mse", 0, 1, torch.randn(rows, c, device="cuda"),
                 lambda y, ws, n: lib.gcs_regression_loss(1, 1.0, p(z), p(y), rows, c, None, p(la), p(dl), gs, p(ws), n,
                                                          st()),
                 lib.gcs_regression_loss_workspace_bytes)):
            nu = int(plain_ws(rows, c))
            wsu = torch.empty(max(nu, 8), dtype=torch.uint8, device="cuda")
            nw = int(lib.gcs_weighted_loss_workspace_bytes(head, rows, c))
            wsw = torch.empty(max(nw, 8), dtype=torch.uint8, device="cuda")
            pr = None if head == 0 else probs
            weighted = lambda: lib.gcs_weighted_loss(head, kind, 1.0, p(z), p(y), p(w), rows, c, p(pr), p(la),  # noqa: E731
                                                     p(dl), gs, p(wsw), nw, st())
            unweighted = lambda: plain(y, wsu, nu)                                           # noqa: E731
            rec[f"{name}_unweighted_ms"] = time_calls(torch, unweighted, args.kernel_iters)
            rec[f"{name}_weighted_ms"] = time_calls(torch, weighted, args.kernel_iters)
        kernels.append(rec)
        del z, w, dl, probs

    gl = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=N_DEG, n_feat=N_FEAT)
    nl = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=N_DEG, n_feat=N_FEAT, node_level=True)
    batches = {"graph": next(g.DisjointLoader(gl, batch_size=args.graphs, epochs=1, shuffle=False, symmetric=True)),
               "node": next(g.DisjointLoader(nl, batch_size=args.graphs, epochs=1, shuffle=False, node_level=True,
                                             symmetric=True))}
    (x, a, _), _ = batches["node"]
    n_nodes = int(x.shape[0])
    rng = np.random.default_rng(0)
    weights = {"graph": torch.from_numpy(rng.uniform(0.0, 2.0, args.graphs).astype(np.float32)).cuda(),
               "node": torch.from_numpy((rng.random(n_nodes) < 0.5).astype(np.float32)).cuda()}
    opt = g.optimizers.SGD(learning_rate=1e-4)
    models = {}
    for level, pool in (("graph", "sum"), ("node", None)):
        for weighted in (False, True):
            m = g.GeneralGNN(2, activation="softmax", hidden=HIDDEN, message_passing=LAYERS, pool=pool, seed=0)
            m.build(N_FEAT)
            models[(level, weighted)] = m

    def step(key):
        m = models[key]
        inputs, y = batches[key[0]]
        m.train_step_grads(inputs, y, sample_weight=weights[key[0]] if key[1] else None)
        opt.apply_flat(m.params, m.grads)

    for key in models:
        for _ in range(args.warmup):
            step(key)
    torch.cuda.synchronize()
    per_step = {key: [] for key in models}
    for _ in range(args.reps):
        for key in models:
            per_step[key].append(time_calls(torch, lambda: step(key), args.steps))
    name = lambda k: f"{k[0]}_{'weighted' if k[1] else 'unweighted'}"      # noqa: E731
    line = {
        "gpu": info,
        "shape": {"graphs": args.graphs, "nodes": n_nodes, "nnz": int(a.nnz), "hidden": HIDDEN, "layers": LAYERS,
                  "features": N_FEAT},
        "loss_kernels": kernels,
        "ms_per_step": {name(k): float(np.median(v)) for k, v in per_step.items()},
        "ms_per_step_spread": {name(k): float(max(v) - min(v)) for k, v in per_step.items()},
        "ms_per_step_all_rounds": {name(k): v for k, v in per_step.items()},
        "notes": ("loss_kernels: CUDA events over --kernel-iters calls, loss_acc and dlogits requested (and probs for the "
                  "softmax and sigmoid heads), half the weights zero; ms_per_step: CUDA events over --steps train steps "
                  "(train_step_grads + SGD) on one fixed batch per level, median and max - min of --reps rounds, the four "
                  "models alternated; graph level: uniform [0, 2) weights per graph, node level: a 50 % mask"),
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
