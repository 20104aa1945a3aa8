"""Cost of GeneralGNN(dropout=rate) on one GPU.

    python scripts/dropout_bench.py [--steps 20] [--warmup 5] [--reps 3] [--out FILE]

Reports, as one JSON line (also written to --out):
  * ms per train step (train_step_grads + SGD) at the cfg3 per-GPU shape (1024 synthetic E. coli-shaped graphs, ~508 k
    nodes, F 32, hidden 256, 4 GeneralConv layers, 'cat', sum aggregation, sum pool, softmax C = 2) at dropout 0, 0.1
    and 0.5, the three models alternated in one process after warm-up, median and spread (max - min) over --reps rounds;
  * the same at the cfg5 per-GPU shape (64 graphs of ~5000 nodes, degree 32, hidden 512) at dropout 0 and 0.5;
  * the per-op device times (the library's op timer) of one cfg3 step at each rate, in a separate pass after the timing;
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


def measure(g, torch, np, batch, feat, hidden, rates, args, profile=False):
    opt = g.optimizers.SGD(learning_rate=1e-4)
    models = {}
    for rate in rates:
        m = g.GeneralGNN(2, activation="softmax", hidden=hidden, message_passing=LAYERS, seed=0, dropout=rate)
        m.build(feat)
        models[rate] = m
    inputs, y = batch

    def step(rate):
        m = models[rate]
        m.train_step_grads(inputs, y)
        opt.apply_flat(m.params, m.grads)

    for rate in rates:
        for _ in range(args.warmup):
            step(rate)
    torch.cuda.synchronize()
    per_step = {rate: [] for rate in rates}
    for _ in range(args.reps):
        for rate in rates:
            per_step[rate].append(time_calls(torch, lambda: step(rate), args.steps))
    out = {"ms_per_step": {str(r): float(np.median(v)) for r, v in per_step.items()},
           "ms_per_step_spread": {str(r): float(max(v) - min(v)) for r, v in per_step.items()},
           "ms_per_step_all_rounds": {str(r): v for r, v in per_step.items()}}
    base = out["ms_per_step"][str(rates[0])]
    out["relative_to_rate0"] = {str(r): out["ms_per_step"][str(r)] / base for r in rates}
    if profile:
        from gcn_string_b200 import _lib
        ops = {}
        for rate in rates:
            torch.cuda.synchronize()
            _lib.profile_begin()
            step(rate)
            torch.cuda.synchronize()
            ops[str(rate)] = {k: round(v[1], 4) for k, v in sorted(_lib.profile_end().items())}
        out["op_ms_one_step"] = ops
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    import gcn_string_b200 as g
    from gcn_string_b200 import synthetic
    if not torch.cuda.is_available():
        raise SystemExit("dropout_bench needs a CUDA device")
    info = gpu_info()
    ds = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=N_DEG, n_feat=N_FEAT)
    batch = next(g.DisjointLoader(ds, batch_size=args.graphs, epochs=1, shuffle=False, symmetric=True))
    (x, a, _), _ = batch
    cfg3 = measure(g, torch, np, batch, N_FEAT, HIDDEN, (0.0, 0.1, 0.5), args, profile=True)
    cfg3["shape"] = {"graphs": args.graphs, "nodes": int(x.shape[0]), "nnz": int(a.nnz), "hidden": HIDDEN,
                     "layers": LAYERS, "features": N_FEAT}
    del batch, ds, x, a
    ds5 = synthetic.make_dataset_parallel(64, seed=0, n_mean=5000, deg=32, n_feat=N_FEAT)
    batch5 = next(g.DisjointLoader(ds5, batch_size=64, epochs=1, shuffle=False, symmetric=True))
    (x5, a5, _), _ = batch5
    cfg5 = measure(g, torch, np, batch5, N_FEAT, 512, (0.0, 0.5), args)
    cfg5["shape"] = {"graphs": 64, "nodes": int(x5.shape[0]), "nnz": int(a5.nnz), "hidden": 512, "layers": LAYERS,
                     "features": N_FEAT}
    line = {
        "gpu": info,
        "cfg3": cfg3,
        "cfg5": cfg5,
        "notes": ("ms_per_step: CUDA events over --steps train steps (train_step_grads + SGD) on one fixed batch, median and "
                  "max - min of --reps rounds, the models of one shape alternated; with dropout > 0 every conv block "
                  "writes a = prelu(dropout(bn(h))) once ('dropout_act') and the aggregation gathers it with the "
                  "transform off; op_ms_one_step: the library's per-op device timer over one step per rate, in a pass "
                  "of its own after the timing"),
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
