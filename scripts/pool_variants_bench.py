"""Cost of GeneralGNN(pool='avg' | 'attn_sum') against the default pool='sum' on one GPU, at the cfg3 per-GPU train-step
shape (1024 synthetic E. coli-shaped graphs of ~500 residues, F 32, hidden 256, 4 GeneralConv layers, 'cat').

    python scripts/pool_variants_bench.py [--steps 20] [--warmup 5] [--reps 3] [--out FILE]

Reports, as one JSON line (also written to --out):
  * ms per train step (forward + loss + backward + SGD) from CUDA events, the three pools alternated in one process after
    warm-up, median over --reps rounds;
  * per-op device times of the pool forward / backward from the library's op timer (labels pool_fwd / pool_bwd; a
    separate, profiled pass - the per-step numbers above are taken with the timer off);
  * the pool kernels alone on an [N, Wc] input of the step's shape (2.6 GB: far beyond the 126 MB L2, every pass reads
    HBM): segment_sum_fwd, attention forward and backward, and a device-to-device copy of the same tensor as the
    measured copy peak.  Achieved bytes/s use the algorithmic bytes: forward reads N*Wc*4, backward reads and writes
    N*Wc*4 each (dOut, out, the scores and the kernel are noise), the copy reads and writes N*Wc*4 each;
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
POOLS = ("sum", "avg", "attn_sum")


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
    ap.add_argument("--kernel-iters", type=int, default=20)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, ops, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("pool_variants_bench needs a CUDA device")
    info = gpu_info()
    ds = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=DEG, n_feat=N_FEAT)
    (x, a, i), y = next(g.DisjointLoader(ds, batch_size=args.graphs, epochs=1, shuffle=False, symmetric=True))
    n_nodes = int(x.shape[0])
    models, opt = {}, g.optimizers.SGD(learning_rate=1e-4)
    for pool in POOLS:
        m = g.GeneralGNN(CLASSES, activation="softmax", hidden=HIDDEN, message_passing=LAYERS, pool=pool, seed=0)
        m.build(N_FEAT)
        models[pool] = m

    def step(m):
        m.train_step_grads((x, a, i), y)
        opt.apply_flat(m.params, m.grads)

    for pool in POOLS:
        for _ in range(args.warmup):
            step(models[pool])
    torch.cuda.synchronize()
    per_step = {p: [] for p in POOLS}
    for _ in range(args.reps):
        for pool in POOLS:
            per_step[pool].append(time_calls(torch, lambda: step(models[pool]), args.steps))
    ms = {p: float(np.median(v)) for p, v in per_step.items()}

    per_op = {}
    for pool in POOLS:
        _lib.profile_begin()
        for _ in range(args.steps):
            step(models[pool])
        torch.cuda.synchronize()
        ops_ms = _lib.profile_end()
        per_op[pool] = {k: v[1] / args.steps for k, v in ops_ms.items() if k.startswith("pool")}

    # kernels alone at the step's pool-input shape
    wc = HIDDEN * (LAYERS + 1)
    gp = a.graph_ptr
    X = torch.randn(n_nodes, wc, device="cuda")
    dst = torch.empty_like(X)
    lim = float(np.sqrt(6.0 / (wc + 1)))
    kern = (torch.rand(wc, device="cuda") * 2 - 1) * lim
    out, scores, gstats = ops.attn_sum_pool_fwd(X, kern, gp)
    dout = torch.randn(args.graphs, wc, device="cuda")
    dx = torch.empty_like(X)
    n = args.kernel_iters
    t = {"copy": time_calls(torch, lambda: dst.copy_(X), n),
         "segment_sum_fwd": time_calls(torch, lambda: ops.segment_sum_fwd(X, gp, out=out), n),
         "segment_mean_fwd": time_calls(torch, lambda: ops.segment_mean_fwd(X, gp, out=out), n),
         "attn_sum_pool_fwd": time_calls(torch, lambda: ops.attn_sum_pool_fwd(X, kern, gp, out=out), n),
         "attn_sum_pool_bwd": time_calls(torch, lambda: ops.attn_sum_pool_bwd(dout, X, kern, gp, out, scores, gstats, dx=dx), n)}
    nb = n_nodes * wc * 4
    bytes_ = {"copy": 2 * nb, "segment_sum_fwd": nb, "segment_mean_fwd": nb, "attn_sum_pool_fwd": nb, "attn_sum_pool_bwd": 2 * nb}
    tbs = {k: bytes_[k] / (t[k] * 1e-3) / 1e12 for k in t}
    line = {
        "gpu": info, "shape": {"graphs": args.graphs, "nodes": n_nodes, "nnz": int(a.nnz), "Wc": wc, "hidden": HIDDEN,
                               "layers": LAYERS, "features": N_FEAT},
        "ms_per_step": ms, "ms_per_step_all_rounds": per_step,
        "step_delta_vs_sum_ms": {p: ms[p] - ms["sum"] for p in POOLS},
        "pool_ops_ms_per_step": per_op,
        "kernel_ms": t, "kernel_TBps": tbs,
        "kernel_share_of_copy_peak": {k: tbs[k] / tbs["copy"] for k in t if k != "copy"},
        "attn_fwd_over_segment_sum_fwd": t["attn_sum_pool_fwd"] / t["segment_sum_fwd"],
        "notes": ("ms_per_step: CUDA events over --steps train steps (train_step_grads + SGD), median of --reps rounds with "
                  "the pools alternated; kernel_*: CUDA events over --kernel-iters launches on a 2.6 GB input (no L2 "
                  "reuse); TB/s over algorithmic bytes (forward N*Wc*4 read, backward N*Wc*4 read + N*Wc*4 written, copy "
                  "the same as the backward)"),
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
