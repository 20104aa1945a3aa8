"""Cost of the regression head (GeneralGNN(activation=None) + MeanSquaredError / Huber) on one GPU.

    python scripts/regression_head_bench.py [--steps 20] [--warmup 5] [--reps 3] [--out FILE]

Reports, as one JSON line (also written to --out):
  * the loss kernels alone: gcs_regression_loss (MSE and Huber) at [1024, 1] and [508 428, C] for C in {1, 2, 16, 64}
    (predictions, loss, mean absolute error and dlogits all requested), with gcs_sigmoid_bce and gcs_softmax_xent_ws
    at the same shapes beside it; CUDA events over --kernel-iters calls each, with the bytes the regression kernel must
    move (16 rows C: predictions and targets read, predictions and dlogits written) over its time.  The [508 428, 64]
    arrays (520 MB) exceed the 126 MB L2; the smaller ones do not;
  * the copy peak: a device-to-device copy of 1 GB, bytes read + written over its time;
  * ms per train step (train_step_grads + SGD) at the cfg3 per-GPU shape (1024 synthetic E. coli-shaped graphs, ~508 k
    nodes, F 32, hidden 256, 4 GeneralConv layers, 'cat'), graph-level (pool='sum') and node-level (pool=None), with
    softmax C = 2, linear MSE C = 1 and linear Huber C = 1 alternated in one process: median and spread (max - min)
    over --reps rounds;
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

N_MEAN, DEG, N_FEAT, HIDDEN, LAYERS = 500, 12, 32, 256, 4


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
    ap.add_argument("--kernel-iters", type=int, default=100)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("regression_head_bench needs a CUDA device")
    info = gpu_info()
    lib = _lib.load()
    p = lambda t: t.data_ptr() if t is not None else None       # noqa: E731

    # copy peak: 1 GB device-to-device, 2 GB moved
    src = torch.empty(1 << 28, device="cuda")
    dst = torch.empty_like(src)
    copy_ms = time_calls(torch, lambda: dst.copy_(src), 20)
    copy_gbs = 2 * src.numel() * 4 / copy_ms / 1e6
    del src, dst

    kernels = []
    for rows, c in ((1024, 1), (508_428, 1), (508_428, 2), (508_428, 16), (508_428, 64)):
        z = torch.randn(rows, c, device="cuda")
        y = torch.randn(rows, c, device="cuda")
        probs, dl = torch.empty_like(z), torch.empty_like(z)
        la = torch.empty(2, device="cuda")
        gs = 1.0 / rows
        moved = 16 * rows * c
        rec = {"rows": rows, "C": c, "bytes_moved": moved}
        ws_b = int(lib.gcs_regression_loss_workspace_bytes(rows, c))
        ws = torch.empty(max(ws_b, 1), dtype=torch.uint8, device="cuda")
        for name, kind in (("mse", 1), ("huber", 3)):
            reg = lambda: lib.gcs_regression_loss(kind, 1.0, p(z), p(y), rows, c, p(probs), p(la), p(dl), gs,  # noqa: E731
                                                  p(ws), ws_b, _lib.stream_ptr())
            ms = time_calls(torch, reg, args.kernel_iters)
            rec[f"{name}_ms"] = ms
            rec[f"{name}_gbs"] = moved / ms / 1e6
            rec[f"{name}_over_copy_peak"] = moved / ms / 1e6 / copy_gbs
        yb = (y > 0).float()
        ws2_b = int(lib.gcs_sigmoid_bce_workspace_bytes(rows, c))
        ws2 = torch.empty(max(ws2_b, 1), dtype=torch.uint8, device="cuda")
        bce = lambda: lib.gcs_sigmoid_bce(p(z), p(yb), rows, c, p(probs), p(la), p(dl), gs, p(ws2), ws2_b,  # noqa: E731
                                          _lib.stream_ptr())
        rec["sigmoid_bce_ms"] = time_calls(torch, bce, args.kernel_iters)
        ws3_b = int(lib.gcs_softmax_xent_workspace_bytes(rows, c))
        ws3 = torch.empty(max(ws3_b, 1), dtype=torch.uint8, device="cuda")
        yo = torch.nn.functional.one_hot(torch.randint(0, c, (rows,), device="cuda"), c).float()
        xent = lambda: lib.gcs_softmax_xent_ws(p(z), p(yo), rows, c, p(probs), p(la), p(dl), gs, p(ws3), ws3_b,  # noqa: E731
                                               _lib.stream_ptr())
        rec["softmax_xent_ws_ms"] = time_calls(torch, xent, args.kernel_iters)
        kernels.append(rec)
        del z, y, yb, yo, probs, dl, ws, ws2, ws3

    gl = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=DEG, n_feat=N_FEAT)
    nl = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=DEG, n_feat=N_FEAT, node_level=True)
    batches = {"graph": next(g.DisjointLoader(gl, batch_size=args.graphs, epochs=1, shuffle=False, symmetric=True)),
               "node": next(g.DisjointLoader(nl, batch_size=args.graphs, epochs=1, shuffle=False, node_level=True,
                                             symmetric=True))}
    (x, a, _), _ = batches["node"]
    n_nodes = int(x.shape[0])
    heads = {"softmax_c2": ("softmax", 2, None), "linear_mse_c1": (None, 1, g.MeanSquaredError()),
             "linear_huber_c1": (None, 1, g.Huber())}
    opt = g.optimizers.SGD(learning_rate=1e-4)
    models, targets, losses = {}, {}, {}
    for level, pool in (("graph", "sum"), ("node", None)):
        inputs, y2 = batches[level]
        for head, (act, c, loss) in heads.items():
            m = g.GeneralGNN(c, activation=act, hidden=HIDDEN, message_passing=LAYERS, pool=pool, seed=0)
            m.build(N_FEAT)
            models[(level, head)] = m
            targets[(level, head)] = y2[:, :c].contiguous() if c < 2 else y2     # one-hot, or its first column
            losses[(level, head)] = loss

    def step(key):
        m = models[key]
        m.train_step_grads(batches[key[0]][0], targets[key], loss=losses[key])
        opt.apply_flat(m.params, m.grads)

    for key in models:
        for _ in range(args.warmup):
            step(key)
    torch.cuda.synchronize()
    per_step = {key: [] for key in models}
    for _ in range(args.reps):
        for key in models:
            per_step[key].append(time_calls(torch, lambda: step(key), args.steps))
    ms = {f"{lv}_{hd}": float(np.median(v)) for (lv, hd), v in per_step.items()}
    spread = {f"{lv}_{hd}": float(max(v) - min(v)) for (lv, hd), v in per_step.items()}

    line = {
        "gpu": info, "copy_peak_gbs": copy_gbs,
        "shape": {"graphs": args.graphs, "nodes": n_nodes, "nnz": int(a.nnz), "hidden": HIDDEN, "layers": LAYERS,
                  "features": N_FEAT},
        "loss_kernels": kernels,
        "ms_per_step": ms,
        "ms_per_step_spread": spread,
        "ms_per_step_all_rounds": {f"{lv}_{hd}": v for (lv, hd), v in per_step.items()},
        "notes": ("loss_kernels: CUDA events over --kernel-iters calls; regression: predictions + loss + MAE + dlogits "
                  "requested, bytes_moved = 16 rows C; sigmoid_bce and softmax_xent_ws at the same shape for reference; "
                  "copy_peak_gbs: 1 GB device-to-device copy, read + written bytes; ms_per_step: CUDA events over "
                  "--steps train steps (train_step_grads + SGD) on one fixed batch per level, median and max - min of "
                  "--reps rounds, the six models alternated; no multi-GPU run"),
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
