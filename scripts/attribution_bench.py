"""Cost of residue / contact attributions (GradientTape.watch on x and the edge weights) on one GPU.

    python scripts/attribution_bench.py [--steps 20] [--warmup 5] [--reps 3] [--out FILE]

Reports, as one JSON line (also written to --out), at the cfg3 per-GPU shape (1024 synthetic E. coli-shaped graphs,
~508 k nodes, F 32, hidden 256, 4 GeneralConv layers, 'cat', softmax C = 2, use_edge_weights=True with all-ones
weights):
  * ms per call, alternated in one process after warm-up, median and spread (max - min) over --reps rounds: the plain
    inference forward, the inference-mode attribution (attribution forward + input-gradient backward for dx and the
    edge weights), the training-mode attribution, and the train step (train_step_grads + SGD);
  * the per-op device times (the library's op timer) of one inference-mode attribution, in a pass of its own:
    edge_grad (one launch per GeneralConv layer), linear_bwd_input_x (dX of the first dense block) and
    bn_prelu_bwd_frozen, with the bytes each must move and the copy-bandwidth time of those bytes;
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


def copy_gbps(torch, nbytes=1 << 30, iters=20):
    """Device-to-device copy bandwidth (read + write bytes per second) on a buffer larger than L2."""
    src = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    ms = time_calls(torch, lambda: dst.copy_(src), iters)
    return 2 * nbytes / (ms * 1e-3) / 1e9


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
    from gcn_string_b200 import _lib, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("attribution_bench needs a CUDA device")
    info = gpu_info()
    ds = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=N_DEG, n_feat=N_FEAT)
    (x, a, i), y = next(g.DisjointLoader(ds, batch_size=args.graphs, epochs=1, shuffle=False, symmetric=True))
    a.edge_weight = torch.ones(a.nnz, dtype=torch.float32, device="cuda")
    model = g.GeneralGNN(2, activation="softmax", hidden=HIDDEN, message_passing=LAYERS, seed=0, use_edge_weights=True)
    model.build(N_FEAT)
    opt = g.optimizers.SGD(learning_rate=0.0)
    og = torch.zeros(args.graphs, 2, device="cuda")
    og[:, 1] = 1.0

    def attr(training):
        with g.GradientTape() as tape:
            tape.watch(x)
            tape.watch(a)
            pred = model((x, a, i), training=training)
        return tape.gradient(pred, [x, a], output_gradients=og)

    calls = {
        "inference_forward": lambda: model((x, a, i), training=False),
        "attribution_inference": lambda: attr(False),
        "attribution_training": lambda: attr(True),
        "train_step": lambda: (model.train_step_grads((x, a, i), y), opt.apply_flat(model.params, model.grads)),
    }
    for f in calls.values():
        for _ in range(args.warmup):
            f()
    torch.cuda.synchronize()
    per = {k: [] for k in calls}
    for _ in range(args.reps):
        for k, f in calls.items():
            per[k].append(time_calls(torch, f, args.steps))
    torch.cuda.synchronize()
    _lib.profile_begin()
    attr(False)
    torch.cuda.synchronize()
    ops = {k: (v[0], round(v[1], 4)) for k, v in sorted(_lib.profile_end().items())}
    n, nnz, H, L = int(x.shape[0]), int(a.nnz), HIDDEN, LAYERS
    bw = copy_gbps(torch)
    # bytes each kernel must move at least: edge_grad per layer reads dZ and the transformed rows once (N x H each, as
    # a forward aggregation does) and writes nnz; dX reads dh_0 [N, H] and writes [N, F]; the frozen BatchNorm backward
    # of a node-level block reads da and h and writes dh, [N, H] each
    need = {"edge_grad_per_layer": 4 * (2 * n * H + 2 * nnz), "linear_bwd_input_x": 4 * (n * H + n * N_FEAT),
            "bn_prelu_bwd_frozen_per_node_block": 4 * 3 * n * H}
    kernels = {}
    for label, key, count in (("edge_grad", "edge_grad_per_layer", L), ("linear_bwd_input_x", "linear_bwd_input_x", 1)):
        if label in ops:
            ms = ops[label][1] / max(ops[label][0], 1)
            kernels[key] = {"ms": ms, "bytes": need[key], "copy_bandwidth_ms": need[key] / (bw * 1e9) * 1e3,
                            "launches": ops[label][0]}
    if "spmm_fwd" in ops:
        kernels["forward_aggregation_per_layer_ms"] = ops["spmm_fwd"][1] / max(ops["spmm_fwd"][0], 1)
    line = {
        "gpu": info,
        "copy_bandwidth_GBps": bw,
        "shape": {"graphs": args.graphs, "nodes": n, "nnz": nnz, "hidden": H, "layers": L, "features": N_FEAT},
        "ms_per_call": {k: float(np.median(v)) for k, v in per.items()},
        "ms_per_call_spread": {k: float(max(v) - min(v)) for k, v in per.items()},
        "kernels": kernels,
        "op_ms_one_inference_attribution": ops,
        "notes": ("ms_per_call: CUDA events over --steps calls on one fixed batch, median and max - min of --reps "
                  "rounds, the four calls alternated; attribution_*: the model call under a tape watching x and the "
                  "adjacency plus tape.gradient(pred, [x, a], output_gradients=one-hot class 1); op_ms: the library's "
                  "per-op device timer over one inference-mode attribution, (launches, total ms); copy_bandwidth_ms: "
                  "the kernel's minimum bytes at the measured device-to-device copy rate"),
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
