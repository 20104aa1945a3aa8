"""Cost of the optimizer options (momentum, Nesterov, amsgrad, clipping) on one GPU.

    python scripts/optimizer_bench.py [--warmup 50] [--iters 500] [--steps 20] [--reps 3] [--out FILE]

Reports, as one JSON line (also written to --out):
  * the optimizer step alone for {SGD, SGD momentum, Nesterov, Adam, amsgrad} x {no clip, clipvalue, clipnorm,
    global_clipnorm} over the flat buffers of the cfg3 model (hidden 256, 1 064 454 parameters) and of the hidden-512
    model (4 226 054): CUDA events around each of --iters steps after --warmup, median per step.  The buffers fit in
    L2, so this is the step as a training loop sees it (the same parameters updated again and again);
  * ms per train step (train_step_grads + optimizer) at the cfg3 per-GPU shape (1024 synthetic E. coli-shaped graphs,
    ~508 k nodes) with plain SGD and with SGD(momentum=0.9, global_clipnorm=1.0), alternated in one process, median
    and spread (max - min) of --reps rounds of --steps steps;
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

VARIANTS = {"sgd": ("SGD", {}), "momentum": ("SGD", {"momentum": 0.9}),
            "nesterov": ("SGD", {"momentum": 0.9, "nesterov": True}),
            "adam": ("Adam", {}), "amsgrad": ("Adam", {"amsgrad": True})}
CLIPS = {"none": {}, "clipvalue": {"clipvalue": 0.01}, "clipnorm": {"clipnorm": 0.1}, "global_clipnorm": {"global_clipnorm": 1.0}}


def step_ms(torch, fn, warmup, iters):
    """Median of per-step CUDA-event times."""
    for _ in range(warmup):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    torch.cuda.synchronize()
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in ev)
    return t[len(t) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--iters", type=int, default=500)
    ap.add_argument("--graphs", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("optimizer_bench needs a CUDA device")
    info = gpu_info()
    lib = _lib.load()

    steps = {}
    for hidden in (HIDDEN, 512):
        m = g.GeneralGNN(2, activation="softmax", hidden=hidden, message_passing=LAYERS, seed=0)
        m.build(N_FEAT)
        m.grads.copy_(torch.randn_like(m.grads) * 1e-2)
        params0 = m.params.clone()
        rec = {"hidden": hidden, "parameters": int(m.params.numel())}
        for vname, (cls, kw) in VARIANTS.items():
            for cname, ckw in CLIPS.items():
                opt = getattr(g.optimizers, cls)(learning_rate=1e-6, **kw, **ckw)
                variables = m.trainable_variables
                n0 = lib.gcs_debug_launch_count()
                opt.apply_flat(m.params, m.grads, variables=variables)
                launches = lib.gcs_debug_launch_count() - n0
                rec[f"{vname}_{cname}_ms"] = step_ms(
                    torch, lambda: opt.apply_flat(m.params, m.grads, variables=variables), args.warmup, args.iters)
                rec[f"{vname}_{cname}_launches"] = int(launches)
                m.params.copy_(params0)
        steps[f"hidden_{hidden}"] = rec
        del m

    ds = synthetic.make_dataset_parallel(args.graphs, seed=0, n_mean=N_MEAN, deg=N_DEG, n_feat=N_FEAT)
    (x, a, i), y = next(g.DisjointLoader(ds, batch_size=args.graphs, epochs=1, shuffle=False, symmetric=True))
    runs = {}
    for name, kw in (("sgd", {}), ("momentum_global_clipnorm", {"momentum": 0.9, "global_clipnorm": 1.0})):
        mdl = g.GeneralGNN(2, activation="softmax", hidden=HIDDEN, message_passing=LAYERS, seed=0)
        mdl.build(N_FEAT)
        runs[name] = (mdl, g.optimizers.SGD(learning_rate=1e-4, **kw))

    def train(name):
        mdl, opt = runs[name]
        mdl.train_step_grads((x, a, i), y)
        opt.apply_flat(mdl.params, mdl.grads, variables=mdl.trainable_variables)

    for name in runs:
        for _ in range(5):
            train(name)
    torch.cuda.synchronize()
    per_step = {name: [] for name in runs}
    for _ in range(args.reps):
        for name in runs:
            per_step[name].append(time_calls(torch, lambda: train(name), args.steps))
    line = {
        "gpu": info,
        "optimizer_step": steps,
        "train_shape": {"graphs": args.graphs, "nodes": int(x.shape[0]), "nnz": int(a.nnz), "hidden": HIDDEN,
                        "layers": LAYERS, "features": N_FEAT},
        "train_ms_per_step": {k: float(np.median(v)) for k, v in per_step.items()},
        "train_ms_per_step_spread": {k: float(max(v) - min(v)) for k, v in per_step.items()},
        "train_ms_per_step_all_rounds": per_step,
        "notes": ("optimizer_step: median of per-step CUDA-event times over --iters steps after --warmup, gradients "
                  "N(0, 1e-4) so every clip mode fires; launches counted by the library for one step. train: CUDA events "
                  "over --steps train steps (train_step_grads + apply_flat) on one fixed batch, the two optimizers "
                  "alternated, median and max - min of --reps rounds"),
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
