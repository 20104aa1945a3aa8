#!/usr/bin/env python
"""Benchmark of the GeneralGNN hot path (BASELINE.json metric: train graphs/sec and
GCN-layer edges/sec at 1/2/4/8 B200; SpMM HBM GB/s vs peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one full training step on one disjoint batch of 1024 synthetic E. coli-shaped
graphs per GPU (~500 nodes, stored degree ~12, 32-d features; default GeneralGNN: hidden 256,
4 GeneralConv layers, sum aggregation, sum pool, 2 classes): device batching (K0) -> forward
-> categorical cross-entropy -> backward -> [NCCL gradient all-reduce] -> fused SGD.  That is
the per-GPU step of BASELINE.json configs[2] (same shape as configs[1], which is its forward
half; the forward-only rate is reported beside it as `fwd_graphs_per_sec`).  Graphs shard by
graph across ranks (weak scaling: 1024 graphs per GPU per step).

`value`  : graphs/s, dataset resident in HBM, timed with CUDA events, max over ranks.
`e2e`    : the same step through the public loader with the dataset in PINNED HOST memory:
           every step uploads its graphs (H2D) and reads the loss back (D2H) inside the timing.
`roofline`: the aggregation kernel (SpMM fwd), algorithmic bytes / CUDA-event time vs the
           measured HBM peak in MEASURED_PEAKS.json.
`cpu_baseline` / `--impl reference`: the CPU restatement of the reference's op sequence
           (oracle O2, PyTorch-CPU fp32; kind "port" — TensorFlow/Spektral cannot be installed
           here) on the host cores, bounded sample.
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step of the `value` arm
           returned to its caller - {loss, accuracy}, the class probabilities - and the model's gradients,
           parameters and BatchNorm state after it, as DIR/<name>.npy (float32).  The inputs depend on the
           arguments only, so two builds run with the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_GRAPHS = 1024
N_MEAN, DEG, N_FEAT, HIDDEN, LAYERS, CLASSES = 500, 12, 32, 256, 4, 2
WORKLOAD = ("cfg3 per-GPU train step (= cfg2 shape): GeneralGNN hidden 256 x 4 GeneralConv, sum agg, sum pool, "
            "1024 synthetic E.coli-shaped graphs/GPU/step (~500 nodes, deg ~12, 32-d features)")
CPU_SAMPLE_GRAPHS = 32      # BASELINE cfg1: the sample both CPU arms (in-line cpu_baseline and --impl reference) time
WORKLOADS = {
    # name: (graphs per GPU per step, n_mean, deg, hidden, description)
    "cfg3": (1024, 500, 12, 256, WORKLOAD),
    "cfg5": (64, 5000, 32, 512, "cfg5 per-GPU train step: GeneralGNN hidden 512 x 4 GeneralConv, sum agg, sum pool, 64 synthetic "
                               "inter-protein graphs/GPU/step (~5000 residues, deg ~32, 32-d features)"),
}


def _peaks():
    """(HBM GB/s, sustained bf16 TFLOP/s, source) - measured by the driver on this pool, else the recipe's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1400.0))), "measured"
    except Exception:
        return 6650.0, 1400.0, "fallback"


def _ncu_traffic():
    """DRAM bytes per launch of the roofline kernel from the committed ncu --set full capture (or None)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_spmm_slab_ncu.json")) as f:
            d = json.load(f)
        return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"])
    except Exception:
        return None


DUMP_ARRAY_BYTES = 8 << 20      # per array: the five arrays of --dump-outputs stay well inside 64 MB


def dump_outputs(out_dir, arrays):
    """Write every tensor of ``arrays`` as out_dir/<name>.npy in float32.  An array larger than DUMP_ARRAY_BYTES
    (the parameters at hidden >= 512) is replaced by a fixed, seeded sample of its flat elements in index order:
    the same positions in every run, so that two builds still compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        keep = DUMP_ARRAY_BYTES // a.itemsize
        if a.size > keep:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks.mem,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = None

    def mark_begin(self):
        """Start of the timed region: the sampler itself is started earlier (before the warm-up steps), because
        nvidia-smi's start-up (NVML initialisation) stalls kernel launches for tens of milliseconds."""
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def wait_ready(self, timeout=3.0):
        """Block until nvidia-smi has delivered its first line (its initialisation is over)."""
        t = time.perf_counter()
        while self.proc is not None and not self.lines and time.perf_counter() - t < timeout:
            time.sleep(0.01)

    def start(self):
        if os.environ.get("GCS_BENCH_NO_SAMPLER"):        # diagnostic: is a stall in the timed region the sampler's doing?
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", os.environ.get("GCS_BENCH_SAMPLE_MS", "20")],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = [ln for t, ln in self.lines if (self.t0 is None or t >= self.t0) and (self.t1 is None or t <= self.t1 + 0.03)]
        if not lines:                                     # a timed region shorter than one sampling period
            lines = [ln for t, ln in self.lines if self.t0 is None or t >= self.t0] or [ln for _, ln in self.lines[-1:]]
        for ln in lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_rate(n_graphs, steps, warmup, train=True):
    """graphs/s of the CPU restatement (oracle O2) on `n_graphs` graphs of the bench workload."""
    import torch
    import gcn_string_b200 as g
    from gcn_string_b200 import synthetic
    from oracle import model_ref_torch as O2
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    ds = synthetic.make_dataset(n_graphs, seed=0, n_mean=N_MEAN, deg=DEG, n_feat=N_FEAT)
    graphs = [ds.graph(k) for k in range(n_graphs)]
    cfg = g.GNNConfig(in_features=N_FEAT, output=CLASSES, activation="softmax", hidden=HIDDEN, message_passing=LAYERS)
    w, s = g.init_params(cfg, seed=0)
    sec, threads = O2.time_reference_path(cfg, g.block_specs(cfg), w, s, graphs, n_steps=steps, warmup=warmup,
                                          train=train, lr=0.0002, threads=cores)
    return n_graphs / sec, threads, sec, int(ds.n_edges.sum())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n = CPU_SAMPLE_GRAPHS
    rate, threads, sec, nnz = cpu_reference_rate(n, max(1, args.steps), max(1, args.warmup))
    sample = (f"{n} graphs/step of the same workload (host scipy collate + fwd + bwd + SGD, PyTorch-CPU fp32 restatement "
              f"of the reference op sequence; TensorFlow/Spektral not installable here), median of {max(1, args.steps)} steps")
    line = {"impl": "reference", "metric": "train_graphs_per_sec", "value": rate, "unit": "graphs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample_graphs_per_step": n,
                       "same_config_as_gpu_arm": False,
                       "note": "bounded sample: 32 graphs/step (BASELINE cfg1) of the workload whose GPU arm runs 1024 graphs/GPU/step"},
            "cpu_baseline": {"value": rate, "unit": "graphs/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


def _init_dist(torch, dist):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def run_check(args):
    """Multi-GPU correctness of the data-parallel step on real NCCL (bench.py --gpus N --check [--sync-bn]).
    One train step of the default architecture on a global batch of 48 * N graphs sharded through the loader:
      * the parameters after the step are BIT-IDENTICAL on every rank (all-gather + compare);
      * replica-local BatchNorm: they equal (1e-5) the step rank 0 computes alone as the sum over shards of the
        1/global_batch-scaled shard gradients;
      * --sync-bn: they equal (1e-5) ONE single-GPU step on the union batch."""
    import torch
    import torch.distributed as dist
    import gcn_string_b200 as g
    from gcn_string_b200 import synthetic
    from gcn_string_b200.distributed import DataParallelTrainer
    per_gpu = 48
    ds = None
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ds = synthetic.make_dataset(per_gpu * world, seed=11, n_mean=300, deg=DEG, n_feat=N_FEAT)
    rank, world, local = _init_dist(torch, dist)
    lr = 0.02

    def one_step(r, w, sync_bn, native):
        model = g.GeneralGNN(CLASSES, activation="softmax", hidden=HIDDEN, message_passing=LAYERS, seed=0)
        model.build(N_FEAT)
        loader = g.DisjointLoader(ds, batch_size=per_gpu * world, epochs=1, shuffle=False, symmetric=True, rank=r, world_size=w,
                                  balance="nnz" if w > 1 else None)
        (x, a, i), y = next(loader)
        return model, (x, a, i), y

    results = {}
    for native in (True, False):
        model, inputs, y = one_step(rank, world, args.sync_bn, native)
        trainer = DataParallelTrainer(model, g.optimizers.SGD(learning_rate=lr), sync_bn=args.sync_bn, native_comm=native)
        loss_acc, _ = trainer.train_step(inputs, y)
        torch.cuda.synchronize()
        results[native] = model.params.clone()
        if world > 1:
            gathered = [torch.empty_like(model.params) for _ in range(world)]
            dist.all_gather(gathered, model.params)
            same = all(torch.equal(gathered[0], t) for t in gathered[1:])
        else:
            same = True
        results[("same", native)] = same
    ok_bits = results[("same", True)] and results[("same", False)]
    diff_paths = float((results[True] - results[False]).abs().max() / results[False].abs().max())
    ref_diff = None
    if rank == 0:
        base = g.GeneralGNN(CLASSES, activation="softmax", hidden=HIDDEN, message_passing=LAYERS, seed=0)
        base.build(N_FEAT)
        w0 = base.params.clone()
        if args.sync_bn or world == 1:
            loader = g.DisjointLoader(ds, batch_size=per_gpu * world, epochs=1, shuffle=False, symmetric=True)
            (x, a, i), yy = next(loader)
            base.train_step_grads((x, a, i), yy)
            expect = w0 - lr * base.grads
        else:
            total = torch.zeros_like(w0)
            for r in range(world):
                m, inputs, yy = one_step(r, world, False, False)
                m.train_step_grads(inputs, yy, grad_scale=1.0 / (per_gpu * world))
                total += m.grads
            expect = w0 - lr * total
        torch.cuda.synchronize()
        ref_diff = float((results[True] - expect).abs().max() / expect.abs().max())
    if world > 1:
        dist.barrier()
    if rank == 0:
        ok = ok_bits and diff_paths < 1e-5 and ref_diff < 1e-5
        emit({"check": "ok" if ok else "FAILED", "n_gpus": world, "sync_bn": bool(args.sync_bn),
              "params_bit_identical_across_ranks": {"bucketed_nccl_c_abi": results[("same", True)], "torch_distributed": results[("same", False)]},
              "max_rel_diff_bucketed_vs_single_allreduce": diff_paths,
              "max_rel_diff_vs_rank0_recomputation": ref_diff,
              "reference": ("one single-GPU step on the union batch" if (args.sync_bn or world == 1) else
                            "sum over shards of the 1/global_batch-scaled shard gradients, computed by rank 0 alone"),
              "graphs_per_gpu": per_gpu})
    if world > 1:
        dist.destroy_process_group()
    return 0 if rank != 0 or ok else 1


def run_epoch(args):
    """BASELINE.json configs[2] as written: ONE FULL EPOCH over args.epoch synthetic graphs, data-parallel through the
    sharded loader (DisjointLoader(rank, world_size, balance='nnz') + DataParallelTrainer), global batch 1024 * N."""
    import torch
    import torch.distributed as dist
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, synthetic
    from gcn_string_b200.distributed import DataParallelTrainer
    world = int(os.environ.get("WORLD_SIZE", "1"))
    B, n_mean, deg, hidden, workload = WORKLOADS["cfg3"]
    n_total = int(args.epoch)
    unique = min(n_total, max(args.unique_graphs, B))
    ds = synthetic.make_dataset_parallel(unique, seed=0, n_mean=n_mean, deg=deg, n_feat=N_FEAT)
    if unique < n_total:
        ds = synthetic.tile_dataset(ds, n_total)
    rank, world, local = _init_dist(torch, dist)
    lib = _lib.load()
    sched = g.optimizers.schedules.PiecewiseConstantDecay([0, 1], [0.02, 0.002, 0.0002])
    np.random.seed(4321)
    loader = g.DisjointLoader(ds, batch_size=B * world, epochs=1, shuffle=True, symmetric=True, rank=rank, world_size=world,
                              balance="nnz" if world > 1 else None)
    model = g.GeneralGNN(CLASSES, activation="softmax", hidden=hidden, message_passing=LAYERS, seed=0)
    model.build(N_FEAT)
    trainer = DataParallelTrainer(model, g.optimizers.SGD(learning_rate=sched), sync_bn=args.sync_bn, native_comm=not args.torch_allreduce)
    # warm-up on a throw-away loader over the first batches (allocator, workspace, NCCL channels); the epoch itself is timed whole
    warm = g.DisjointLoader(ds, batch_size=B * world, epochs=1, shuffle=False, symmetric=True, rank=rank, world_size=world,
                            balance="nnz" if world > 1 else None)
    for _ in range(max(3, args.warmup)):
        (x, a, i), y = next(warm)
        trainer.train_step((x, a, i), y)
    del warm
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_ready()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = lib.gcs_debug_launch_count()
    sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    steps, graphs_mine, loss_acc = 0, 0, None
    for (x, a, i), y in loader:
        loss_acc, _ = trainer.train_step((x, a, i), y)
        steps += 1
        graphs_mine += y.shape[0]
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.mark_end()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    cnt = torch.tensor([graphs_mine], device="cuda", dtype=torch.int64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    launches = lib.gcs_debug_launch_count() - launches0
    if rank == 0:
        clocks = sampler.stop()
        total = int(cnt.item())
        emit({"metric": "train_graphs_per_sec", "value": total / (float(ms.item()) / 1e3), "unit": "graphs/s", "n_gpus": world,
              "steps": steps, "warmup": max(3, args.warmup), "ms_per_step": float(ms.item()) / max(steps, 1), "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
              "config": {"workload": f"cfg3 as written: one full training epoch over {n_total} synthetic E.coli-shaped graphs "
                                     f"({unique} unique, repeated), GeneralGNN hidden 256 x 4, global batch {B * world} = 1024 graphs/GPU/step, "
                                     f"sharded by DisjointLoader(rank, world_size, balance='nnz'), DataParallelTrainer",
                         "epoch_graphs": total, "epoch_ms": float(ms.item()), "dataset": "resident in HBM on every rank; batches "
                         "reshuffled (np.random permutation of the epoch), device batching per step",
                         "l2": "working set per step far exceeds the 126 MB L2"},
              "gpu_launches": int(launches), "clocks": clocks,
              "final_loss": float(loss_acc[0]) if loss_acc is not None else None})
    if world > 1:
        dist.destroy_process_group()
    return 0



def run_b200(args):
    import torch
    import torch.distributed as dist
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, synthetic
    from gcn_string_b200.distributed import DataParallelTrainer

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference)")

    K, W = args.steps, args.warmup
    B, n_mean, deg, hidden, workload = WORKLOADS[args.workload]
    if args.batch_graphs:
        B = args.batch_graphs
    # ONE dataset, identical on every rank (graph g is seeded by its id), sharded per global batch by the loader:
    # rank r of `world` takes its work-balanced part (balance='nnz') of every global batch of B * world graphs.
    # Per-GPU work is fixed as N grows (weak scaling).  The pool is `pool_batches` global batches; unique graphs are
    # generated up to --unique-graphs and repeated beyond that (content repeats, the working set per step does not).
    pool = args.pool_batches * B * world
    unique = min(pool, max(args.unique_graphs, B))
    ds = synthetic.make_dataset_parallel(unique, seed=7, n_mean=n_mean, deg=deg, n_feat=N_FEAT)
    if unique < pool:
        ds = synthetic.tile_dataset(ds, pool)
    # CUDA / NCCL only now: the dataset was generated by a forked process pool
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout for the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    np.random.seed(1234)                                            # the same epoch permutations on every rank
    sched = g.optimizers.schedules.PiecewiseConstantDecay([0, 1], [0.02, 0.002, 0.0002])   # gcn.py:321-325
    balance = "nnz" if world > 1 else None

    def make(device_resident, shuffle, **store_kw):
        np.random.seed(1234)
        # host-resident arm without reshuffling: contiguous shards, so that a rank's graphs are ONE slice of the pinned
        # arrays (plain cudaMemcpyAsync per step); everything else is work-balanced
        bal = balance if (device_resident or shuffle) else None
        loader = g.DisjointLoader(ds, batch_size=B * world, epochs=None, shuffle=shuffle, symmetric=True, rank=rank,
                                  world_size=world, balance=bal, device_resident=device_resident, **store_kw)
        model = g.GeneralGNN(CLASSES, activation="softmax", hidden=hidden, message_passing=LAYERS, seed=0)
        model.build(N_FEAT)
        trainer = DataParallelTrainer(model, g.optimizers.SGD(learning_rate=sched), sync_bn=args.sync_bn,
                                      native_comm=not args.torch_allreduce)
        return loader, model, trainer

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_step = {}

    def timed(loop_body, n_steps, tag=None):
        """CUDA-event time of n_steps, max over ranks (ms).  With a tag, an event after every step as well (the per-step
        times go into the JSON line as a diagnostic: a stall of the queue - an allocation, a host hiccup - shows as one
        long step)."""
        # CPython's cyclic collector stays out of the timed region: a full collection walks every tracked object of the
        # process (torch + numpy + scipy: ~10^6) and pauses the launching thread for 50-200 ms, which showed up as one
        # 100-190 ms step in about one of five 10-step regions (measured with and without the clock sampler); a
        # training loop that cares does the same (gc.freeze() after set-up, collections between epochs)
        use_gc = not os.environ.get("GCS_BENCH_KEEP_GC")
        if use_gc:
            gc.collect()
            gc.disable()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(n_steps)] if tag else []
        host = []
        e0.record()
        for k in range(n_steps):
            th = time.perf_counter()
            loop_body()
            if tag:
                marks[k].record()
                host.append(round((time.perf_counter() - th) * 1e3, 3))
        e1.record()
        barrier()
        if use_gc:
            gc.enable()
        if tag:
            per_step[tag + "_host_enqueue"] = host
        if tag:
            prev, out = e0, []
            for m in marks:
                out.append(round(prev.elapsed_time(m), 3))
                prev = m
            per_step[tag] = out
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ------------------------------------------------ device-resident arm (`value`)
    loader, model, trainer = make(True, True)
    stats = {}

    def step():
        (x, a, i), y = next(loader)
        stats["n"], stats["nnz"] = a.n_rows, a.nnz
        stats["out"] = trainer.train_step((x, a, i), y)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                   # before the warm-up: its start-up must not sit in the timed region
        sampler.wait_ready()
    for _ in range(W):
        step()
    launches0 = lib.gcs_debug_launch_count()
    segs0 = torch.cuda.memory_stats().get("num_device_alloc", 0)
    sampler.mark_begin()
    ms_total = timed(step, K, "value")
    sampler.mark_end()
    per_step["device_allocs_in_timed_region"] = torch.cuda.memory_stats().get("num_device_alloc", 0) - segs0
    launches = lib.gcs_debug_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        loss_acc, probs = stats["out"]
        dump_outputs(args.dump_outputs, {"loss_acc": loss_acc, "probs": probs, "grads": model.grads,
                                         "params": model.params, "bn_state": model.state})
    ms_step = ms_total / K
    value = world * B * K / (ms_total / 1e3)

    # forward-only rate (BASELINE cfg2: inference forward, batch resident in HBM)
    (xf, af, i_f), _yf = next(loader)

    def fwd():
        model((xf, af, i_f), training=False)
    for _ in range(3):
        fwd()
    n_fwd = max(5, K)
    ms_fwd = timed(fwd, n_fwd) / n_fwd

    def fwd_batched():                       # the same with shuffling + device batching of every batch inside the timing
        (x, a, i), y = next(loader)
        model((x, a, i), training=False)
    for _ in range(2):
        fwd_batched()
    ms_fwd_batched = timed(fwd_batched, max(3, K // 2)) / max(3, K // 2)

    # per-op device times of two more steps (CUDA events around every op, same stream)
    _lib.profile_begin()
    step()
    step()
    torch.cuda.synchronize()
    prof = _lib.profile_end()
    n_nodes, nnz = stats["n"], stats["nnz"]
    hbm_peak, tensor_peak, peak_src = _peaks()
    roofline, roofline_tensor, ops_report = None, None, {}
    tot = sum(ms for _, ms in prof.values()) or 1.0
    for label, (cnt, ms) in prof.items():
        ops_report[label] = {"launches_timed": cnt, "ms_per_call": ms / cnt, "share_of_step": ms / tot}
    if "spmm_fwd" in prof:
        cnt, ms = prof["spmm_fwd"]
        t = ms / cnt / 1e3
        alg = 4.0 * n_nodes * hidden * 2 + 4.0 * nnz + 4.0 * (n_nodes + 1)       # SURVEY.md §8d
        ach = alg / t / 1e9
        slab = af.slab_ok()
        roofline = {"kernel": ("spmm_slab_kernel<4, true> (K3, GeneralConv aggregation fwd: per-graph shared-memory slabs, TMA-staged, "
                               "BN+PReLU applied once per element)") if slab else
                              "spmm_rb4_kernel<true> (K3, GeneralConv aggregation fwd, BN+PReLU fused on load; graphs too long for a slab)",
                    "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs)", "traffic": _ncu_traffic() if slab and args.workload == "cfg3" else None,
                    "traffic_source": "profiles/r02_spmm_slab_ncu.json (dram__bytes_read.sum + dram__bytes_write.sum, one launch, cfg2 batch)",
                    "algorithmic_bytes_per_launch": alg, "us_per_launch": t * 1e6,
                    "edges_per_sec": nnz / t, "frac_of_nominal_8TBs": ach / 8000.0}
    # the time-dominant kernels are the dense transforms (error-compensated fp16 split on tcgen05): fp32-equivalent rate of the forward GEMMs
    if "linear_fwd" in prof:
        cnt, ms = prof["linear_fwd"]
        steps_prof = 2
        flops = 2.0 * n_nodes * (N_FEAT * hidden + hidden * hidden + hidden * hidden * sum(range(1, LAYERS + 1)))
        t = ms / steps_prof / 1e3
        ach = flops / t / 1e12
        roofline_tensor = {"kernel": "linear_tc_pair_kernel<f16> (K1, forward dense transforms; 3 fp16 tcgen05 MMAs per fp32 "
                                     "product: hi*hi + hi*lo + lo*hi of fp16-split operands)",
                           "bound": "tensor", "achieved": ach, "achieved_executed_f16": 3.0 * ach, "peak": tensor_peak,
                           "unit": "TFLOP/s", "frac": ach / tensor_peak, "frac_executed_f16": 3.0 * ach / tensor_peak,
                           "peak_source": peak_src + " (MEASURED_PEAKS.json bf16_tflops_sustained: kind::f16 runs at the bf16 "
                                          "rate; sustained figure, the GEMMs run back to back under the power cap)",
                           "flops_per_step_fwd": flops, "ms_per_step_fwd_gemms": t * 1e3,
                           "note": "frac = fp32-equivalent flops / peak; frac_executed_f16 counts the three fp16 passes of the "
                                   "error-compensated split as executed work; the kernel is bound by the L2->SM "
                                   "ingest of the raw fp32 activations (32 of 48 KB per 64-wide K block), not by the tensor "
                                   "pipe; the first layer (K=32, tf32 split) and the pooled post-MLP are included in the time"}
    del loader, model, trainer
    torch.cuda.empty_cache()

    # ------------------------------------------------ host-resident arm (`e2e`)
    loader_h, model_h, trainer_h = (make(False, True, device_gather=True) if args.e2e_shuffle else make(False, False))
    io = {"k": 0}
    host_loss = [torch.empty(2, dtype=torch.float32).pin_memory() for _ in range(2)]
    copied = [torch.cuda.Event(), torch.cuda.Event()]

    def step_e2e():
        # every step: the batch's graphs are copied out of pinned host memory (H2D, cudaMemcpyAsync of the slices), the
        # batching kernel and the train step run, {loss, acc} go back to a pinned host buffer (D2H); the host READS the
        # result of step t-1 while step t runs, so that the read does not drain the GPU queue (the copies of all K
        # steps are inside the timed region)
        k = io["k"]
        (x, a, i), y = next(loader_h)
        loss_acc, _ = trainer_h.train_step((x, a, i), y)
        host_loss[k % 2].copy_(loss_acc, non_blocking=True)
        copied[k % 2].record()
        if k > 0:
            copied[(k - 1) % 2].synchronize()
            io["loss"] = float(host_loss[(k - 1) % 2][0])
        io["h2d"] = loader_h.store.h2d_bytes_last
        io["k"] = k + 1
    for _ in range(W):
        step_e2e()
    ms_e2e = timed(step_e2e, K, "e2e")
    e2e_value = world * B * K / (ms_e2e / 1e3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        n = CPU_SAMPLE_GRAPHS
        rate, threads, sec, _ = cpu_reference_rate(n, 3, 1)
        cpu = {"value": rate, "unit": "graphs/s", "cores": threads, "kind": "port",
               "sample": f"{n} graphs/step (BASELINE cfg1) of the same workload through the CPU restatement of the "
                         f"reference op sequence (scipy collate + PyTorch-CPU fp32 fwd/bwd/SGD), median of 3 steps, "
                         f"{sec * 1e3:.0f} ms/step"}
    line = {
        "metric": "train_graphs_per_sec", "value": value, "unit": "graphs/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload, "graphs_per_gpu_per_step": B, "nodes_per_step_per_gpu": n_nodes,
                   "sharding": (f"global batches of {B * world} graphs out of one dataset of {pool} ({unique} unique), rank r takes its "
                                f"work-balanced part of every global batch (DisjointLoader rank/world_size, balance='nnz')") if world > 1
                               else f"one dataset of {pool} graphs ({unique} unique), batches of {B}",
                   "collective": ("torch.distributed all_reduce after the backward" if args.torch_allreduce else
                                  "gcs_model_train_step_dp: NCCL all-reduce in 3 buckets on its own stream during the backward") if world > 1 else None,
                   "nnz_per_step_per_gpu": nnz, "optimizer": "SGD PiecewiseConstantDecay (gcn.py:321-325)",
                   "parallelism": f"graph-sharded data parallel x{world}, one flat NCCL all-reduce (4.26 MB)/step",
                   "l2": "activations per step (cat 2.6 GB, h 0.5 GB/layer) far exceed the 126 MB L2; batches reshuffled "
                         "every step", "bn": ("synchronised BatchNorm statistics (16 extra fp64 all-reduces of <= 3H+1 values per step)"
                          if args.sync_bn and world > 1 else "replica-local BatchNorm statistics")},
        "e2e": {"value": e2e_value, "unit": "graphs/s", "ms_per_step": ms_e2e / K, "h2d_bytes_per_step": int(io["h2d"]),
                "d2h_bytes_per_step": 8, "note": ("dataset in pinned host memory, reshuffled batches; per step: a device kernel gathers "
                         "the batch's packed graphs out of the pinned arrays (H2D), device batching, train step, D2H of {loss, acc} "
                         "into a pinned buffer that the host reads one step later") if args.e2e_shuffle else
                "dataset in pinned host memory, consecutive batches; per step: H2D of the batch's "
                "packed graphs (cudaMemcpyAsync from the pinned arrays), device batching, train step, D2H of {loss, acc} into a "
                "pinned buffer that the host reads one step later"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "roofline_tensor": roofline_tensor,
        "cpu_baseline": cpu,
        "fwd_graphs_per_sec": world * B / (ms_fwd / 1e3), "fwd_ms_per_step": ms_fwd,
        "fwd_with_batching_ms_per_step": ms_fwd_batched,
        "edges_per_sec_train_step": world * nnz / (ms_step / 1e3),
        "ops": ops_report,
        "per_step_ms": per_step,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def _claim_stdout():
    """Keep stdout for the ONE JSON line: everything else any library writes to file descriptor 1 (NCCL's version
    banner lands there on some launches) is sent to stderr for the duration of the run."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch-graphs", type=int, default=0, help="graphs per GPU per step (default: the workload's)")
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS), help="BASELINE.json configs[2] (default) / configs[4]")
    ap.add_argument("--unique-graphs", type=int, default=4096, help="unique synthetic graphs generated; larger pools repeat them")
    ap.add_argument("--torch-allreduce", action="store_true", help="one torch.distributed all-reduce after the backward "
                    "instead of the library's own bucketed NCCL all-reduce (gcs_model_train_step_dp)")
    ap.add_argument("--check", action="store_true", help="multi-GPU correctness: one step, parameters bit-identical on "
                    "every rank; with --sync-bn also equal to one single-GPU step on the union batch")
    ap.add_argument("--epoch", type=int, default=0, metavar="GRAPHS", help="BASELINE cfg3 as written: one full epoch over "
                    "this many graphs (100000) through the sharded loader, reported as graphs/s of the epoch")
    ap.add_argument("--pool-batches", type=int, default=4, help="synthetic pool size in batches per rank")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-shuffle", action="store_true", help="e2e arm with reshuffled batches: the selected graphs are "
                    "gathered out of pinned host memory by a device kernel (gcs_gather_graphs) instead of sliced copies")
    ap.add_argument("--sync-bn", action="store_true", help="all-reduce the BatchNorm statistics too (a G-GPU step then "
                    "equals one step on the union batch); off by default: the gradient all-reduce is the only collective")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed train step as "
                    "DIR/<name>.npy (default benchmark only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.check or args.epoch):
        ap.error("--dump-outputs applies to the default benchmark only")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    if args.check:
        return run_check(args)
    if args.epoch:
        return run_epoch(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
