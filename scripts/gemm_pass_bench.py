"""Kernel A/B of the fp16-split forward GEMM between two builds of the library, alternated in one process.

    python scripts/gemm_pass_bench.py --base gcn-string_b200/variants/libbase.so [--iters 20] [--out FILE]

Each shape runs base, new, base, new.  Per arm: the GEMM kernels' device time from torch.profiler (CUPTI timestamps,
median over --iters calls; the standalone op in fp16 debug mode also runs a |max| pass over A and the weight split,
which are excluded), CUDA-event time of the whole op, fp32-equivalent TFLOP/s of the kernel, and the L2 -> SM bytes the
kernels must ingest, from the shapes: per CTA, K block of 64 and 256 output columns, 96 KB for 256 x 128 tiles (A
fetched and split once per 128-column tile) and 64 KB for 256-column passes.  The outputs of both arms are compared
on the same inputs.  Inputs are >= 520 MB, far past the 126 MB of L2.
"""
import argparse
import ctypes
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = os.path.join(ROOT, "gcn-string_b200", "libgcnstring_b200.so")
SHAPES = [(508180, 256, k) for k in (256, 512, 768, 1024)] + [(318000, 512, k) for k in (512, 1024, 2048)]
GEMM_KERNELS = ("linear_tc_pair_kernel", "linear_f16_pass256_kernel")


def load(path):
    lib = ctypes.CDLL(path)
    P, I32, I64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    lib.gcs_linear_workspace_bytes.restype = I64
    lib.gcs_linear_workspace_bytes.argtypes = [I64, I32, I32]
    lib.gcs_linear_fwd.restype = I32
    lib.gcs_linear_fwd.argtypes = [P, I64, P, P, P, I64, I64, I32, I32, P, I64, P]
    lib.gcs_debug_set_param.argtypes = [I32, I32]
    lib.gcs_debug_set_gemm_mode.argtypes = [I32]
    lib.gcs_debug_set_param(7, 2)          # fp16 split kernels for every GEMM ...
    lib.gcs_debug_set_gemm_mode(2)         # ... with the operand |max| from an extra pass
    return lib


def run(lib, a, w, b, out, ws):
    M, K = a.shape
    N = w.shape[1]
    st = torch.cuda.current_stream().cuda_stream
    r = lib.gcs_linear_fwd(a.data_ptr(), K, w.data_ptr(), b.data_ptr(), out.data_ptr(), N, M, K, N, ws.data_ptr(),
                           ws.numel(), st)
    if r != 0:
        raise RuntimeError(f"gcs_linear_fwd failed with status {r}")


def time_arm(lib, a, w, b, out, ws, iters):
    for _ in range(3):
        run(lib, a, w, b, out, ws)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        run(lib, a, w, b, out, ws)
    e1.record()
    torch.cuda.synchronize()
    op_us = e0.elapsed_time(e1) * 1e3 / iters
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            run(lib, a, w, b, out, ws)
        torch.cuda.synchronize()
    durs, names = [], set()
    for ev in prof.events():
        if any(k in ev.name for k in GEMM_KERNELS) and ev.device_type.name == "CUDA":
            durs.append(ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total)
            names.add(ev.name.split("(")[0])
    per_call = len(durs) // iters
    calls = [sum(durs[i * per_call:(i + 1) * per_call]) for i in range(iters)]
    return statistics.median(calls), op_us, sorted(names), per_call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    libs = {"base": load(os.path.abspath(args.base)), "new": load(NEW)}
    rows = []
    for M, N, K in SHAPES:
        g = torch.Generator(device="cuda").manual_seed(M + N + K)
        a = torch.randn(M, K, device="cuda", generator=g)
        w = torch.randn(K, N, device="cuda", generator=g) / K ** 0.5
        b = torch.randn(N, device="cuda", generator=g)
        ws = torch.empty(max(libs[x].gcs_linear_workspace_bytes(M, K, N) for x in libs), dtype=torch.uint8, device="cuda")
        outs = {x: torch.empty(M, N, device="cuda") for x in libs}
        res = {x: [] for x in libs}
        for arm in ("base", "new", "base", "new"):
            res[arm].append(time_arm(libs[arm], a, w, b, outs[arm], ws, args.iters))
        ref = outs["base"].double()
        rel = float((outs["new"].double() - ref).abs().max() / ref.abs().max())
        tiles_rows = -(-M // 256)
        kb = K // 64
        row = {"M": M, "N": N, "K": K, "max_rel_diff_new_vs_base": rel}
        for arm in libs:
            us = statistics.median(r[0] for r in res[arm])
            per_cta_kb = 96 if arm == "base" else 64
            l2_bytes = tiles_rows * 2 * kb * (N // 256) * per_cta_kb * 1024
            row[arm] = {"kernel_us": round(us, 1), "kernel_us_runs": [round(r[0], 1) for r in res[arm]],
                        "op_us_events": [round(r[1], 1) for r in res[arm]], "kernels": res[arm][0][2],
                        "launches_per_call": res[arm][0][3],
                        "tflops_fp32_equiv": round(2.0 * M * N * K / (us * 1e-6) / 1e12, 1),
                        "l2_to_sm_GB": round(l2_bytes / 1e9, 2), "l2_to_sm_TBps": round(l2_bytes / (us * 1e-6) / 1e12, 2)}
        row["speedup"] = round(row["base"]["kernel_us"] / row["new"]["kernel_us"], 3)
        line = json.dumps(row)
        print(line, flush=True)
        rows.append(line)
        del a, w, b, ws, outs, ref
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    sys.exit(main())
