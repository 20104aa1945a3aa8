#!/bin/bash
# A/B of the 256-column fp16 GEMM pass against a build of the parent commit (gcn-string_b200/variants/libbase.so,
# e.g. scripts/build_variant.sh or csrc/build.py in a worktree of the parent), everything in one GPU session:
#   scripts/pass256_ab.sh OUT_DIR
# kernel A/B (scripts/gemm_pass_bench.py), then bench.py three times per arm alternated, each arm once with
# --dump-outputs and once at --workload cfg5.  JSON lines and the dumped arrays go to OUT_DIR.
if [ -z "$1" ]; then echo "usage: $0 OUT_DIR" >&2; exit 2; fi
out=$1; mkdir -p $out
base=$PWD/gcn-string_b200/variants/libbase.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $out/gpu.csv
timeout 900 python scripts/gemm_pass_bench.py --base $base --iters 20 --out $out/gemm_pass_bench.jsonl 2> $out/gemm_pass_bench.err
tail -3 $out/gemm_pass_bench.err
arm() {   # arm NAME ARGS...: bench.py on the base library or on the in-tree one
  local name=$1; shift
  if [ $name == base ]; then export GCS_LIB_PATH=$base; else unset GCS_LIB_PATH; fi
  timeout 600 python bench.py "$@" 2>> $out/bench.err | tail -1 | python -c "import json,sys; d=json.loads(sys.stdin.read()); d['arm']='$name'; print(json.dumps(d))" >> $out/bench_ab.jsonl
  unset GCS_LIB_PATH
}
: > $out/bench_ab.jsonl
for i in 1 2 3; do arm base; arm new; done
arm base --dump-outputs $out/dump_base
arm new --dump-outputs $out/dump_new
arm base --workload cfg5
arm new --workload cfg5
python - "$out" <<'P'
import json, sys
rows = [json.loads(l) for l in open(sys.argv[1] + "/bench_ab.jsonl")]
for d in rows:
    ops = d.get("ops", {})
    lin = sum(ops[k]["ms_per_call"] * ops[k]["launches_timed"] / 2 for k in ("linear_fwd", "linear_bwd_input") if k in ops)
    print(d["arm"], d.get("workload", ""), d.get("value"), d.get("unit", ""), "ms/step", round(d.get("ms_per_step", 0), 3),
          "linear_fwd+bwd_input ms/step", round(lin, 3), "allocs", d.get("per_step_ms", {}).get("device_allocs_in_timed_region"),
          "launches", d.get("gpu_launches"))
import glob, os
import numpy as np
for f in sorted(glob.glob(sys.argv[1] + "/dump_base/*.npy")):
    a = np.load(f).astype(np.float64)
    b = np.load(f.replace("dump_base", "dump_new")).astype(np.float64)
    d = np.abs(a - b)
    print("dump", os.path.basename(f), a.shape, "max rel (to max |base|)", float(d.max() / max(np.abs(a).max(), 1e-300)),
          "elements differing by > 1e-4 relative", int((d > 1e-4 * np.abs(a).max()).sum()))
P
tail -3 $out/bench.err
