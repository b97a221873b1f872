#!/bin/bash
# 2-GPU: peer exchange at C2, row-sharded C5, pull micro-benchmark, scatter tests
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
N=${1:-2}
run() { name=$1; shift; timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus $N "$@" > gpurun_out/r2_mgpu_${name}_n$N.json 2> gpurun_out/r2_mgpu_${name}_n$N.err; echo "$name rc=$?"; python - <<PY
import json
try:
    d=json.loads([l for l in open("gpurun_out/r2_mgpu_${name}_n$N.json") if l.startswith("{")][-1])
    print({k:d.get(k) for k in ("value","ms_per_step","step_split","launches_per_step")}); print("   e2e", d["e2e"]["value"], "dp_parity", d.get("dp_parity"))
except Exception as e:
    print("no json", e); import subprocess; print(subprocess.run("grep -v Warn gpurun_out/r2_mgpu_${name}_n$N.err | tail -12 | cut -c1-300", shell=True, capture_output=True, text=True).stdout)
PY
}
timeout 600 python -m pytest tests/test_scatter.py -m gpu -x -q 2>&1 | tail -2
run c2peer --steps 20 --warmup 5 --no_profile --no_cpu_baseline --no_eval
run c5peer --config c5 --steps 10 --warmup 3 --no_profile --no_cpu_baseline --no_eval
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29531 scripts/bench_pull.py c5 2>&1 | grep "^rank"
