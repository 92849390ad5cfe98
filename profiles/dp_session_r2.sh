#!/bin/bash
# Multi-GPU session: DP correctness (fused peer all-reduce + Adam vs NCCL + Adam) and the bench line for the optimizer-kernel
# variants.   usage: bash profiles/dp_session_r2.sh <N> <tag> [variants...]   (variants: default pipeline nccl ...)
N=${1:-2}
TAG=${2:-r2}
shift 2
VARIANTS=${@:-default pipeline}
O=gpurun_out
mkdir -p $O
RUN="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29533"
if [ -z "$SKIP_DP_CHECK" ]; then
$RUN tests/dp_peer_check.py > $O/dp_check_${TAG}_n$N.json 2> $O/dp_check_${TAG}_n$N.err; echo "dp_check rc $?"; cat $O/dp_check_${TAG}_n$N.json
fi
for v in $VARIANTS; do
  case $v in
    default) ENVV=""; ARGS="";;
    overlap) ENVV=""; ARGS="--overlap";;
    no_pipeline) ENVV=""; ARGS="--no-pipeline";;
    skip_check) ENVV=""; ARGS="";;
    pipeline) ENVV=""; ARGS="--pipeline";;
    nccl) ENVV=""; ARGS="--nccl";;
    chunks1) ENVV=""; ARGS="--chunks 1";;
    chunks1_pipeline) ENVV=""; ARGS="--chunks 1 --pipeline";;
  esac
  env $ENVV $RUN bench.py --gpus $N --steps 96 --warmup 16 --no-cpu-baseline --no-ref-cuda --no-shading $ARGS > $O/bench_${TAG}_${v}_n$N.json 2> $O/bench_${TAG}_${v}_n$N.err
  echo "bench $v rc $?"
  python - <<PY
import json
try:
    d = json.load(open("$O/bench_${TAG}_${v}_n$N.json"))
    k = d["roofline"]["kernels_ms_per_step"]
    print("$v", "ms/step", round(d["ms_per_step"], 4), "value", round(d["value"] / 1e9, 3), "G/s  e2e", round(d["e2e"]["value"] / 1e9, 3), "median", round(d["config"]["step_ms"]["median"], 4), "dp_check", d.get("dp_check", {}).get("ok"), {a: round(b, 4) for a, b in k.items()})
except Exception as e:
    print("$v failed", e)
PY
done
