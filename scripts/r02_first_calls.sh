#!/bin/bash
# First GPU calls of the next round: validate and time the multi-GPU path.  The two opt-in schedules it also timed, since removed, were written at the end of
# round 1 without hardware (DESIGN.md section 8 items 1-2).  Run with:  gpurun --gpus 8 --timeout 600 -- 'bash scripts/r02_first_calls.sh 8'
# Every command is bounded by `timeout`; a hang in a new NCCL / symmetric-memory schedule must not hold the box.
N=${1:-8}
OUT=gpurun_out/r02_first
mkdir -p $OUT
# 0. single GPU: random-geometry fuzz of ac_embed against the oracle (promote into tests/ once green)
timeout 200 python scripts/fuzz_embed_gpu.py 60 > $OUT/fuzz_embed.log 2>&1; echo "fuzz embed rc=$?"; tail -3 $OUT/fuzz_embed.log
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1"
# 1. the sharded path (symmetric-memory transport, NCCL collectives, all-pairs form) against one GPU
timeout 150 $TR --master-port 29551 scripts/check_sharded.py > $OUT/check_sharded_n$N.log 2>&1; echo "check sharded rc=$?"
# 2. timing, config 2
timeout 120 $TR --master-port 29553 bench.py --gpus $N --steps 20 --warmup 5 --no-e2e > $OUT/bench_default_n$N.json 2> $OUT/bench_default_n$N.err
# 3. sharded supervised path at N ranks (validated at 1 and 2 ranks in round 1)
timeout 150 $TR --master-port 29556 scripts/check_supervised_sharded.py > $OUT/check_supervised_n$N.log 2>&1; echo "check supervised rc=$?"
# 4. configs 3 and 5 at N ranks (1-GPU numbers: scripts/run_configs.py)
timeout 240 $TR --master-port 29557 scripts/run_configs_sharded.py > $OUT/configs_n$N.log 2>&1; echo "configs rc=$?"; tail -1 $OUT/configs_n$N.log
grep -h "OK\|MISMATCH" $OUT/check_*_n$N.log | tail -40
for f in $OUT/bench_*_n$N.json; do python - "$f" <<'PY'
import json, sys
try:
    d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
    print(sys.argv[1], "images/s", round(d["value"]), "ms/step", round(d["ms_per_step"], 3), d.get("stages", {}).get("comm_ms_per_step_rank0"))
except Exception as e:
    print(sys.argv[1], "no result:", e)
PY
done
