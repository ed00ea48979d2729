#!/bin/bash
# 2 GPUs: push kernel with the chunk cursor: single-GPU test, every gather kind on real peers, one bench line
cd "$(dirname "$0")/.." || exit 1
OUT=${OUT:-session_out}; mkdir -p "$OUT"
N=${1:-2}
T="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29544"
timeout 300 python -m pytest tests/test_snowfall_gpu.py -q -m gpu -k "gather_push" 2>&1 | tail -2
timeout 300 $T tools/check_gather_ranks.py 2> $OUT/r2n${N}e_gather_check.err | grep '^{' > $OUT/r2n${N}e_gather_check.json; echo "gather check rc=${PIPESTATUS[0]}"; cat $OUT/r2n${N}e_gather_check.json
LSS_GATHER=push timeout 300 $T bench.py --gpus $N --steps 20 --warmup 5 --no-e2e 2> $OUT/r2n${N}e_bench_push.err | grep '^{' > $OUT/r2n${N}e_bench_push.json; echo "bench rc=${PIPESTATUS[0]}"
python - <<PY
import json
b = json.loads(open('$OUT/r2n${N}e_bench_push.json').read().strip().splitlines()[-1])
print('ms', round(b['ms_per_step'], 4), 'value', '%.3e' % b['value'], {k: round(v, 3) for k, v in b['roofline']['kernel_ms_all'].items() if 'snow' in k}, b['engine'])
PY
