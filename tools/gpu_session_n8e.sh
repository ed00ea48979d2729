#!/bin/bash
# 8 GPUs: one bench line without the e2e leg (default exchange)
cd "$(dirname "$0")/.." || exit 1
OUT=${OUT:-session_out}; mkdir -p "$OUT"
N=${1:-8}
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29544 bench.py --gpus $N --steps 20 --warmup 5 --no-e2e 2> $OUT/r2n${N}e_bench.err | grep '^{' > $OUT/r2n${N}e_bench.json; echo "bench rc=${PIPESTATUS[0]}"
python - <<PY
import json
b = json.loads(open('$OUT/r2n${N}e_bench.json').read().strip().splitlines()[-1])
print('ms', round(b['ms_per_step'], 4), 'value', '%.3e' % b['value'], {k: round(v, 3) for k, v in b['roofline']['kernel_ms_all'].items() if 'snow' in k}, b['engine'])
PY
