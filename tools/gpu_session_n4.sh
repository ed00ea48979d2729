#!/bin/bash
# N GPUs: the driver's own command line (default gather, e2e leg included)
cd "$(dirname "$0")/.." || exit 1
OUT=${OUT:-session_out}; mkdir -p "$OUT"
N=${1:-4}
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29544 bench.py --gpus $N --steps 20 --warmup 5 2> $OUT/r2n${N}_bench_driver.err | grep '^{' > $OUT/r2n${N}_bench_driver.json; echo "bench rc=${PIPESTATUS[0]}"
python - <<PY
import json
b = json.loads(open('$OUT/r2n${N}_bench_driver.json').read().strip().splitlines()[-1])
print('ms', round(b['ms_per_step'], 4), 'value', '%.3e' % b['value'], {k: round(v, 3) for k, v in b['roofline']['kernel_ms_all'].items() if 'snow' in k}, b['engine'], 'e2e', b['e2e'] and (round(b['e2e']['ms_per_step'], 3), '%.3e' % b['e2e']['value'], b['e2e']['copy_out'], b['e2e']['d2h_bytes_per_step']))
PY
tail -3 $OUT/r2n${N}_bench_driver.err
