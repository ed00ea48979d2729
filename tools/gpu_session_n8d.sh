#!/bin/bash
# 8 GPUs, last pass: the exchange step alone (every kind / block count), bench with multicast push at two block counts, then the
# full bench line (e2e included) of the best configuration
cd "$(dirname "$0")/.." || exit 1
OUT=${OUT:-session_out}; mkdir -p "$OUT"
N=${1:-8}
T="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29544"
timeout 240 $T tools/gather_bench_ranks.py 2> $OUT/r2n${N}d_gather_alone.err | grep '^{' > $OUT/r2n${N}d_gather_alone.json; echo "gather alone rc=$?"; cat $OUT/r2n${N}d_gather_alone.json
run() { # name, extra args, env...
  local name=$1; local extra=$2; shift 2
  env "$@" timeout 300 $T bench.py --gpus $N --steps 20 --warmup 5 $extra 2> $OUT/r2n${N}d_bench_$name.err | grep '^{' > $OUT/r2n${N}d_bench_$name.json; echo "bench $name rc=$?"
}
run push_b74 --no-e2e LSS_GATHER=push LSS_GATHER_BLOCKS=74
run push_b148 --no-e2e LSS_GATHER=push LSS_GATHER_BLOCKS=148
BEST=$(python - <<PY
import json
best, arg = 1e9, '0'
for name, blocks in (('push_b74', '74'), ('push_b148', '148')):
    try:
        b = json.loads(open('$OUT/r2n${N}d_bench_%s.json' % name).read().strip().splitlines()[-1])
        if b['ms_per_step'] < best:
            best, arg = b['ms_per_step'], blocks
    except Exception:
        pass
print(arg if best < 1.10 else '37')
PY
)
echo "best multicast block count: $BEST"
run final "" LSS_GATHER=push LSS_GATHER_BLOCKS=$BEST
python - <<PY
import json, glob
for f in sorted(glob.glob('$OUT/r2n${N}d_bench*.json')):
    try:
        b = json.loads(open(f).read().strip().splitlines()[-1])
        print(f, 'ms', round(b['ms_per_step'], 4), 'value', '%.3e' % b['value'], {k: round(v, 3) for k, v in b['roofline']['kernel_ms_all'].items() if 'snow' in k}, b['engine'].get('gather'), 'mc', b['engine'].get('gather_multicast'), 'e2e', b['e2e'] and (round(b['e2e']['ms_per_step'], 3), '%.3e' % b['e2e']['value']))
    except Exception as e:
        print(f, 'ERR', e, open(f.replace('.json', '.err')).read()[-1500:])
PY
