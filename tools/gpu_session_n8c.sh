#!/bin/bash
# 8 GPUs: correctness of every gather kind on real peers, bench with the push kernel (multicast / per-peer stores), device
# timeline of the host-to-host calls with all ranks active
cd "$(dirname "$0")/.." || exit 1
OUT=${OUT:-session_out}; mkdir -p "$OUT"
N=${1:-8}
T="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29544"
timeout 300 $T tools/check_gather_ranks.py > $OUT/r2n${N}c_gather_check.json 2> $OUT/r2n${N}c_gather_check.err; echo "gather check rc=$?"; cat $OUT/r2n${N}c_gather_check.json
run() { # name, env...
  local name=$1; shift
  env "$@" timeout 300 $T bench.py --gpus $N --steps 20 --warmup 5 --no-e2e > $OUT/r2n${N}c_bench_$name.json 2> $OUT/r2n${N}c_bench_$name.err; echo "bench $name rc=$?"
}
run push LSS_GATHER=push
run push_b37 LSS_GATHER=push LSS_GATHER_BLOCKS=37
run push_unicast LSS_GATHER=push LSS_GATHER_MULTICAST=0
run push_unicast_b64 LSS_GATHER=push LSS_GATHER_MULTICAST=0 LSS_GATHER_BLOCKS=64
timeout 300 $T tools/e2e_probe_ranks.py --bind 0 --trace 1 > $OUT/r2n${N}c_probe_trace.json 2> $OUT/r2n${N}c_probe_trace.err; echo "probe trace rc=$?"
python - <<PY
import json, glob
for f in sorted(glob.glob('$OUT/r2n${N}c_bench*.json')):
    try:
        b = json.loads(open(f).read().strip().splitlines()[-1])
        print(f, 'ms', round(b['ms_per_step'], 4), 'value', '%.3e' % b['value'], {k: round(v, 3) for k, v in b['roofline']['kernel_ms_all'].items() if 'snow' in k}, b['engine'].get('gather'), 'mc', b['engine'].get('gather_multicast'), b['engine'].get('gather_fallback'))
    except Exception as e:
        print(f, 'ERR', e, open(f.replace('.json', '.err')).read()[-1500:])
b = json.loads(open('$OUT/r2n${N}c_probe_trace.json').read().strip().splitlines()[-1])
for k in ('sync_chunks1', 'sync_chunks2', 'sync_chunks4'):
    print(k, b.get(k))
PY
