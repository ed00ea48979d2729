#!/bin/bash
# 1 GPU: build-flag variants of the solve kernel (CTAs per SM / arena slots per warp), parity tests + bench line for each
cd "$(dirname "$0")/.." || exit 1
OUT=${OUT:-session_out}; mkdir -p "$OUT"
B="python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-e2e"
timeout 600 $B > $OUT/r2v_bench_default.json 2> $OUT/r2v_bench_default.err; echo "default rc=$?"
for V in "7 128" "8 112" "5 192"; do
  set -- $V
  LSS_NVCC_FLAGS="-DLSS_SOLVE_CTAS=$1 -DLSS_SOLVE_ARENA=$2" python -m lidar_snow_sim_b200.build > $OUT/r2v_build_c$1_a$2.log 2>&1
  grep -E "spill|error" $OUT/r2v_build_c$1_a$2.log | head -3
  timeout 300 python -m pytest tests/test_snowfall_gpu.py tests/test_reference_replay_gpu.py -m gpu -x -q 2>&1 | tail -1
  timeout 600 $B > $OUT/r2v_bench_c$1_a$2.json 2> $OUT/r2v_bench_c$1_a$2.err; echo "c$1 a$2 rc=$?"
done
OUT=$OUT python - <<'PY'
import json, glob, os
for f in sorted(glob.glob(os.environ['OUT'] + '/r2v_bench*.json')):
    try:
        b = json.loads(open(f).read().strip().splitlines()[-1])
        print(f, round(b['ms_per_step'], 4), {k: round(v, 4) for k, v in b['roofline']['kernel_ms_all'].items() if 'snow' in k or 'pre' in k})
    except Exception as e:
        print(f, 'ERR', e)
PY
