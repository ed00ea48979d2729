#!/bin/bash
# final single-GPU evidence run: smoke, parity suite, compute-sanitizer over the small tests of the round-2 kernels, bench lines
# (config 1 with the CPU baseline, config 2), ncu launch list + full capture of the beam stage
cd "$(dirname "$0")/.." || exit 1
OUT=${OUT:-session_out}; mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/r2g_smoke.txt 2>&1; echo "smoke rc=$?"
timeout 900 python -m pytest tests -m gpu -q > $OUT/r2g_gpu_tests.txt 2>&1
echo "tests rc=$?"; tail -3 $OUT/r2g_gpu_tests.txt
SEL='test_golden_kat_channel or test_golden_channel_cases or test_batch_ragged_and_empty or test_degenerate_rows or test_beams_with_dozens or test_gather_push or test_device_fixed_seed or (test_batch_matches_the_oracle and 3000)'
timeout 240 compute-sanitizer --tool memcheck --print-limit 20 python -m pytest tests -m gpu -q -k "$SEL" > $OUT/r2g_memcheck.log 2>&1; echo "memcheck rc=$?"
grep -E "passed|failed|ERROR SUMMARY" $OUT/r2g_memcheck.log | head -5
RSEL='test_golden_kat_channel or test_beams_with_dozens or test_gather_push'
timeout 240 compute-sanitizer --tool racecheck --print-limit 20 python -m pytest tests -m gpu -q -k "$RSEL" > $OUT/r2g_racecheck.log 2>&1; echo "racecheck rc=$?"
grep -E "passed|failed|RACECHECK SUMMARY" $OUT/r2g_racecheck.log | head -5
timeout 600 python bench.py --steps 20 --warmup 5 > $OUT/r2g_bench.json 2> $OUT/r2g_bench.err; echo "bench rc=$?"
timeout 300 python bench.py --steps 20 --warmup 5 --config 2 --no-cpu-baseline > $OUT/r2g_bench_cfg2.json 2> $OUT/r2g_bench_cfg2.err; echo "bench cfg2 rc=$?"
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -s 120 -c 100 --csv --log-file $OUT/r2g_launches.csv python tools/profile_step.py --steps 10 > $OUT/r2g_ncu_list.log 2>&1; echo "list rc=$?"
timeout 400 ncu --set full --clock-control none --import-source on -k "regex:k_scan|k_list_sort|k_solve|k_overflow" -s 16 -c 4 -f -o $OUT/r2g_beam python tools/profile_step.py --steps 6 > $OUT/r2g_ncu_beam.log 2>&1; echo "ncu beam rc=$?"
python - <<PY
import json
for f in ('$OUT/r2g_bench.json', '$OUT/r2g_bench_cfg2.json'):
    b = json.loads(open(f).read().strip().splitlines()[-1])
    print(f, 'ms', round(b['ms_per_step'], 4), 'frac', round(b['roofline']['frac'], 4), 'e2e', b['e2e'] and round(b['e2e']['ms_per_step'], 3), 'cpu', b.get('cpu_baseline', {}).get('value'), 'theta', b.get('theta_label_mismatch', {}).get('differing_labels'))
PY
