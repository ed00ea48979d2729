#!/bin/bash
# 1 GPU: full GPU suite + bench line after a kernel change
cd "$(dirname "$0")/.." || exit 1
OUT=${OUT:-session_out}; mkdir -p "$OUT"
TAG=${1:-check}
timeout 900 python -m pytest tests -m gpu -x -q > $OUT/${TAG}_pytest.log 2>&1; echo "pytest rc=$?"; tail -3 $OUT/${TAG}_pytest.log
timeout 600 python bench.py --no-cpu-baseline > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err; echo "bench rc=$?"
python - <<PY
import json
b = json.loads(open('$OUT/${TAG}_bench.json').read().strip().splitlines()[-1])
print('ms', round(b['ms_per_step'], 4), {k: round(v, 3) for k, v in b['roofline']['kernel_ms_all'].items()}, 'e2e', b['e2e'] and round(b['e2e']['ms_per_step'], 3), 'theta', b.get('theta_label_mismatch', {}).get('differing_labels'))
PY
