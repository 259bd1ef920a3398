#!/bin/bash
# potrf iteration pass: tests, LAPACK check, default bench
mkdir -p gpurun_out
( timeout 900 python -m pytest tests -m gpu -x -q ) > gpurun_out/pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/pytest_gpu.log
tail -3 gpurun_out/pytest_gpu.log
timeout 600 python scripts/gpu_check_potrf.py > gpurun_out/potrf_check.log 2>&1; tail -25 gpurun_out/potrf_check.log
timeout 900 python bench.py > gpurun_out/bench_sweep.json 2> gpurun_out/bench_sweep.err
python - <<'PY'
import json
d=json.load(open('gpurun_out/bench_sweep.json'))
print(d['value'], d['ms_per_step'], d['roofline']['frac'], d['roofline']['stage_ms_total'], d['parity_vs_reference_golden'], d['e2e']['value'])
PY
