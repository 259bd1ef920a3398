#!/bin/bash
# full pass: tests, smoke, bench (both arms + ensemble), other configs, launch list, full ncu captures
mkdir -p gpurun_out
( timeout 900 python -m pytest tests -m gpu -q ) > gpurun_out/pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/pytest_gpu.log
timeout 600 python __graft_entry__.py --smoke > gpurun_out/smoke.log 2>&1
timeout 900 python bench.py --impl reference --steps 3 --warmup 1 > gpurun_out/bench_reference.json 2> gpurun_out/bench_reference.err
timeout 900 python bench.py > gpurun_out/bench_sweep.json 2> gpurun_out/bench_sweep.err
timeout 600 python bench.py --workload ensemble > gpurun_out/bench_ensemble.json 2> gpurun_out/bench_ensemble.err
timeout 900 python scripts/gpu_configs.py > gpurun_out/configs.log 2>&1
timeout 600 python scripts/gpu_check_potrf.py > gpurun_out/potrf_check.log 2>&1
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv \
   --log-file gpurun_out/launches_sweep.csv python scripts/prof_driver.py sweep 1184 2 > gpurun_out/ncu_list.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'potrf_lnlike|rowsum_sym|moments_k|gemm_nt|marginal' -c 14 \
   -o gpurun_out/prof_sweep_final -f python scripts/prof_driver.py sweep 592 1 > gpurun_out/ncu_full.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:'design_rows' -c 1 \
   -o gpurun_out/prof_design_final -f python scripts/prof_driver.py design 16 1 >> gpurun_out/ncu_full.log 2>&1
tail -3 gpurun_out/pytest_gpu.log; tail -1 gpurun_out/smoke.log; python - <<'PY'
import json
for f in ("bench_sweep","bench_ensemble","bench_reference"):
    try:
        d=json.load(open('gpurun_out/%s.json'%f))
        print(f, d['value'], d.get('ms_per_step'), (d.get('roofline') or {}).get('frac'), (d.get('roofline') or {}).get('stage_ms_total'), d.get('cpu_baseline',{}).get('value'), d.get('cpu_baseline',{}).get('cores'))
    except Exception as e: print(f, "ERR", e)
PY
