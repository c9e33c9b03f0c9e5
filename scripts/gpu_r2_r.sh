#!/usr/bin/env bash
set -u
mkdir -p gpurun_out
timeout 300 python -m pytest tests/test_gpu_kernels.py -m gpu -x -q -k "umma" > gpurun_out/r2r_umma.log 2>&1
echo "umma tests rc=$?"; tail -n 3 gpurun_out/r2r_umma.log
timeout 600 python -m pytest tests -m gpu -x -q > gpurun_out/r2r_pytest.log 2>&1
echo "pytest rc=$?"; tail -n 3 gpurun_out/r2r_pytest.log
timeout 300 python bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-extras > gpurun_out/r2r_bench.json 2> gpurun_out/r2r_bench.err
echo "bench rc=$?"; python - <<'PY'
import json
d=json.load(open('gpurun_out/r2r_bench.json'))
print({k:d[k] for k in ['value','ms_per_step','launches_per_step']}, d['e2e']['value'])
for r in d['ops']: print(r['op'], r['ms'], r['share'])
PY
