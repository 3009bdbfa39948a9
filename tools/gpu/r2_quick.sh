#!/bin/bash
# quick check of a kernel change: ResUNet against the rounding emulator, the G-path parity tests, headline bench twice
mkdir -p gpurun_out
timeout 600 python -m pytest -q tests/test_resunet_rounding.py 2>&1 | tail -4
timeout 900 python -m pytest tests/test_gpu_parity.py tests/test_gpu_parity_wide.py tests/test_gpu_switches.py -m gpu -q -x --tb=short 2>&1 | tail -4
for i in 1 2; do timeout 300 python bench.py --steps 6 --warmup 3 --no-cpu-baseline 2>/dev/null | python -c "import sys,json; d=json.loads(sys.stdin.read()); print('bench', round(d['value']), round(d['e2e']['value']), d['ms_per_step'])"; done
