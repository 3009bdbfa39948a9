#!/bin/bash
# full GPU pass: every gpu test, the headline bench with the CPU baseline, configs 1-2, parity report
mkdir -p gpurun_out
timeout 1500 python -m pytest tests -q -m gpu -x --tb=short > gpurun_out/t_gpu.log 2>&1; echo "pytest rc=$?"; tail -n 25 gpurun_out/t_gpu.log
timeout 400 python bench.py --steps 5 --warmup 3 > gpurun_out/b_full.json 2> gpurun_out/b1.err; echo "bench rc=$?"; cut -c1-900 gpurun_out/b_full.json; tail -3 gpurun_out/b1.err
timeout 300 python tools/bench_configs.py > gpurun_out/configs12.jsonl 2>&1; cut -c1-220 gpurun_out/configs12.jsonl
timeout 600 python tools/parity_report.py 48 > gpurun_out/parity_r02.md 2> gpurun_out/parity.err; echo "parity rc=$?"; cat gpurun_out/parity_r02.md
