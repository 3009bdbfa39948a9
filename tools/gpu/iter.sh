#!/bin/bash
# Fast iteration pass: GPU tests, headline bench (optionally under A/B environment switches given as arguments, e.g.
# "GDECONV_CLUSTER=1"), and the per-layer ncu table of one denoiser call.
#   gpurun --timeout 1200 -- 'bash tools/gpu/iter.sh [ENV=VAL ...]'
mkdir -p gpurun_out
timeout 900 python -m pytest tests -q -m gpu -x --tb=short > gpurun_out/t_gpu.log 2>&1; echo "pytest rc=$?"; tail -n 15 gpurun_out/t_gpu.log
timeout 600 python bench.py --steps 5 --warmup 3 --no-cpu-baseline > gpurun_out/bench_iter.json 2> gpurun_out/bench_iter.err; echo "bench rc=$?"; cut -c1-160 gpurun_out/bench_iter.json
for kv in "$@"; do
  timeout 600 env $kv python bench.py --steps 5 --warmup 3 --no-cpu-baseline > "gpurun_out/bench_iter_${kv}.json" 2>> gpurun_out/bench_iter.err; echo "bench $kv rc=$?"; cut -c1-160 "gpurun_out/bench_iter_${kv}.json"
done
BCMD="python bench.py --steps 1 --warmup 3 --stamps 5000 --no-cpu-baseline"
timeout 1200 ncu --metrics gpu__time_duration.sum,sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active,dram__bytes_read.sum,dram__bytes_write.sum,lts__throughput.avg.pct_of_peak_sustained_elapsed --clock-control none -k regex:"k_conv_umma|k_rb_umma|k_head|k_tail|k_g_xupdate|k_subnet|k_g_prologue|k_moments" -s 185 -c 40 --csv --log-file gpurun_out/layers_iter.csv $BCMD > gpurun_out/ncu_iter.log 2>&1; echo "ncu layers rc=$?"
# one full-section capture of up1 + the four level-0 convs behind it (launches 29..33 of the second denoiser call)
if [ -n "$NCU_FULL" ]; then
timeout 1200 ncu --set full --import-source on --clock-control none -k regex:"k_conv_umma" -s 301 -c 5 -o gpurun_out/full_iter -f $BCMD > gpurun_out/ncu_full.log 2>&1; echo "ncu full rc=$?"
fi
