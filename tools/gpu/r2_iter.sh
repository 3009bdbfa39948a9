#!/bin/bash
# Round-2 iteration pass: chain-kernel debug, headline bench (A/B switches as arguments "ENV=VAL"), per-layer ncu table.
#   gpurun --timeout 1200 -- 'bash tools/gpu/r2_iter.sh [ENV=VAL ...]'
mkdir -p gpurun_out
timeout 600 python -m pytest -q tests/test_resunet_rounding.py 2>&1 | tail -4
timeout 300 python bench.py --steps 4 --warmup 3 --no-cpu-baseline > gpurun_out/b_default.json 2> gpurun_out/b1.err; echo "bench rc=$?"; cut -c1-180 gpurun_out/b_default.json
for kv in "$@"; do
  timeout 300 env $kv python bench.py --steps 4 --warmup 3 --no-cpu-baseline > "gpurun_out/b_${kv}.json" 2>> gpurun_out/b1.err; echo "bench $kv rc=$?"; cut -c1-180 "gpurun_out/b_${kv}.json"
done
BCMD="python bench.py --steps 1 --warmup 3 --stamps 5000 --no-cpu-baseline"
$BCMD > gpurun_out/plain.log 2>&1 && timeout 800 ncu --metrics gpu__time_duration.sum,sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active,dram__bytes_read.sum,dram__bytes_write.sum,lts__throughput.avg.pct_of_peak_sustained_elapsed,sm__pipe_tc_cycles_active.avg.pct_of_peak_sustained_active --clock-control none -k regex:"k_conv_umma|k_rb_umma|k_l1_chain|k_head|k_tail|k_g_xupdate|k_subnet|k_g_prologue|k_moments" -s ${NCU_SKIP:-150} -c ${NCU_COUNT:-32} --csv --log-file gpurun_out/layers_iter.csv $BCMD > gpurun_out/ncu_iter.log 2>&1; echo "ncu rc=$?"
