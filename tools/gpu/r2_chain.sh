#!/bin/bash
# chain-kernel check: debug parity, headline bench, ncu time of the level-0 kernels
mkdir -p gpurun_out
timeout 600 python -m pytest -q tests/test_resunet_rounding.py 2>&1 | tail -4
timeout 300 python bench.py --steps 4 --warmup 3 --no-cpu-baseline > gpurun_out/b_default.json 2> gpurun_out/b1.err; echo "bench rc=$?"; cut -c1-180 gpurun_out/b_default.json
BCMD="python bench.py --steps 1 --warmup 3 --stamps 5000 --no-cpu-baseline"
$BCMD > gpurun_out/plain.log 2>&1 && timeout 800 ncu --metrics gpu__time_duration.sum,sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active,dram__bytes_read.sum,dram__bytes_write.sum,lts__throughput.avg.pct_of_peak_sustained_elapsed --clock-control none -k regex:"k_l1_chain|k_l2_chain" -s 16 -c 8 --csv --log-file gpurun_out/layers_iter.csv $BCMD > gpurun_out/ncu_iter.log 2>&1; echo "ncu rc=$?"
