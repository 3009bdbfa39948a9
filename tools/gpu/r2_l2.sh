#!/bin/bash
# level-1 chain kernel check: debug parity, headline bench, one full ncu capture (source-level) of the two k_l2_chain launches
mkdir -p gpurun_out
timeout 600 python -m pytest -q tests/test_resunet_rounding.py 2>&1 | tail -4
timeout 300 python bench.py --steps 4 --warmup 3 --no-cpu-baseline > gpurun_out/b_default.json 2> gpurun_out/b1.err; echo "bench rc=$?"; cut -c1-180 gpurun_out/b_default.json
BCMD="python bench.py --steps 1 --warmup 3 --stamps 5000 --no-cpu-baseline"
$BCMD > gpurun_out/plain.log 2>&1 && timeout 800 ncu --set full --import-source on --clock-control none -k regex:"k_l2_chain" -s 8 -c 2 -o gpurun_out/l2chain_full -f $BCMD > gpurun_out/ncu_iter.log 2>&1; echo "ncu rc=$?"
