#!/bin/bash
mkdir -p gpurun_out
timeout 300 python -m pytest tests/test_gpu_stages.py -x -q > gpurun_out/r2f_stages.log 2>&1; rc=$?
tail -25 gpurun_out/r2f_stages.log
if [ $rc -eq 124 ]; then echo "STAGE TEST HUNG"; exit 1; fi
if [ $rc -ne 0 ]; then echo "stage tests failed"; exit 1; fi
timeout 900 python -m pytest tests/test_gpu_parity.py tests/test_flow_decoder.py -x -q > gpurun_out/r2f_parity.log 2>&1; tail -8 gpurun_out/r2f_parity.log
timeout 600 python tools/ps_timing.py f16f8 > gpurun_out/r2f_ps_timing.log 2>&1; tail -3 gpurun_out/r2f_ps_timing.log | cut -c1-900
timeout 600 python bench.py --no-cpu-baseline --no-extra > gpurun_out/r2f_bench.json 2> gpurun_out/r2f_bench.err; tail -c 2600 gpurun_out/r2f_bench.json
