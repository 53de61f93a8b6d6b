#!/bin/bash
# round-2 first GPU pass: stage parity of the persistent layer kernel, its timing, full GPU suite, bench
mkdir -p gpurun_out
timeout 600 python -m pytest tests/test_gpu_stages.py -x -q > gpurun_out/r2a_stages.log 2>&1; rc=$?
tail -15 gpurun_out/r2a_stages.log
if [ $rc -eq 124 ]; then echo "STAGE TEST HUNG"; exit 1; fi
timeout 600 python tools/ps_timing.py > gpurun_out/r2a_ps_timing.log 2>&1; rc2=$?
tail -12 gpurun_out/r2a_ps_timing.log
if [ $rc2 -eq 124 ]; then echo "TIMING HUNG"; exit 1; fi
if [ $rc -ne 0 ]; then echo "stage tests failed; skipping the rest"; exit 1; fi
timeout 1500 python -m pytest tests -m gpu -x -q > gpurun_out/r2a_gpu_tests.log 2>&1
tail -8 gpurun_out/r2a_gpu_tests.log
timeout 600 python bench.py > gpurun_out/r2a_bench.json 2> gpurun_out/r2a_bench.err
tail -2 gpurun_out/r2a_bench.json
