#!/bin/bash
# Round-2 GPU job G: flow / material tests with the tcgen05 coupling-block forward, material bench (tcgen05 vs FP32-pipe A/B).
set -u
mkdir -p gpurun_out
timeout 600 python -m pytest tests/test_flow_gpu.py tests/test_golden.py tests/test_mc_gpu.py -q -m gpu -x 2>&1 | tail -40 > gpurun_out/r2g_pytest.log
tail -25 gpurun_out/r2g_pytest.log
timeout 300 python scripts/bench_material.py --steps 5 > gpurun_out/r2g_bench_material.json 2> gpurun_out/r2g_bench_material.err; tail -c 1700 gpurun_out/r2g_bench_material.json; tail -3 gpurun_out/r2g_bench_material.err
