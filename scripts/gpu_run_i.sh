#!/bin/bash
# Round-2 GPU job I: final single-GPU evidence: full GPU suite (+ FP32-pipe flow path, + sanitizer passes on the new kernels),
# headline bench line, secondary benches, launch lists restricted to the timed steps.
set -u
mkdir -p gpurun_out
rm -f gpurun_out/gpu_test_errors.json
python -m pytest tests/ -q -m gpu 2>&1 | tail -30 > gpurun_out/r2i_pytest.log; tail -8 gpurun_out/r2i_pytest.log
timeout 1200 compute-sanitizer --tool memcheck --error-exitcode 1 python -m pytest tests/test_shape_gpu.py tests/test_renderer.py tests/test_shader.py -q -x \
    -k "vm_feature or neus_composite or tv_loss or gaussian or sampler or probe or alpha_mask or cuda_shader" > gpurun_out/r2i_sanitizer_memcheck.log 2>&1
echo "memcheck rc=$?" | tee -a gpurun_out/r2i_sanitizer_memcheck.log
timeout 1200 compute-sanitizer --tool racecheck --error-exitcode 1 python -m pytest tests/test_shape_gpu.py tests/test_renderer.py -q -x \
    -k "neus_composite or tv_loss or gaussian or sampler or probe" > gpurun_out/r2i_sanitizer_racecheck.log 2>&1
echo "racecheck rc=$?" | tee -a gpurun_out/r2i_sanitizer_racecheck.log
python bench.py 2> gpurun_out/r2i_bench.err | tee gpurun_out/r2i_bench.json | python -c "
import json,sys
d=json.loads(sys.stdin.read())
print(d['value'], d['ms_per_step'], d['e2e']['value'], d['gpu_launches'], d['roofline']['frac'], d['cpu_baseline'], d['clocks'])
print('check', d['check']['max_output'], d['check']['max_grad'], d['check']['within_tolerance'])
print('secondary', d['secondary'])
print(d['roofline']['kernels_ms_per_step'])"
tail -3 gpurun_out/r2i_bench.err
python bench.py --impl reference --steps 3 --warmup 1 > gpurun_out/r2i_bench_reference.json 2> gpurun_out/r2i_bench_reference.err; tail -c 600 gpurun_out/r2i_bench_reference.json
python scripts/bench_material.py --steps 10 > gpurun_out/r2i_bench_material.json 2>/dev/null; tail -c 300 gpurun_out/r2i_bench_material.json
python scripts/bench_shape_renderer.py --steps 10 > gpurun_out/r2i_bench_shape_renderer.json 2>/dev/null; tail -c 300 gpurun_out/r2i_bench_shape_renderer.json
python scripts/bench_adam.py > gpurun_out/r2i_bench_adam.json 2>/dev/null; tail -c 300 gpurun_out/r2i_bench_adam.json
export TF_PROFILE_RANGE=1
timeout 900 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/r2i_launches_bench.csv \
    python bench.py --steps 1 --warmup 3 --no-cpu-baseline --no-secondary --check-rays 0 > gpurun_out/r2i_launches_bench.log 2>&1
timeout 900 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/r2i_launches_material.csv \
    python scripts/bench_material.py --steps 1 > gpurun_out/r2i_launches_material.log 2>&1
timeout 900 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/r2i_launches_renderer.csv \
    python scripts/bench_shape_renderer.py --steps 1 > gpurun_out/r2i_launches_renderer.log 2>&1
wc -l gpurun_out/r2i_launches_*.csv
