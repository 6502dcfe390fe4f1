#!/usr/bin/env bash
# GPU-box helper: the whole -m gpu suite, smoke, then bench at 1 GPU.
mkdir -p gpurun_out
timeout 1500 python -m pytest tests -q -m gpu -x --durations=8 > gpurun_out/gpu_tests.log 2>&1; echo "gpu tests rc=$?"; tail -14 gpurun_out/gpu_tests.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python bench.py --gpus 1 --steps 30 --warmup 5 > gpurun_out/bench_1gpu.json 2> gpurun_out/bench_1gpu.err; echo "bench rc=$?"; head -c 1500 gpurun_out/bench_1gpu.json; tail -3 gpurun_out/bench_1gpu.err
