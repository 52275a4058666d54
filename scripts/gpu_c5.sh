#!/bin/bash
# Runs on the GPU box: GPU tests, A/B of scratch libs, C2 line, C5 line, default line.
mkdir -p gpurun_out; : > gpurun_out/ab_ransac.txt
bash scripts/gpu_tests.sh
for lib in scratch_libs/*.so; do SFMGPU_LIB=$PWD/$lib timeout 300 python scripts/ab_ransac.py >> gpurun_out/ab_ransac.txt 2>&1; done
timeout 300 python scripts/ab_ransac.py >> gpurun_out/ab_ransac.txt 2>&1
timeout -k 10 600 python bench.py --workload c2 --steps 3 --warmup 2 > gpurun_out/bench_c2.json 2> gpurun_out/bench_c2.err; echo "c2 rc=$?" | tee -a gpurun_out/summary.txt
timeout -k 10 900 python bench.py --workload c5 --steps 3 --warmup 1 > gpurun_out/bench_c5.json 2> gpurun_out/bench_c5.err; echo "c5 rc=$?" | tee -a gpurun_out/summary.txt
timeout -k 10 900 python bench.py > gpurun_out/bench.json 2> gpurun_out/bench.err; echo "bench rc=$?" | tee -a gpurun_out/summary.txt
