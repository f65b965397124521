#!/bin/bash
# round 2, first GPU call: issue-rate microbenchmarks, the GPU test-suite, the headline bench, A/B of the scan cell
mkdir -p gpurun_out/r2a
nvidia-smi --query-gpu=name,clocks.max.sm,clocks.sm --format=csv > gpurun_out/r2a/gpu.txt
tools/dpx_bench gpurun_out/r2a/dpx_peak.json > gpurun_out/r2a/dpx_bench.txt 2>&1
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -o tools/cell_bench tools/cell_bench.cu
tools/cell_bench gpurun_out/r2a/cell_bench.json > gpurun_out/r2a/cell_bench.txt 2>&1
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/r2a/pytest_gpu.txt 2>&1
echo "pytest exit $?" >> gpurun_out/r2a/pytest_gpu.txt
timeout 600 python bench.py > gpurun_out/r2a/bench.json 2> gpurun_out/r2a/bench.err
tools/variant_bench.sh parasail_rs_b200/libparasail_b200.so variants/lib_shifted.so > gpurun_out/r2a/variants.txt 2>&1
tail -3 gpurun_out/r2a/pytest_gpu.txt; cat gpurun_out/r2a/variants.txt; cat gpurun_out/r2a/cell_bench.txt
