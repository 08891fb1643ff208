#!/bin/bash
# Intensity GEMM with per-accumulator hand-over and bulk-store epilogue: parity tests and timing.
set -u
TAG=${1:-r2q}
OUT=gpurun_out
mkdir -p $OUT
echo "=== pytest feature + tensor-core decode ==="
timeout 600 python -m pytest tests/test_feature_gpu.py tests/test_parity_gpu.py -q -x -k "intensity or mining or tensor_core or feature_helper" 2>&1 | tail -15 | tee $OUT/pytest_int_$TAG.log
echo "=== bench intensity ==="
for t in 131072 262144; do timeout 120 python tools/bench_intensity.py --tokens $t 2>&1 | tail -1 | cut -c1-200 | tee -a $OUT/bench_intensity_$TAG.log; done
