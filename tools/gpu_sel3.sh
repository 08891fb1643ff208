#!/bin/bash
# Selection v3 (sample-bracketed single pass): tests, A/B timing against the three-pass kernel on
# normal rows and on the intensity GEMM's own rows
set -u
TAG=${1:-r5}
OUT=gpurun_out; mkdir -p $OUT
timeout 600 python -m pytest tests/test_feature_gpu.py -x -q -k "select or mining or helper" 2>&1 | tail -8 | tee $OUT/select_tests_$TAG.log
for v in 0 1; do RQAE_MINE_V2=$v timeout 120 python tools/bench_select.py 2>&1 | tail -1; done | tee $OUT/select_ab_$TAG.log
timeout 200 python tools/select_gemm_rows.py 2>&1 | tail -30 | tee $OUT/select_gemm_rows_$TAG.log
