#!/bin/bash
# the evidence visit of tools/gpu_r5.sh without the sanitizer passes
# selection kernel, ncu --set full of it
set -u
TAG=${1:-r5p}
OUT=gpurun_out
mkdir -p $OUT
CS=/usr/local/cuda/bin/compute-sanitizer
echo "=== pytest -m gpu ==="
timeout 1200 python -m pytest tests -m gpu -x -q 2>&1 | tail -4 | tee $OUT/pytest_gpu_$TAG.log
echo "=== smoke ==="
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee $OUT/smoke_$TAG.log
echo "=== selection A/B (normal rows) ==="
for v in 0 1; do RQAE_MINE_V2=$v timeout 120 python tools/bench_select.py 2>&1 | tail -1; done | tee $OUT/select_ab_$TAG.log
echo "=== bench ==="
timeout 900 python bench.py --steps 5 --warmup 3 > $OUT/bench_$TAG.json 2> $OUT/bench_$TAG.err; echo "bench exit=$?"
tail -3 $OUT/bench_$TAG.err
if false; then
timeout 400 $CS --tool racecheck --error-exitcode 9 python -m pytest tests/test_feature_gpu.py -q -x -k "65536 or short_16384 or heavy_median_tie or few_values or 20000" 2>&1 | tail -4 | tee $OUT/sanitize_racecheck_mine3_$TAG.log
timeout 400 $CS --tool memcheck --error-exitcode 9 python -m pytest tests/test_feature_gpu.py -q -x -k "(adversarial and not long_2M) or 16384 or 40003" 2>&1 | tail -4 | tee $OUT/sanitize_memcheck_mine3_$TAG.log
timeout 400 $CS --tool initcheck --error-exitcode 9 python -m pytest tests/test_feature_gpu.py -q -x -k "short_16384 or zero_centered or specials or 20000" 2>&1 | tail -4 | tee $OUT/sanitize_initcheck_mine3_$TAG.log
fi
echo "=== ncu full: selection v3 ==="
timeout 600 ncu --set full --clock-control none --import-source on -k regex:rq_mine3 -s 1 -c 1 -f \
  -o $OUT/prof_mine3_$TAG python tools/bench_select.py --rows 2368 --reps 1 > $OUT/ncu_mine3_$TAG.log 2>&1
tail -2 $OUT/ncu_mine3_$TAG.log
