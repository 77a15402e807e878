#!/bin/bash
# Evidence capture for the f16 select filter (run through gpurun; writes into gpurun_out/):  bash profiles/capture_filter_f16.sh <tag>
# 1. CUDA-event times tf32 vs f16 filter, 2. ncu --set full of the filter + refine at C4 and C2 (feeds profiles/traffic.json),
# 3. launch list of the default bench step, 4. compute-sanitizer memcheck on the tcgen05 tests, 5. the TMEM micro-benchmark.
set -u
TAG=${1:-r2t}
OUT=gpurun_out
mkdir -p $OUT
python profiles/probe_kernels.py select_f16 > $OUT/${TAG}_probe_select.txt 2>&1
./profiles/micro/tmem_f16 > $OUT/${TAG}_tmem_f16.txt 2>&1
PROBE_WARM=0 PROBE_ITERS=1 ncu --set full --clock-control none -k "regex:score_select_tc_kernel|tc_refine_kernel" \
    -o $OUT/${TAG}_filter -f python profiles/probe_kernels.py select select_c2 > $OUT/${TAG}_probe_under_ncu.txt 2>&1
ncu -i $OUT/${TAG}_filter.ncu-rep --page raw --csv > $OUT/${TAG}_filter_raw.csv 2>/dev/null
ls -la $OUT/${TAG}_filter.ncu-rep
ncu --metrics gpu__time_duration.sum --clock-control none --cache-control none -c 600 --csv \
    --log-file $OUT/${TAG}_launches_c4.csv python bench.py --steps 3 --warmup 3 --no-cpu --no-also \
    > $OUT/${TAG}_bench_under_ncu.log 2>&1
timeout 600 compute-sanitizer --tool memcheck --error-exitcode 1 python -m pytest tests/test_gpu_tcgen05.py \
    -x -q -m gpu -k "not full_size and not max_size" > $OUT/${TAG}_memcheck.txt 2>&1
echo "memcheck rc=$?" >> $OUT/${TAG}_memcheck.txt
tail -n 4 $OUT/${TAG}_memcheck.txt; cat $OUT/${TAG}_probe_select.txt
