#!/bin/bash
# Evidence capture for the tcgen05 MLP engine (csrc/mlp_tc.cu) on the GPU box (run through gpurun; writes into gpurun_out/):
#   bash profiles/capture_mlp_tc.sh <tag>
# 1. CUDA-event times of every MLP block with both engines, 2. launch list of the default bench (C4) step,
# 3. ncu --set full of mlp_tc_kernel (the three blocks of a C4 step), 4. compute-sanitizer memcheck + racecheck on its tests.
set -u
TAG=${1:-r2s}
OUT=gpurun_out
mkdir -p $OUT
python profiles/probe_kernels.py mlp_engines mlp_tc > $OUT/${TAG}_probe_mlp.txt 2>&1
python profiles/probe_tc_accum.py > $OUT/${TAG}_tc_accum.txt 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none --cache-control none -c 600 --csv \
    --log-file $OUT/${TAG}_launches_c4.csv python bench.py --steps 3 --warmup 3 --no-cpu --no-also \
    > $OUT/${TAG}_bench_under_ncu.log 2>&1
PROBE_WARM=1 PROBE_ITERS=1 ncu --set full --clock-control none --import-source on -k "regex:mlp_tc_kernel" -s 3 -c 3 \
    -o $OUT/${TAG}_mlp_tc -f python profiles/probe_kernels.py mlp_tc > $OUT/${TAG}_probe_under_ncu.txt 2>&1
ncu -i $OUT/${TAG}_mlp_tc.ncu-rep --page raw --csv > $OUT/${TAG}_mlp_tc_raw.csv 2>/dev/null
ncu -i $OUT/${TAG}_mlp_tc.ncu-rep --page source --csv > $OUT/${TAG}_mlp_tc_source.csv 2>/dev/null
ls -la $OUT/${TAG}_mlp_tc.ncu-rep
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 1 python -m pytest tests/test_gpu_mlp_tc.py \
    -x -q -m gpu -k "not 4096" > $OUT/${TAG}_memcheck.txt 2>&1
echo "memcheck rc=$?" >> $OUT/${TAG}_memcheck.txt
timeout 900 compute-sanitizer --tool racecheck --error-exitcode 1 python -m pytest tests/test_gpu_mlp_tc.py \
    -x -q -m gpu -k "not 4096 and not 1000" > $OUT/${TAG}_racecheck.txt 2>&1
echo "racecheck rc=$?" >> $OUT/${TAG}_racecheck.txt
tail -4 $OUT/${TAG}_memcheck.txt $OUT/${TAG}_racecheck.txt; cat $OUT/${TAG}_probe_mlp.txt
