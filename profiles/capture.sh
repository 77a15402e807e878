#!/bin/bash
# Evidence capture on the GPU box (run through gpurun; writes into gpurun_out/):
#   bash profiles/capture.sh <tag>
# 1. launch list of the default bench (C4) step, 2. ncu --set full of every shipped kernel at a representative
# size (profiles/probe_kernels.py), 3. compute-sanitizer memcheck + racecheck on small shapes.
set -u
TAG=${1:-r2}
OUT=gpurun_out
mkdir -p $OUT
python profiles/probe_kernels.py > $OUT/${TAG}_probe.txt 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none --cache-control none -c 600 --csv \
    --log-file $OUT/${TAG}_launches_c4.csv python bench.py --steps 3 --warmup 3 --no-cpu --no-also \
    > $OUT/${TAG}_bench_under_ncu.log 2>&1
KERNELS='score_select_tc_kernel|tc_refine_kernel|mlp_cluster_kernel|mlp_tc_kernel|sigmoid_categorical|urm_kernel|slate_metrics_kernel|ce_tc2_kernel|ce_sparse_kernel|cand_ce_kernel|ce_kernel|score_select_kernel|gemm_tn_tc_kernel|topk_kernel'
PROBE_WARM=0 PROBE_ITERS=1 ncu --set full --clock-control none -k "regex:$KERNELS" -o $OUT/${TAG}_kernels -f \
    python profiles/probe_kernels.py > $OUT/${TAG}_probe_under_ncu.txt 2>&1
ncu -i $OUT/${TAG}_kernels.ncu-rep --page raw --csv > $OUT/${TAG}_kernels_raw.csv 2>/dev/null
ls -la $OUT/${TAG}_kernels.ncu-rep; [ $(stat -c %s $OUT/${TAG}_kernels.ncu-rep) -gt 40000000 ] && rm -f $OUT/${TAG}_kernels.ncu-rep
# launch list of the C3 training step (own backward GEMMs, tensor-core CE)
ncu --metrics gpu__time_duration.sum --clock-control none --cache-control none -c 1500 --csv \
    --log-file $OUT/${TAG}_launches_c3_train.csv python bench.py --workload c3 --mode train --steps 3 --warmup 3 \
    --no-cpu --no-also > /dev/null 2>&1
# tensor-pipe evidence of the generalised filter: D = 128 at the C4 shape
PROBE_WARM=1 PROBE_ITERS=1 ncu --set full --clock-control none -k "regex:score_select_tc_kernel" -s 1 -c 1 \
    -o $OUT/${TAG}_filter_d128 -f python profiles/probe_kernels.py select_d128 > /dev/null 2>&1
ncu -i $OUT/${TAG}_filter_d128.ncu-rep --page raw --csv > $OUT/${TAG}_filter_d128_raw.csv 2>/dev/null
# the dominant kernel with source-level stall samples
PROBE_WARM=1 PROBE_ITERS=1 ncu --set full --clock-control none --import-source on -k "regex:score_select_tc_kernel" -s 1 -c 1 \
    -o $OUT/${TAG}_filter_c4 -f python profiles/probe_kernels.py select > /dev/null 2>&1
# sanitizer: the small-shape tcgen05 / kernel tests (bit-exact checks run under the tool)
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 1 python -m pytest tests/test_gpu_tcgen05.py tests/test_gpu_kernels.py tests/test_gpu_mlp_tc.py \
    -x -q -m gpu -k "not full_size and not max_size and not big and not 4096" > $OUT/${TAG}_memcheck.txt 2>&1
echo "memcheck rc=$?" >> $OUT/${TAG}_memcheck.txt
timeout 900 compute-sanitizer --tool racecheck --error-exitcode 1 python -m pytest tests/test_gpu_tcgen05.py tests/test_gpu_mlp_tc.py \
    -x -q -m gpu -k "not full_size and not max_size and not big and not 4096 and not 1000" > $OUT/${TAG}_racecheck.txt 2>&1
echo "racecheck rc=$?" >> $OUT/${TAG}_racecheck.txt
tail -3 $OUT/${TAG}_memcheck.txt $OUT/${TAG}_racecheck.txt; cat $OUT/${TAG}_probe.txt
