#!/bin/bash
# Round-2 closing batch (one B200): GPU tests, both bench arms, the ncu launch list of one eager step and --set full captures
# of the kernels that changed last (unit-list fused / layer kernels, pruned FPS, culled ball query).  Outputs -> gpurun_out/.
cd "$(dirname "$0")/.."
O=gpurun_out
mkdir -p $O
timeout 900 python -m pytest tests -m gpu -q 2>&1 | tail -15 > $O/tests_final.log
python bench.py --impl reference --steps 10 > $O/bench_ref_final.json 2> $O/bench_ref_final.err
python bench.py > $O/bench_final.json 2> $O/bench_final.err
BENCH1="python bench.py --no-graph --pipeline 1 --no-cpu-baseline --steps 3 --warmup 3 --brackets 1"
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/launches_final.csv $BENCH1 > $O/ncu_bench_final.log 2>&1
NCU="ncu --set full --clock-control none --import-source on --launch-count 1"
cap() {  # name, kernel regex, launch-skip
  timeout 400 $NCU -k regex:$2 --launch-skip $3 -f -o $O/r02f_$1 $BENCH1 > $O/ncu_$1.log 2>&1
  python tools/ncu_export.py $O/r02f_$1.ncu-rep > $O/r02f_ncu_$1.txt 2>/dev/null
}
cap fused_l1s3_units  sa_fused_kernel        8
cap fused_l2s3_units  sa_fused_kernel        11
cap tc_l4_last_units  linear_tc_kernel       43
cap tc_l3_hoist_units linear_tc_kernel       30
cap fps_bucket_l1     fps3_bucket_kernel     1
cap bq_grid_l1        ball_query_grid_kernel 2
tail -3 $O/tests_final.log
grep -h -E "kernel:|gpu__time_duration|pipe_tensor_cycles|dram__bytes" $O/r02f_ncu_*.txt | head -40
