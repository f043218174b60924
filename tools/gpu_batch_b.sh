#!/bin/bash
# Round-2 measurement batch (run on the GPU box through gpurun): sweeps, probes, sanitizer, ncu.  Outputs -> gpurun_out/.
cd "$(dirname "$0")/.."
O=gpurun_out
mkdir -p $O
export PYTHONUNBUFFERED=1
timeout 600 python tools/sweeps.py fps $O/r02_sweep_fps.json > $O/sweep_fps.log 2>&1
timeout 600 python tools/sweeps.py bq $O/r02_sweep_bq.json > $O/sweep_bq.log 2>&1
timeout 300 python tools/ffps_agreement.py 32 $O/r02_ffps_agreement.json > $O/ffps_agreement.log 2>&1
timeout 300 python tools/time_ops.py $O/r02_time_ops.json > $O/time_ops.log 2>&1
# phase profiles of the tensor-core kernels (instrumented build)
SSD3D_LIB=3dssd_b200/libssd3d_prof.so timeout 300 python tools/tc_probe.py 9 10 11 1 2 3 > $O/tc_prof.log 2>&1
SSD3D_LIB=3dssd_b200/libssd3d_prof.so timeout 300 python tools/fused_probe.py 0 1 2 3 > $O/fused_prof.log 2>&1
# A/B: compile-time-shape kernels vs the run-time-shape kernel (dev-hook build)
for a in "" "dyn=1" ; do SSD3D_LIB=3dssd_b200/libssd3d_dev.so timeout 120 python tools/fused_probe.py 0 1 2 3 $a >> $O/fused_ab.log 2>&1; done
# sanitizer (small shapes)
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 python tools/sanitize_probe.py > $O/r02_sanitizer_memcheck.txt 2>&1; echo "exit $?" >> $O/r02_sanitizer_memcheck.txt
timeout 900 compute-sanitizer --tool racecheck --error-exitcode 9 python tools/sanitize_probe.py > $O/r02_sanitizer_racecheck.txt 2>&1; echo "exit $?" >> $O/r02_sanitizer_racecheck.txt
# launch list of one eager step (throughput schedule and latency schedule)
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/launches_r02.csv python bench.py --no-graph --pipeline 1 --no-cpu-baseline --steps 3 --warmup 3 --brackets 1 > $O/ncu_bench.log 2>&1
cat $O/fused_ab.log; tail -3 $O/sweep_fps.log $O/sweep_bq.log $O/tc_prof.log $O/fused_prof.log
tail -4 $O/r02_sanitizer_memcheck.txt $O/r02_sanitizer_racecheck.txt
