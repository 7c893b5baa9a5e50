#!/bin/bash
# Round profiles (B200_PROFILING.md recipe): launch list of the bench command + one --set full capture per kernel.
# Every ncu run is preceded by the same command exiting 0 without ncu.  Numbers printed under ncu are never bench values.
mkdir -p gpurun_out
R=${1:-r01}
NCU="ncu --set full --clock-control none --import-source on"
BENCH="python bench.py --steps 2 --warmup 3 --no-cpu-baseline --core-only"
$BENCH > gpurun_out/${R}_plain_bench.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/${R}_launches_bench.csv $BENCH > /dev/null 2>&1
echo "launch list rc=$?"
$NCU -k regex:k_dist_dmma -s 3 -c 1 -f -o gpurun_out/${R}_dist_dmma_c2 $BENCH > gpurun_out/${R}_ncu1.log 2>&1
echo "dist rc=$?"
$NCU -k 'regex:k_frontend$' -s 3 -c 1 -f -o gpurun_out/${R}_frontend_c2 $BENCH > gpurun_out/${R}_ncu2.log 2>&1
echo "frontend rc=$?"
C3="python tools/bench_c3.py --n-sites 100000 --reps 1"
$C3 > gpurun_out/${R}_plain_c3.log 2>&1 &&
$NCU -k regex:k_mask_count -s 2 -c 1 -f -o gpurun_out/${R}_mask_count_c3 $C3 > gpurun_out/${R}_ncu3.log 2>&1
echo "count rc=$?"
$NCU -k 'regex:k_dist_dmma' -s 2 -c 1 -f -o gpurun_out/${R}_dist_dmma_weighted_c3 $C3 > gpurun_out/${R}_ncu4.log 2>&1
echo "weighted dist rc=$?"
EM="env N_SITES=20000 python tools/bench_em.py"
$EM > gpurun_out/${R}_plain_em.log 2>&1 &&
$NCU -k regex:k_dist_em -s 1 -c 1 -f -o gpurun_out/${R}_dist_em $EM > gpurun_out/${R}_ncu5.log 2>&1
echo "em rc=$?"
C4="env N_SITES=50000 PDEL=0 python tools/bench_c4.py"
$C4 > gpurun_out/${R}_plain_c4.log 2>&1 &&
$NCU -k regex:k_dist_umma -s 1 -c 1 -f -o gpurun_out/${R}_dist_umma $C4 > gpurun_out/${R}_ncu8.log 2>&1
echo "umma rc=$?"
$NCU -k regex:k_frontend_codes -s 2 -c 1 -f -o gpurun_out/${R}_frontend_codes $C4 > gpurun_out/${R}_ncu7.log 2>&1
echo "frontend codes rc=$?"
ls -la gpurun_out | grep $R
