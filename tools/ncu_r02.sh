#!/bin/bash
# Round-2 ncu evidence (run under gpurun, one GPU): launch list of the default bench + one full capture per dominant kernel.
# Every profiled command line first exits 0 without ncu (B200_PROFILING.md).
set -u
OUT=gpurun_out
B="python bench.py --steps 3 --warmup 3 --no-selfplay --no-cpu-baseline"
$B > $OUT/r2_plain_bench.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $OUT/r2_launches_bench.csv $B > $OUT/r2_ncu_launch.log 2>&1
$B > $OUT/r2_plain_bench2.log 2>&1 &&
ncu --set full --clock-control none --import-source on -k regex:k_env_step -s 4 -c 1 -o $OUT/r2_env_step -f $B > $OUT/r2_ncu_env.log 2>&1
M="python tools/mcts_time.py"
$M > $OUT/r2_plain_mcts.log 2>&1 &&
ncu --set full --clock-control none --import-source on -k regex:k_mcts_run_g -s 3 -c 1 -o $OUT/r2_mcts_run_g -f $M > $OUT/r2_ncu_mcts.log 2>&1
for P in f32 f16; do
  N="python tools/net_check.py 16384 3 $P"
  $N > $OUT/r2_plain_net_$P.log 2>&1 &&
  ncu --set full --clock-control none --import-source on -k regex:k_net_forward -s 1 -c 1 -o $OUT/r2_net_$P -f $N > $OUT/r2_ncu_net_$P.log 2>&1
done
ls -la $OUT/*.ncu-rep | tail
