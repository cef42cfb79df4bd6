#!/bin/bash
# Round-end evidence on one B200 (under gpurun):  tools/profile_round.sh <tag>   -> files under gpurun_out/
#   bench line of the driver's regime, ncu launch list of the same command, full captures of the step kernel in the cold
#   (launch 13 after the reset) and steady (10th launch after the 600-step pre-roll) regimes and of the fused rollout kernel
#   (all observations written) cold and steady, compute-sanitizer memcheck + initcheck of the edge-case parity tests.
TAG=${1:-r02}
O=gpurun_out
python bench.py --steps 20 --warmup 5 > $O/bench_$TAG.json 2> $O/bench_$TAG.err || { tail -5 $O/bench_$TAG.err; exit 1; }
python bench.py --steps 1000 --warmup 50 > $O/bench_${TAG}_long.json 2> $O/bench_${TAG}_long.err
CMD="python bench.py --steps 20 --warmup 5 --no-extras --e2e-steps 3"
$CMD > $O/plain_$TAG.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -c 200 --csv --log-file $O/launches_$TAG.csv $CMD > $O/ncu_l_$TAG.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:step_tpe -s 12 -c 1 -o $O/prof_step_${TAG}_cold $CMD > $O/ncu_fc_$TAG.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:step_tpe -s 35 -c 1 -o $O/prof_step_${TAG}_steady $CMD > $O/ncu_fs_$TAG.log 2>&1
RC="python tools/rollout_bench.py --T 32 --reps 2 --only all_obs"
ncu --set full --clock-control none --import-source on -k regex:rollout -s 1 -c 1 -o $O/prof_rollout_${TAG}_cold $RC > $O/ncu_rc_$TAG.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:rollout -s 19 -c 1 -o $O/prof_rollout_${TAG}_steady $RC --preroll 576 > $O/ncu_rs_$TAG.log 2>&1
# the reports stay on the box (gpurun brings back at most 64 MiB): summaries, raw metric tables and per-line instruction /
# stall-sample tables are made here
for r in step_${TAG}_cold step_${TAG}_steady rollout_${TAG}_cold rollout_${TAG}_steady; do
  case $r in step_*) N=1048576; K=15step_tpe_kernelE;; *) N=33554432; K=rollout_tpe_kernelILb0E;; esac
  python tools/ncu_summary.py $O/prof_$r.ncu-rep $N > $O/${r}_summary.txt 2>&1
  ncu -i $O/prof_$r.ncu-rep --page raw --csv > $O/${r}_details.csv 2>/dev/null
  python tools/sass_lines.py $O/prof_$r.ncu-rep $K $N 60 > $O/${r}_lines.txt 2>&1
  NAV3D_SORT=samples python tools/sass_lines.py $O/prof_$r.ncu-rep $K $N 40 > $O/${r}_stall_lines.txt 2>&1
  rm -f $O/prof_$r.ncu-rep
done
# compute-sanitizer is closed on this GPU pool ("runs under it have left GPUs needing a reset"): the memory-safety evidence is
# tools/emu_asan.sh (the device source under ASan + UBSan on the host), logged in profiles/sanitizer_r02.txt
ls -la $O/*$TAG*
