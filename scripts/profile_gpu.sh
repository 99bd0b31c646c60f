#!/bin/bash
# ncu recipe of /opt/skills/guides/B200_PROFILING.md for one bench workload (run under gpurun, 1 GPU).
#   scripts/profile_gpu.sh <workload> <kernel-regex> [tag] [skip] [count]
set -u
W=${1:-c2}; K=${2:-tc2_|tc_reduce|mm_|stage_grad}; TAG=${3:-$W}; SKIP=${4:-8}; CNT=${5:-4}
CMD="python bench.py --workload $W --steps 3 --warmup 3 --no-cpu-baseline"
mkdir -p gpurun_out
$CMD > gpurun_out/plain_$TAG.log 2>&1 || { echo "plain run failed"; tail -5 gpurun_out/plain_$TAG.log; exit 1; }
tail -c 600 gpurun_out/plain_$TAG.log; echo
ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv --log-file gpurun_out/launches_$TAG.csv $CMD > gpurun_out/ncu_list_$TAG.log 2>&1
echo "launch list rc=$?"
ncu --set full --clock-control none --import-source on -k regex:"$K" -s $SKIP -c $CNT -f -o gpurun_out/prof_$TAG $CMD > gpurun_out/ncu_full_$TAG.log 2>&1
echo "full capture rc=$?"; ls -la gpurun_out | grep $TAG
