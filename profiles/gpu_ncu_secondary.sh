#!/bin/bash
# ncu --set full captures of the secondary kernels (trace write-out, N-wave comb and table kernels) and of the
# z-segment scheduler on the shard one of 8 GPUs gets (125 000 points).  Usage: bash profiles/gpu_ncu_secondary.sh [cases...]
set -u
OUT=gpurun_out
mkdir -p $OUT
CASES=${@:-"seg125k comb1024 comb trace table"}
for c in $CASES; do
  case $c in trace) K=yaman4_fast;; comb*) K=nwave_comb;; table*) K=nwave_rk4;; seg125k) K=yaman4_sweep;; esac
  if [ $c = seg125k ]; then CMD="python bench.py --steps 2 --warmup 3 --shard-of 8 --no-cpu-baseline --no-secondary"; SKIP=3
  else CMD="python tools/profile_cases.py $c"; SKIP=1; fi
  $CMD > $OUT/plain_$c.log 2>&1 &&
  ncu --set full --clock-control none --import-source on -k regex:$K -s $SKIP -c 1 -f -o $OUT/prof_$c $CMD > $OUT/ncu_$c.log 2>&1
  echo "$c rc=$?"
  python tools/ncu_summary.py $OUT/prof_$c.ncu-rep $OUT/ncu_summary_$c.csv > /dev/null 2>&1
done
ls -la $OUT | grep "prof_\|ncu_summary"
