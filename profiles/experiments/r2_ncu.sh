#!/bin/bash
# Round-2 ncu captures (one gpurun call).  Every command first runs plain; ncu only after it exited 0.
set -x
O=gpurun_out
B="python bench.py --steps 20 --warmup 5 --no-extra --no-cpu --ramp-ms 0 --e2e-steps 0"
NCU="ncu --set full --clock-control none --import-source on"
$B --config c3 > $O/r2_plain_c3.log 2>&1 || exit 1
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/r2_launches_c3.csv $B --config c3 > $O/r2_ncu_launches.log 2>&1
$NCU -k regex:step_kernel -s 40 -c 2 -o $O/r2_step_c3 $B --config c3 > $O/r2_ncu_c3.log 2>&1
$NCU --cache-control none -k regex:step_kernel -s 40 -c 2 -o $O/r2_step_c3_warm $B --config c3 > $O/r2_ncu_c3w.log 2>&1
$B --config c4 > $O/r2_plain_c4.log 2>&1 && $NCU -k regex:wide_step_kernel -s 40 -c 2 -o $O/r2_step_c4 $B --config c4 > $O/r2_ncu_c4.log 2>&1
$NCU --cache-control none -k regex:wide_step_kernel -s 40 -c 2 -o $O/r2_step_c4_warm $B --config c4 > $O/r2_ncu_c4w.log 2>&1
$B --config c2 > $O/r2_plain_c2.log 2>&1 && $NCU --cache-control none -k regex:step_kernel -s 40 -c 2 -o $O/r2_step_c2_warm $B --config c2 > $O/r2_ncu_c2.log 2>&1
T="python profiles/experiments/r2_targets.py"
for w in observe valid goal; do
  $T $w > $O/r2_plain_$w.log 2>&1 && $NCU -k regex:${w}_kernel -s 1 -c 1 -o $O/r2_$w $T $w > $O/r2_ncu_$w.log 2>&1
done
$T bfs_local > $O/r2_plain_bfs_local.log 2>&1 && $NCU -k regex:bfs_local_kernel -s 1 -c 1 -o $O/r2_bfs_local $T bfs_local > $O/r2_ncu_bfs_local.log 2>&1
$T bfs_hash > $O/r2_plain_bfs_hash.log 2>&1 && $NCU -k regex:bfs_hash_insert_kernel -s 12 -c 1 -o $O/r2_bfs_insert $T bfs_hash > $O/r2_ncu_bfs_insert.log 2>&1
$NCU -k regex:bfs_expand_kernel -s 12 -c 1 -o $O/r2_bfs_expand $T bfs_hash > $O/r2_ncu_bfs_expand.log 2>&1
# gpurun brings back at most 64 MiB: export the pages here, keep only the headline report
for r in $O/r2_*.ncu-rep; do
  b=${r%.ncu-rep}
  ncu -i $r --page raw --csv > ${b}_raw.csv 2>/dev/null
  ncu -i $r --page source --csv > ${b}_source.csv 2>/dev/null
  case $r in *r2_step_c3.ncu-rep) ;; *) rm -f $r ;; esac
done
ls -la $O | tail -40
