#!/bin/bash
# Round-2 final evidence call: ncu launch list + --set full captures (fused tile kernel cfg3 / cfg4, recompute, wire,
# the compact tile kernel the e2e step runs), SASS mnemonic summary, then the bench lines (driver flags) for cfg3 /
# cfg4 / cfg5-per-GPU and the reference arm.  usage: scripts/gpu_final_r2.sh <tag>
TAG=${1:-r02c}; OUT=gpurun_out/$TAG; mkdir -p $OUT
timeout 1500 python -m pytest tests -q -m gpu 2>&1 | grep -v "^    " | tail -6 > $OUT/pytest_gpu.txt; cat $OUT/pytest_gpu.txt
PROF="python bench.py --profile --steps 8 --warmup 3"
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $OUT/launches.csv $PROF > $OUT/ncu_launches.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:step_tile_kernel -s 6 -c 1 -f -o $OUT/prof_fused $PROF > $OUT/ncu_fused.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:step_tile_kernel -s 6 -c 1 -f -o $OUT/prof_fused_cfg4 $PROF --workload cfg4 > $OUT/ncu_fused_cfg4.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:recompute_kernel -s 4 -c 1 -f -o $OUT/prof_recompute python scripts/micro_recompute.py > $OUT/ncu_recompute.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:wire_ -c 2 -f -o $OUT/prof_wire python scripts/micro_wire.py > $OUT/ncu_wire.log 2>&1
timeout 400 ncu --set full --clock-control none --import-source on -k regex:tile_compact -s 8 -c 1 -f -o $OUT/prof_compact python bench.py --steps 3 --warmup 3 --e2e-steps 12 --no-sublegs --no-cpu-baseline > $OUT/ncu_compact.log 2>&1
for k in step_tile_kernel step_tile_compact; do
  echo "== $k"; cuobjdump -sass raft-rs_b200/libraftgpu.so 2>/dev/null | awk -v k="$k" '/Function :/{on=index($0,k)>0} on' | grep -oE "UBLKCP[.A-Z0-9]*|SYNCS[.A-Z0-9]*|REDUX[.A-Z0-9]*|UTMA[.A-Z0-9]*|BAR[.A-Z0-9]*|MEMBAR[.A-Z0-9]*|FENCE[.A-Z0-9]*|CCTL[.A-Z0-9]*" | sort | uniq -c | sort -rn | head -20
done > $OUT/sass_summary.txt 2>&1
for w in cfg3 cfg4 cfg5; do
  timeout 300 python bench.py --steps 20 --warmup 5 --workload $w > $OUT/bench_$w.json 2> $OUT/bench_$w.err
done
timeout 200 python bench.py --impl reference --steps 20 --warmup 5 > $OUT/bench_reference.json 2> $OUT/bench_reference.err
RAFTGPU_TILE_DEBUG=1 R=4 CONFIGS='RAFTGPU_TILE_SKIP=1;RAFTGPU_TILE_SKIP=3;RAFTGPU_TILE_SKIP=7' timeout 300 python scripts/micro_tile.py > $OUT/micro_tile.txt 2>&1
ls -la $OUT | tail -n 24
for w in cfg3 cfg4 cfg5; do echo "== $w"; python scripts/show_bench.py $OUT/bench_$w.json 2>&1 | tail -8; done; tail -c 600 $OUT/bench_reference.json
