#!/bin/bash
# Evidence run of a round on one B200 (under gpurun): the contract benchmark, the reference arm, BASELINE's five
# configurations, then the ncu captures profiles/summarize.py turns into profiles/<tag>_*.md.  Every ncu pass runs a
# command line that has just exited 0 without ncu; numbers printed under ncu are never bench values.
#   bash benchmarks/profile_round.sh r01e
set -u
TAG=${1:-r01x}
OUT=gpurun_out
mkdir -p $OUT
python bench.py > $OUT/bench_$TAG.log 2>&1; echo "bench rc=$?"; tail -1 $OUT/bench_$TAG.log | cut -c1-400
python bench.py --impl reference --steps 2 --warmup 1 > $OUT/bench_ref_$TAG.log 2>&1; echo "reference arm rc=$?"; tail -1 $OUT/bench_ref_$TAG.log | cut -c1-300
python benchmarks/configs.py --only c1,c1_graph,c2,c2_graph,c3,c3_graph,c4,c4_graph,c5,c5_graph > $OUT/configs_$TAG.log 2>&1; echo "configs rc=$?"
python benchmarks/timeline.py > $OUT/timeline_$TAG.log 2>&1; echo "timeline rc=$?"
SMALL="python bench.py --no-cpu-baseline --no-configs --no-stock --steps 2 --warmup 1 --views-per-rank 2"
$SMALL > $OUT/plain_$TAG.log 2>&1; echo "plain rc=$?"
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv --log-file $OUT/launches_$TAG.csv $SMALL > $OUT/ncu_launches_$TAG.log 2>&1; echo "launch list rc=$?"
timeout 600 ncu --set full --clock-control none --import-source on -k regex:'raster_.wd_fast' -s 6 -c 2 -f -o $OUT/prof_raster_$TAG $SMALL > $OUT/ncu_raster_$TAG.log 2>&1; echo "raster capture rc=$?"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'project_|sh_|onesweep|tile_query|full_cumsum|radix_hist|find_ranges|depth_keys|raster_pack|raster_bwd_moments|camera_position|gather_rows|raster_cull_mask' -s 96 -c 25 -f -o $OUT/prof_points_$TAG $SMALL > $OUT/ncu_points_$TAG.log 2>&1; echo "point kernel capture rc=$?"
# BASELINE config 3 (6 M gaussians, visibility + heuristics): the VIS forward / HEUR backward instantiations
C3="python benchmarks/variants.py --scene c3 --rounds 1 --iters 2"
$C3 > $OUT/c3_plain_$TAG.log 2>&1; echo "c3 plain rc=$?"
timeout 600 ncu --set full --clock-control none --import-source on -k regex:'raster_fwd_fast|raster_bwd_fast' -s 4 -c 2 -f -o $OUT/prof_c3_$TAG $C3 > $OUT/ncu_c3_$TAG.log 2>&1; echo "c3 capture rc=$?"
ls -la $OUT/*$TAG*
