#!/bin/bash
# One-GPU check on a B200: parity tests, smoke, the default bench line, bench lines of the
# other configs, the ncu launch list and full captures of the hot kernels (steady state).
# Usage (from the repo root, under gpurun):  bash tools/final_check.sh <tag> [quick]
tag=${1:-x}
out=gpurun_out
mkdir -p $out
python -m pytest tests -m gpu -x -q -s > $out/pytest_gpu_$tag.log 2>&1; tail -3 $out/pytest_gpu_$tag.log
python __graft_entry__.py smoke > $out/smoke_$tag.log 2>&1; tail -1 $out/smoke_$tag.log
python bench.py > $out/bench_${tag}_c2.json 2> $out/bench_${tag}_c2.err; tail -3 $out/bench_${tag}_c2.err
for c in c3 c4 c5; do
  python bench.py --no-e2e --no-cpu --config $c --steps 10 --warmup 3 > $out/bench_${tag}_$c.json 2> $out/bench_${tag}_$c.err
done
python tools/bench_brief.py $out/bench_${tag}_c*.json
[ "$2" = quick ] && exit 0
args="--no-e2e --no-cpu --no-stream-all --no-bruteforce --steps 3 --warmup 3"
python bench.py $args > $out/plain_$tag.log 2>&1 &&
timeout 300 ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -c 500 --csv \
  --log-file $out/launches_$tag.csv python bench.py $args > $out/ncu1_$tag.log 2>&1
# steady-state iterations of a fit, caches left as the previous kernels left them (what a fit sees)
timeout 300 ncu --set full --clock-control none --cache-control none --import-source on -k regex:lloyd_step -s 47 -c 2 -f \
  -o $out/prof_step_$tag python bench.py $args > $out/ncu2_$tag.log 2>&1
# the once-per-cloud kernels and the final pass
timeout 300 ncu --set full --clock-control none --import-source on \
  -k regex:"raster_gather|unproject_fused|lloyd_final|raster_index" -s 10 -c 5 -f \
  -o $out/prof_build_$tag python bench.py $args > $out/ncu3_$tag.log 2>&1
# many centroids (config 4, k = 1024): FMA pipe and issue rates of the step kernel
args4="--no-e2e --no-cpu --no-stream-all --no-bruteforce --config c4 --steps 3 --warmup 3"
python bench.py $args4 > $out/plain4_$tag.log 2>&1 &&
timeout 300 ncu --set full --clock-control none --cache-control none --import-source on -k regex:lloyd_step -s 25 -c 1 -f \
  -o $out/prof_step_c4_$tag python bench.py $args4 > $out/ncu4_$tag.log 2>&1
tail -1 $out/ncu4_$tag.log
