#!/bin/bash
# One profiling session on a B200 machine with Nsight Compute (ncu) installed, from the repository root: both bench arms,
# the ncu launch list of the default bench command and one `ncu --set full` capture per workload's rollout kernel.
# Afterwards: python profiles/summarize.py <tag>
#   usage: tools/profile_round.sh <tag> [bench|warp|tile|all]
#          -> profile_out/<tag>_bench.json, <tag>_ref.json, launches_bench.csv, prof_c{2,3,4,5}.ncu-rep
# The parts can run one at a time ("bench", "warp", "tile"); clear old profile_out/prof_*.ncu-rep first.
tag=${1:-r02}
part=${2:-all}
mkdir -p profile_out
if [ $part = bench ] || [ $part = all ]; then
  python bench.py --steps 20 --warmup 5 > profile_out/${tag}_bench.json 2> profile_out/${tag}_bench.err; echo "bench rc=$?"
  python bench.py --impl reference --steps 20 --warmup 5 > profile_out/${tag}_ref.json 2> profile_out/${tag}_ref.err; echo "reference rc=$?"
  ncu --metrics gpu__time_duration.sum --clock-control none -c 800 --csv --log-file profile_out/launches_bench.csv \
      python bench.py --steps 20 --warmup 5 --no-python-ref > profile_out/ncu_bench.log 2>&1; echo "launch list rc=$?"
fi
if [ $part = warp ] || [ $part = all ]; then
  ncu --set full --clock-control none --import-source on -k regex:warp_kernel -s 1 -c 1 -f -o profile_out/prof_c2 \
      python bench.py --workload c2 --only-value --steps 256 --warmup 256 > profile_out/ncu_c2.log 2>&1; echo "c2 rc=$?"
  tools/profile_c3.sh
fi
if [ $part = tile ] || [ $part = all ]; then
  for wl in c4 c5; do
    ncu --set full --clock-control none --import-source on -k regex:tile_rollout -s 1 -c 1 -f -o profile_out/prof_$wl \
        python bench.py --workload $wl --chunk 16 --only-value --steps 16 --warmup 16 > profile_out/ncu_$wl.log 2>&1; echo "$wl rc=$?"
  done
fi
