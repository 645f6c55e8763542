#!/bin/bash
# ncu --set full capture of the in-kernel-policy rollout (c3) into profile_out/, on a B200 machine with Nsight Compute:
# list the launches first, then capture the second long one.
mkdir -p profile_out
CMD="python bench.py --workload c3 --only-value --steps 64 --warmup 64"
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:warp_kernel --csv --log-file profile_out/launches_c3.csv $CMD > profile_out/ncu_c3_list.log 2>&1
idx=$(python - <<'P'
import csv
rows = list(csv.reader(open("profile_out/launches_c3.csv")))
h = [i for i, r in enumerate(rows) if r and r[0] == "ID"][0]
c = rows[h]
iv = c.index("Metric Value")
long_ = [n for n, r in enumerate(rows[h + 1:]) if float(r[iv].replace(",", "")) > 2e5]
print(long_[1] if len(long_) > 1 else long_[0])
P
)
echo "capturing warp_kernel launch #$idx"
ncu --set full --clock-control none --import-source on -k regex:warp_kernel -s $idx -c 1 -f -o profile_out/prof_c3 $CMD > profile_out/ncu_c3.log 2>&1; echo "c3 rc=$?"
