#!/usr/bin/env python
"""Turn the ncu artefacts that tools/profile_round.sh writes to profile_out/ into the tracked summaries under profiles/.

usage: python profiles/summarize.py r02
Reads (whatever exists):
  profile_out/launches_bench.csv (and launches_c2/c4/c5.csv)   `ncu --metrics gpu__time_duration.sum ...` launch lists
  profile_out/prof_c2.ncu-rep                      `ncu --set full` capture of wf::warp_kernel (c2, 256 steps per launch)
  profile_out/prof_c4.ncu-rep, prof_c5.ncu-rep     captures of wf::tile_rollout_kernel (c4 / c5, 16 steps per launch)
  profile_out/prof_c3.ncu-rep                      capture of wf::warp_kernel<..., MLP> (c3, 64 steps per launch; tools/profile_c3.sh)
Writes profiles/<round>_*.{csv,txt,json} and profiles/ncu_traffic.json (DRAM bytes per STEP, read by bench.py).
"""
import collections
import csv
import json
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GO = os.path.join(ROOT, "profile_out")
PR = os.path.join(ROOT, "profiles")

KEEP = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum", "dram__throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__throughput.avg.pct_of_peak_sustained_elapsed", "smsp__inst_executed.sum", "sm__inst_executed.avg.per_cycle_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "launch__registers_per_thread", "launch__grid_size",
        "launch__block_size", "launch__occupancy_limit_registers", "l1tex__t_sector_hit_rate.pct", "lts__t_sector_hit_rate.pct",
        "smsp__thread_inst_executed_per_inst_executed.ratio", "launch__shared_mem_per_block_static"]


def ncu(*args):
    return subprocess.run(["ncu", *args], capture_output=True, text=True).stdout


def launch_summary(name, rnd):
    src = os.path.join(GO, f"launches_{name}.csv")
    if not os.path.isfile(src):
        return None
    shutil.copy(src, os.path.join(PR, f"{rnd}_{name}_launches.csv"))
    rows = list(csv.reader(open(src)))
    hdr = [i for i, r in enumerate(rows) if r and r[0] == "ID"][0]
    cols = rows[hdr]
    im, iv, ik = cols.index("Metric Name"), cols.index("Metric Value"), cols.index("Kernel Name")
    t = collections.defaultdict(list)
    for r in rows[hdr + 1:]:
        if r[im] == "gpu__time_duration.sum":
            t[r[ik].split("(")[0].replace("void ", "")].append(float(r[iv].replace(",", "")))
    tot = sum(sum(v) for v in t.values())
    out = {k: {"launches": len(v), "avg_us": sum(v) / len(v) / 1e3, "share_pct": 100 * sum(v) / tot}
           for k, v in sorted(t.items(), key=lambda kv: -sum(kv[1]))}
    return out


def rep_summary(rep, rnd, tag):
    path = os.path.join(GO, rep)
    if not os.path.isfile(path):
        return None
    open(os.path.join(PR, f"{rnd}_{tag}_details.txt"), "w").write(ncu("-i", path, "--page", "details"))
    raw = list(csv.reader(ncu("-i", path, "--page", "raw", "--csv").splitlines()))
    h, units = raw[0], raw[1]
    kernels = []
    for r in raw[2:]:
        d = {"kernel": r[h.index("Kernel Name")]}
        for k in KEEP:
            if k in h:
                d[k] = {"value": r[h.index(k)], "unit": units[h.index(k)]}
        kernels.append(d)
    src_csv = os.path.join("/tmp", f"{tag}_src.csv")
    open(src_csv, "w").write(ncu("-i", path, "--page", "source", "--csv", "--print-source", "cuda,sass"))
    by_line = subprocess.run([sys.executable, os.path.join(PR, "ncu_by_line.py"), src_csv, "30"], capture_output=True, text=True).stdout
    open(os.path.join(PR, f"{rnd}_{tag}_by_line.txt"), "w").write(by_line)
    return kernels


def to_bytes(m):
    v, u = float(m["value"].replace(",", "")), m["unit"].lower()
    return v * {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(u, 1)


def main(rnd):
    summary, traffic = {}, {}
    tpath = os.path.join(PR, "ncu_traffic.json")
    if os.path.isfile(tpath):
        traffic = json.load(open(tpath))
    for name in ("bench", "c2", "c4", "c5"):
        ls = launch_summary(name, rnd)
        if ls:
            summary[f"{name}_launch_list"] = ls
    for rep, tag, key, steps in (("prof_c2.ncu-rep", "c2_warp_kernel", "c2", 256), ("prof_c4.ncu-rep", "c4_tile_rollout", "c4", 16),
                                 ("prof_c5.ncu-rep", "c5_tile_rollout", "c5", 16),
                                 ("prof_c3.ncu-rep", "c3_warp_kernel_mlp", "c3", 64)):  # in-kernel Q-network (tools/profile_c3.sh)
        ks = rep_summary(rep, rnd, tag)
        if ks:
            summary[tag] = ks
            if "dram__bytes_read.sum" in ks[0]:
                per_launch = sum(to_bytes(k["dram__bytes_read.sum"]) + to_bytes(k["dram__bytes_write.sum"]) for k in ks) / len(ks)
                traffic[key] = {"dram_bytes_per_step": per_launch / steps,
                                "source": f"profiles/{rnd}_{tag}_details.txt ({steps}-step launch, ncu --set full)"}
    json.dump(summary, open(os.path.join(PR, f"{rnd}_summary.json"), "w"), indent=1)
    json.dump(traffic, open(tpath, "w"), indent=1)
    print(json.dumps(traffic, indent=1))
    print("wrote", os.path.join(PR, f"{rnd}_summary.json"))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "r01")
