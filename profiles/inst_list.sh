#!/bin/bash
# Per-kernel executed warp instructions, issue utilisation and duration of one warm resident step (cheap metrics only).
# usage: bash profiles/inst_list.sh <tag>   (the environment is passed through, e.g. LFD_B200_LIB=<path> to measure another build)
set -u
TAG=$1
OUT=gpurun_out
CMD="python bench.py --profile --batch 64 --steps 1 --warmup 3"
export LFD_NO_GRAPH=1
timeout 900 ncu --metrics gpu__time_duration.sum,smsp__inst_executed.sum,smsp__issue_active.avg.pct_of_peak_sustained_active,sm__warps_active.avg.pct_of_peak_sustained_active,sm__cycles_active.avg,sm__cycles_elapsed.max,dram__bytes_read.sum,dram__bytes_write.sum \
  --clock-control none --csv --log-file $OUT/inst_$TAG.csv $CMD > $OUT/inst_$TAG.log 2>&1
echo "rc=$?"
python - <<PY
import csv, collections, re
rows = [l for l in open("$OUT/inst_$TAG.csv") if l.startswith('"')]
rd = list(csv.DictReader(rows))
# keep only the launches of the LAST resident step: find the last k_prep launch id
ids = [int(r["ID"]) for r in rd if "k_prep" in r["Kernel Name"]]
# steps: warmup+1 resident runs + upload run + 5 serial runs; take everything between the 5th-from-last k_prep... simpler: aggregate per kernel name over ALL launches and divide by launches of k_ctl_init
per = collections.defaultdict(lambda: collections.defaultdict(float))
cnt = collections.Counter()
for r in rd:
    name = re.sub(r"\(.*", "", r["Kernel Name"]).replace("void ", "")
    name = re.sub(r"<.*", "", name)
    m = r["Metric Name"]; v = float(r["Metric Value"].replace(",", ""))
    per[name][m] += v
    if m == "gpu__time_duration.sum": cnt[name] += 1
nsteps = cnt.get("k_ctl_init", 1)
tot_i = sum(p["smsp__inst_executed.sum"] for p in per.values()); tot_t = sum(p["gpu__time_duration.sum"] for p in per.values())
with open("$OUT/inst_${TAG}_summary.txt", "w") as f:
    f.write("per step of 64 frames (%d steps captured): %.1f M warp-instructions, %.1f us of kernel time (ncu, serialised)\n" % (nsteps, tot_i / nsteps / 1e6, tot_t / nsteps / 1e3))
    f.write("%-28s %8s %10s %8s %8s %8s %9s\n" % ("kernel", "launches", "Minst", "inst%", "us", "issue%", "busy%"))
    for name, p in sorted(per.items(), key=lambda kv: -kv[1]["smsp__inst_executed.sum"]):
        n = cnt[name]
        f.write("%-28s %8.1f %10.2f %8.1f %8.1f %8.1f %9.1f\n" % (name, n / nsteps, p["smsp__inst_executed.sum"] / nsteps / 1e6, 100 * p["smsp__inst_executed.sum"] / tot_i,
                p["gpu__time_duration.sum"] / nsteps / 1e3, p["smsp__issue_active.avg.pct_of_peak_sustained_active"] / n,
                100 * p["sm__cycles_active.avg"] / max(p["sm__cycles_elapsed.max"], 1)))
import json
json.dump({"batch": 64, "workload": "config3", "steps_captured": nsteps, "source": "ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum (profiles/inst_list.sh $TAG)",
           "unit": "bytes per 64-frame step, both passes, all launches of the kernel",
           "per_step_bytes": {name: (p["dram__bytes_read.sum"] + p["dram__bytes_write.sum"]) / nsteps for name, p in per.items()},
           "per_step_minst": {name: p["smsp__inst_executed.sum"] / nsteps / 1e6 for name, p in per.items()}},
          open("$OUT/traffic_$TAG.json", "w"), indent=1)
PY
cat $OUT/inst_${TAG}_summary.txt
