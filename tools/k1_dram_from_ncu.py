"""profiles/r02_k1_dram.json from the per-launch CSV of

    ncu --profile-from-start off --cache-control none --clock-control none \
        --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --csv --log-file <csv> \
        python bench.py --one-pass --no-cpu-baseline

(one pass of the configs[3] step on one context).  Sums the DRAM bytes of every K1 launch (row bucketing, root counting,
marginalisation) and of the other kernels of the step, per kernel; bench.py divides the K1 sum by the K1 kernel time it
measures live.  usage: python tools/k1_dram_from_ncu.py <launches.csv> [out.json]"""
import collections
import csv
import json
import os
import re
import sys

K1 = re.compile(r"bic_root_kernel|cube_derive_kernel|cube_map_kernel|root_map_kernel|tree_key_kernel|tree_scatter_kernel|bic_count_smem_kernel|"
                r"bic_count_global_kernel|bic_score_tables_kernel|DeviceScan|bucket_scan_kernel|sparse_bic")
scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6,
         "nsecond": 1e-3, "usecond": 1.0, "msecond": 1e3, "second": 1e6}

rows = list(csv.reader(open(sys.argv[1])))
hdr = next(i for i, r in enumerate(rows) if r and r[0] == "ID")
h = rows[hdr]
ci = {n: h.index(n) for n in ("ID", "Kernel Name", "Metric Name", "Metric Unit", "Metric Value")}
launch = collections.OrderedDict()
for r in rows[hdr + 1:]:
    if len(r) <= ci["Metric Value"]:
        continue
    d = launch.setdefault(r[ci["ID"]], {"kernel": re.sub(r"\(.*", "", r[ci["Kernel Name"]]).replace("urlgpu::", "")})
    d[r[ci["Metric Name"]]] = float(r[ci["Metric Value"]].replace(",", "")) * scale.get(r[ci["Metric Unit"]], 1.0)

per = collections.defaultdict(lambda: {"launches": 0, "us": 0.0, "dram_read": 0.0, "dram_write": 0.0})
for d in launch.values():
    a = per[d["kernel"]]
    a["launches"] += 1
    a["us"] += d.get("gpu__time_duration.sum", 0.0)
    a["dram_read"] += d.get("dram__bytes_read.sum", 0.0)
    a["dram_write"] += d.get("dram__bytes_write.sum", 0.0)
k1 = {k: v for k, v in per.items() if K1.search(k)}
k1_bytes = sum(v["dram_read"] + v["dram_write"] for v in k1.values())
k1_us = sum(v["us"] for v in k1.values())
tot_us = sum(v["us"] for v in per.values())
for v in per.values():
    v["dram_gbps_under_ncu"] = (v["dram_read"] + v["dram_write"]) / v["us"] / 1e3 if v["us"] else None
    v["share_of_step_time"] = v["us"] / tot_us if tot_us else None
dom = max(k1.items(), key=lambda kv: kv[1]["us"])
out = {
    "source": os.path.basename(sys.argv[1]) + ": ncu --cache-control none --clock-control none, one pass of configs[3] on one context",
    "k1_dram_bytes_per_step": k1_bytes, "k1_us_under_ncu": k1_us, "k1_dram_gbps_under_ncu": k1_bytes / k1_us / 1e3 if k1_us else None,
    "step_us_under_ncu": tot_us, "k1_share_of_step_time": k1_us / tot_us if tot_us else None,
    "dominant_kernel": {"kernel": dom[0], "launches": dom[1]["launches"],
                        "dram_bytes_per_launch": (dom[1]["dram_read"] + dom[1]["dram_write"]) / dom[1]["launches"],
                        "avg_us_under_ncu": dom[1]["us"] / dom[1]["launches"], "dram_gbps_under_ncu": dom[1]["dram_gbps_under_ncu"]},
    "per_kernel": {k: v for k, v in sorted(per.items(), key=lambda kv: -kv[1]["us"])},
}
path = sys.argv[2] if len(sys.argv) > 2 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r02_k1_dram.json")
json.dump(out, open(path, "w"), indent=1)
print(f"{'kernel':48s} {'launches':>8s} {'ms':>9s} {'share':>6s} {'rd GB':>8s} {'wr GB':>8s} {'GB/s':>7s}")
for k, v in out["per_kernel"].items():
    print(f"{k[:48]:48s} {v['launches']:8d} {v['us'] / 1e3:9.2f} {v['share_of_step_time'] * 100:5.1f}% {v['dram_read'] / 1e9:8.2f} {v['dram_write'] / 1e9:8.2f} "
          f"{v['dram_gbps_under_ncu'] or 0:7.0f}")
print(f"K1: {k1_bytes / 1e9:.1f} GB DRAM in {k1_us / 1e3:.1f} ms under ncu = {out['k1_dram_gbps_under_ncu']:.0f} GB/s; step {tot_us / 1e3:.1f} ms")
