"""Leaves scored in the pass that derives their parent, against a build without it -> profiles/r08_leaf_fusion.json.

A leaf is a set without cube bit 0.  This build scores every leaf of a derived table from the digit-0 groups of the pass that
derives its parent (cube_derive_kernel, or bic_root_kernel for the children of fused roots); only leaves of root tables keep
a derive pair of their own.  --base names another checkout of the project, built (`__graft_entry__.build()`), that does not.

Both trees run `bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline --no-subrecords` alternately, --rounds times each
(baseline first); the fields that matter of each run are kept.  Then both run `bench.py --dump-outputs` and the dumped files
are compared byte for byte, and each runs the default `bench.py --gpus 1` line once (sub-records included: fNML, cBIC and
the score file), which is kept whole.  The card's name, power limit and SM clocks are read in the same command."""
from __future__ import annotations

import argparse
import filecmp
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = ["--gpus", "1", "--steps", "10", "--warmup", "3", "--no-cpu-baseline", "--no-subrecords"]


def bench(tree, extra=(), args=BENCH):
    out = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), *args, *extra], cwd=tree, capture_output=True, text=True, check=True)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    return json.loads(lines[-1])


def brief(line):
    rf = line.get("roofline") or {}
    return {"ms_per_step": line.get("ms_per_step"), "value": line.get("value"), "e2e": line.get("e2e"),
            "gpu_launches": line.get("gpu_launches"), "family_ms": rf.get("family_ms"),
            "issued_bytes_per_step": rf.get("issued_bytes_per_step"), "kernel_ms_per_step": rf.get("kernel_ms_per_step")}


def same_files(a, b):
    names_a = sorted(os.listdir(a))
    names_b = sorted(os.listdir(b))
    if names_a != names_b:
        return False, f"file lists differ: {len(names_a)} vs {len(names_b)}"
    diff = [n for n in names_a if not filecmp.cmp(os.path.join(a, n), os.path.join(b, n), shallow=False)]
    return not diff, f"{len(names_a)} files, {len(diff)} differ" + (f": {diff[:5]}" if diff else "")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True, help="a built checkout without leaf scoring in the parent's pass")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_leaf_fusion.json"))
    args = ap.parse_args()
    base = os.path.abspath(args.base)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    runs = {"base": [], "new": []}
    for i in range(args.rounds):
        for name, tree in (("base", base), ("new", ROOT)):
            line = bench(tree)
            runs[name].append(line)
            print(f"round {i} {name}: {line['ms_per_step']:.1f} ms/step", flush=True)
    with tempfile.TemporaryDirectory() as td:
        da, db = os.path.join(td, "base"), os.path.join(td, "new")
        bench(base, ["--dump-outputs", da])
        bench(ROOT, ["--dump-outputs", db])
        identical, detail = same_files(da, db)
    full = {"base": bench(base, args=["--gpus", "1"]), "new": bench(ROOT, args=["--gpus", "1"])}
    med = {k: statistics.median(l["ms_per_step"] for l in v) for k, v in runs.items()}
    res = {
        "what": "configs[3] (p=60, n=1e6, 2-hop skeleton, BIC cap 11, prune), 1 GPU, bench.py " + " ".join(BENCH) + "; base and new alternate",
        "card": card,
        "median_ms_per_step": med,
        "delta_ms": med["base"] - med["new"],
        "every_new_faster_than_every_base": max(l["ms_per_step"] for l in runs["new"]) < min(l["ms_per_step"] for l in runs["base"]),
        "dump_outputs_identical": identical, "dump_outputs_detail": detail,
        "runs": {k: [brief(l) for l in v] for k, v in runs.items()},
        "default_line": full,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "median_ms_per_step", "delta_ms", "every_new_faster_than_every_base", "dump_outputs_identical", "dump_outputs_detail")}))


if __name__ == "__main__":
    main()
