"""urlgpu_order_search with the one layer sweep (two cost layers in colex rank, a leaf byte per node) against a build that
stores every node's cost and leaf (5 bytes a node) at k <= 32 -> profiles/r09_order_search_one_form.json.

--base names another checkout of the project, built (`__graft_entry__.build()`), with the 5-byte-a-node form behind
urlgpu_order_search.  Inputs: the recipe of tools/measure_order_search.py (datagen.discrete_bn(p=k, n=20000, seed=40+k,
window 4, at most 3 parents), BIC at -p 3 with PRUNE_DOMINATED, written as a .pss and read back by search.ScoreCache) at
k = 12, 16, 20, 24, 28, 30 and 32, with no skeleton and with the data's 2-hop skeleton; the caches are built once, by this
tree, and both trees search the same ones.

Each tree runs in a child process of its own, and base runs in two (base and base_again), so the base-vs-base difference
is measured in the same run.  For every cache and round the three children take turns (the first of them rotates from round
to round); a turn is one warm-up call, three calls timed by the host clock around the synchronous call, and one call with
urlgpu_stats timing for the split between the best-parent tables (ms_order_tables) and the layer sweeps (ms_order_layers).
The cost bits, order and parents of every call are compared across the children.  The card's name and power limit are read
in the same command."""
from __future__ import annotations

import argparse
import importlib
import json
import os
import pickle
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYMBOL = "urlgpu_order_search"
TAG = "@order@ "                                                     # marks a child's answer among anything else on stdout


def card_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def load(tree):
    sys.path.insert(0, tree)
    return importlib.import_module("urlearning-cpp_b200")


# ------------------------------------------------------------------------------------------------ child: one tree
def serve(tree):
    """reads one case file per line on stdin, answers one JSON line per case on stdout"""
    import numpy as np
    pkg = load(tree)
    eng = pkg.Engine(0)
    for line in sys.stdin:
        with open(line.strip(), "rb") as f:
            entries, k, comp, nb = pickle.load(f)
        eng._order_search(SYMBOL, entries, k, comp, nb)                # warm-up
        times, results = [], []
        for _ in range(3):
            t0 = time.perf_counter()
            results.append(eng._order_search(SYMBOL, entries, k, comp, nb))
            times.append(time.perf_counter() - t0)
        eng.reset_stats()
        eng.enable_timing(True)
        results.append(eng._order_search(SYMBOL, entries, k, comp, nb))
        st = eng.stats()
        eng.enable_timing(False)
        outs = {json.dumps([int(np.float32(c).view(np.uint32)), [int(x) for x in o], [int(x) for x in np.asarray(p).reshape(-1)]])
                for c, o, p in results}
        cost, order, parents = json.loads(outs.pop()) if len(outs) == 1 else (None, None, None)
        print(TAG + json.dumps({"call_s": times, "ms_tables": st["ms_order_tables"], "ms_layers": st["ms_order_layers"],
                                "cost_bits": cost, "order": order, "parents": parents}), flush=True)
    eng.close()


# ------------------------------------------------------------------------------------------------ parent
def build_cases(sizes, n, tmp):
    """the caches of tools/measure_order_search.py, one pickle (entries, k, comp, skeleton rows) per (k, skeleton)"""
    import numpy as np
    pkg = load(ROOT)
    search = importlib.import_module("urlearning-cpp_b200.search")
    cases = []
    for k in sizes:
        codes, card, edges, _ = pkg.datagen.discrete_bn(p=k, n=n, seed=40 + k, window=4, max_indegree=3)
        hop = [pkg.two_hop_neighbors(edges, k, v) & ~(1 << v) for v in range(k)]
        for skel_name in ("none", "2-hop"):
            nb = hop if skel_name == "2-hop" else None
            scorer = pkg.Engine(0)
            scorer.set_discrete(codes, card)
            caches = {}
            for v in range(k):
                res = scorer.score_variable(v, pkg.two_hop_neighbors(nb, k, v), 3, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
                caches[v] = res.fetch()
                res.free()
            scorer.close()
            pss = os.path.join(tmp, f"k{k}_{skel_name}.pss")
            pkg.pss.write_pss(pss, "bn.csv", n, 3, "BIC", [f"X{v}" for v in range(k)], card, caches)
            cache = search.ScoreCache(pss)
            entries = [cache.entries(v) for v in range(k)]
            comp = (1 << k) - 1
            assert pkg.components(k, nb) == [comp], f"k={k}: the skeleton is not connected"
            path = os.path.join(tmp, f"k{k}_{skel_name}.pkl")
            with open(path, "wb") as f:
                pickle.dump((entries, k, comp, nb), f)
            cand_bits = [bin(int(np.bitwise_or.reduce(m)) if len(m) else 0).count("1") for m, _ in entries]
            cases.append({"k": k, "skeleton": skel_name, "path": path, "entries": int(sum(len(m) for m, _ in entries)),
                          "max_candidates": max(cand_bits)})
    return cases


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", help="a built checkout whose urlgpu_order_search stores 5 bytes a node")
    ap.add_argument("--sizes", default="12,16,20,24,28,30,32")
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_order_search_one_form.json"))
    ap.add_argument("--serve", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.serve:
        return serve(args.serve)
    if not args.base:
        ap.error("--base is required")
    base = os.path.abspath(args.base)
    card = card_info()
    print(card, flush=True)
    tmp = tempfile.mkdtemp(prefix="order_one_form_")
    cases = build_cases([int(x) for x in args.sizes.split(",")], args.n, tmp)
    names = ["base", "new", "base_again"]
    trees = {"base": base, "new": ROOT, "base_again": base}
    kids = {nm: subprocess.Popen([sys.executable, os.path.abspath(__file__), "--serve", trees[nm]], stdin=subprocess.PIPE,
                                 stdout=subprocess.PIPE, text=True, cwd=tmp) for nm in names}
    runs = []
    try:
        for case in cases:
            got = {nm: [] for nm in names}
            for r in range(args.rounds):
                for nm in names[r % 3:] + names[:r % 3]:
                    kids[nm].stdin.write(case["path"] + "\n")
                    kids[nm].stdin.flush()
                    line = ""
                    while not line.startswith(TAG):
                        line = kids[nm].stdout.readline()
                        if not line:
                            raise RuntimeError(f"the {nm} child ended at k = {case['k']}")
                    got[nm].append(json.loads(line[len(TAG):]))
            outs = {json.dumps([g["cost_bits"], g["order"], g["parents"]]) for v in got.values() for g in v}
            first = got["new"][0]
            run = {key: case[key] for key in ("k", "skeleton", "entries", "max_candidates")}
            run["identical"] = len(outs) == 1 and first["cost_bits"] is not None
            run["cost_bits"] = first["cost_bits"]
            for nm in names:
                run[nm] = {"call_ms": [1e3 * statistics.mean(g["call_s"]) for g in got[nm]],
                           "ms_tables": [g["ms_tables"] for g in got[nm]], "ms_layers": [g["ms_layers"] for g in got[nm]]}
            for field in ("call_ms", "ms_layers"):
                b = run["base"][field] + run["base_again"][field]
                med_b, med_n = statistics.median(b), statistics.median(run["new"][field])
                run[f"{field}_median"] = {"base": med_b, "new": med_n}
                run[f"{field}_base_spread"] = max(b) - min(b)
                run[f"{field}_base_vs_base"] = statistics.median(run["base_again"][field]) - statistics.median(run["base"][field])
                run[f"{field}_new_minus_base"] = med_n - med_b
                run[f"{field}_new_slower_than_spread"] = med_n - med_b > max(b) - min(b)
            print(json.dumps({key: run[key] for key in ("k", "skeleton", "identical", "call_ms_median", "ms_layers_median",
                                                         "call_ms_base_spread", "ms_layers_base_spread")}), flush=True)
            runs.append(run)
    finally:
        for p in kids.values():
            p.stdin.close()
        for p in kids.values():
            p.wait(timeout=120)
    res = {"what": f"{SYMBOL} on the caches of tools/measure_order_search.py; base (two children) and new alternate, "
                   f"{args.rounds} rounds; call_ms: host clock around the synchronous call, mean of 3 per round",
           "card": card, "all_identical": all(r["identical"] for r in runs),
           "any_new_slower_than_spread": any(r["call_ms_new_slower_than_spread"] or r["ms_layers_new_slower_than_spread"] for r in runs),
           "runs": runs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for name in os.listdir(tmp):
        os.remove(os.path.join(tmp, name))
    os.rmdir(tmp)
    print(json.dumps({key: res[key] for key in ("card", "all_identical", "any_new_slower_than_spread")}))


if __name__ == "__main__":
    main()
