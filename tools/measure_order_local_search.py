"""The order-graph local search (urlgpu_order_local_search) on configs[3] itself and next to the exact search on the r04/r05
caches -> profiles/r06_order_local_search.json.

configs[3]: datagen.discrete_bn(p=60, n=1e6, seed=4), BIC over each variable's 2-hop candidates at the bench's cap (11) with
PRUNE_DOMINATED, the scores negated into the search sign, the generating skeleton (one component of 60 variables).  At
restarts = 256 and 4096 (seed 0): the call's time (host clock around the synchronous call, warmed, mean of 3), the split between
the best-parent tables and the climb (urlgpu_stats ms_order_tables / ms_order_layers, a separate timed call), restarts per
second, moves per restart, the spread of the restarts' final costs, and the learned DAG against the generating DAG (skeleton
precision and recall, SHD).  The generating DAG's own cost, its families scored with urlgpu_score_sets and summed in float32 in
search sign, is given for scale; its families need not be cache entries.

r04/r05 caches: the recipe of tools/measure_order_search.py (discrete_bn(p=k, n=20000, seed=40+k, window 4, at most 3
parents), BIC at -p 3 with PRUNE_DOMINATED, no skeleton and the 2-hop skeleton) at k = 20..32; the local search (256 restarts)
and Engine.order_search alternate call by call, and the cost gap is reported.  There is no CPU arm: the project has no host
local search.  The card's name and power limit are read in the same command."""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
pkg = importlib.import_module("urlearning-cpp_b200")
from measure_order_search import card_info  # noqa: E402


def search_entries(codes, card, cand, cap):
    """BIC caches with PRUNE_DOMINATED over the given candidate masks, scores negated into the search sign"""
    p = len(card)
    eng = pkg.Engine(0)
    eng.set_discrete(codes, card)
    entries = []
    for v in range(p):
        res = eng.score_variable(v, cand[v], cap, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        m, s = res.fetch()
        res.free()
        entries.append((m[:, 0].copy(), (-s).astype(np.float32)))
    eng.close()
    return entries


def timed_calls(fn, reps=3):
    fn()                                                            # warm-up
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t.append(time.perf_counter() - t0)
    return t


def split(eng, fn):
    eng.reset_stats()
    eng.enable_timing(True)
    fn()
    st = eng.stats()
    eng.enable_timing(False)
    return {"ms_tables": st["ms_order_tables"], "ms_climb": st["ms_order_layers"]}


def dag_compare(learned, truth, p):
    """skeleton precision / recall and SHD (missing + extra + reversed edges) of two DAGs given as parent masks"""
    le = {(a, b) for b in range(p) for a in range(p) if (int(learned[b]) >> a) & 1}
    te = {(a, b) for b in range(p) for a in range(p) if (int(truth[b]) >> a) & 1}
    ls, ts = {frozenset(e) for e in le}, {frozenset(e) for e in te}
    common = ls & ts
    reversed_ = sum(1 for a, b in le if (b, a) in te)
    return {"edges_learned": len(le), "edges_true": len(te), "skeleton_precision": len(common) / max(1, len(ls)),
            "skeleton_recall": len(common) / max(1, len(ts)), "shd": len(ls - ts) + len(ts - ls) + reversed_}


def configs3(eng, restarts_list):
    codes, card, edges, gen_parents = pkg.datagen.discrete_bn(p=60, n=1_000_000, seed=4)
    p = 60
    cap = pkg.effective_max_parents(12, p, 1_000_000, True)
    cand = [pkg.two_hop_neighbors(edges, p, v) for v in range(p)]
    t0 = time.perf_counter()
    entries = search_entries(codes, card, cand, cap)
    score_s = time.perf_counter() - t0
    comp = (1 << p) - 1
    assert pkg.components(p, edges) == [comp]
    cbits = [bin(int(np.bitwise_or.reduce(m)) if len(m) else 0).count("1") for m, _ in entries]
    truth = [sum(1 << u for u in pa) for pa in gen_parents]
    scorer = pkg.Engine(0)
    scorer.set_discrete(codes, card)
    fam, _ = scorer.score_sets(list(range(p)), truth, pkg.BIC)
    scorer.close()
    gen_cost = np.float32(0)
    for v in range(p):                                              # parents come before the child: 0..59 is an order of the DAG
        gen_cost = np.float32(gen_cost - fam[v])
    out = {"workload": f"configs[3]: discrete_bn(p=60, n=1e6, seed=4), BIC cap {cap} over 2-hop candidates, PRUNE_DOMINATED, generating skeleton",
           "scoring_s": score_s, "entries": int(sum(len(m) for m, _ in entries)), "max_candidates": max(cbits),
           "table_bytes": int(sum(4 << c for c in cbits)), "generating_dag_cost": float(gen_cost), "runs": []}
    try:
        eng.order_search(entries, p, comp, edges)
    except pkg.UrlGpuError as e:
        out["exact_search"] = str(e)
    for restarts in restarts_list:
        def call():
            return eng.order_local_search(entries, p, comp, edges, restarts=restarts, seed=0)
        cost, order, parents, rc, rm = call()
        times = timed_calls(call)
        run = {"restarts": restarts, "call_s": times, "call_s_mean3": float(np.mean(times)), **split(eng, call),
               "restarts_per_s": restarts / float(np.mean(times)), "moves_mean": float(rm.mean()), "moves_max": int(rm.max()),
               "best_cost": float(cost), "restart_cost_min": float(rc.min()), "restart_cost_median": float(np.median(rc)),
               "restart_cost_max": float(rc.max()), "restarts_at_best": int((rc == cost).sum()),
               "best_minus_generating_dag_cost": float(cost) - float(gen_cost), "vs_generating_dag": dag_compare(parents, truth, p)}
        print(json.dumps(run), flush=True)
        out["runs"].append(run)
    return out


def r04_r05_caches(eng, sizes, restarts):
    runs = []
    for k in sizes:
        codes, card, edges, _ = pkg.datagen.discrete_bn(p=k, n=20000, seed=40 + k, window=4, max_indegree=3)
        hop = [pkg.two_hop_neighbors(edges, k, v) & ~(1 << v) for v in range(k)]
        for skel_name, nb in (("none", None), ("2-hop", hop)):
            entries = search_entries(codes, card, [pkg.two_hop_neighbors(nb, k, v) for v in range(k)], 3)
            comp = (1 << k) - 1
            exact = eng.order_search(entries, k, comp, nb)
            local = eng.order_local_search(entries, k, comp, nb, restarts=restarts, seed=0)
            te, tl = [], []
            for _ in range(3):                                      # alternating, after the warm-up calls above
                t0 = time.perf_counter()
                eng.order_search(entries, k, comp, nb)
                te.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                eng.order_local_search(entries, k, comp, nb, restarts=restarts, seed=0)
                tl.append(time.perf_counter() - t0)
            run = {"k": k, "skeleton": skel_name, "restarts": restarts, "exact_cost": float(exact[0]), "local_cost": float(local[0]),
                   "gap": float(local[0]) - float(exact[0]), "bit_equal_cost": bool(exact[0].view(np.uint32) == local[0].view(np.uint32)),
                   "restarts_at_exact": int((local[3] == exact[0]).sum()), "moves_mean": float(local[4].mean()),
                   "moves_max": int(local[4].max()), "exact_s_mean3": float(np.mean(te)), "local_s_mean3": float(np.mean(tl))}
            print(json.dumps(run), flush=True)
            runs.append(run)
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--restarts", default="256,4096")
    ap.add_argument("--sizes", default="20,24,28,32")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_order_local_search.json"))
    args = ap.parse_args()
    result = {"card": card_info(), "timing": "host clock around warmed synchronous calls, mean of 3", "cpu_arm": "none: there is no host local search"}
    print(result["card"], flush=True)
    eng = pkg.Engine(0)
    result["configs3"] = configs3(eng, [int(x) for x in args.restarts.split(",") if x])
    result["r04_r05_caches"] = r04_r05_caches(eng, [int(x) for x in args.sizes.split(",") if x], 256)
    result["configs4_shape"] = "not measured"
    eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
