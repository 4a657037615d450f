"""The sparse-list local search (urlgpu_order_local_search_sparse) against the table form, and past the table form's limit
-> profiles/r07_order_local_search_sparse.json.

Crossover: both forms alternate call by call on the same caches, and every run checks that cost, order, parents, restart costs
and restart moves are equal bit for bit.  Caches: the r04/r05/r06 recipe (discrete_bn(p=k, n=20000, seed=40+k, window 4, at
most 3 parents), BIC at -p 3 with PRUNE_DOMINATED, no skeleton and the 2-hop skeleton) at k = 20..32, hepatitis (BIC over all
variables at the reference's default cap, pruned) and configs[3] with its generating skeleton.  Per form: the call's time (host
clock around the synchronous call, warmed, mean of 3) and the split into tables and climb (urlgpu_stats ms_order_tables /
ms_order_layers, CUDA events, a separate call).

Crossover by table size: configs[3]'s data, discrete_bn(p=60, n=1e6, seed=4), BIC at -p 3 with PRUNE_DOMINATED, no skeleton,
each variable's candidates limited to the K variables u with the largest pairwise gain n MI(v; u) - (r_v - 1)(r_u - 1) ln(n)/2,
K = 22..30, so that c_v comes close to K and the tables (4 2^c_v bytes per variable) run from about 1 GB to past the device.
Both forms as in the crossover above, with the tables' bytes; where the table form is refused, its message.

Past the limit: configs[3]'s data, discrete_bn(p=60, n=1e6, seed=4), BIC over all variables at -p 3, pruned, no skeleton, at
256 and 4096 restarts: entries per variable, the c_v distribution, the mean scan length (entries tested per look-up, counted on
the host over the best order's k look-ups), moves per restart, and the learned DAG against the generating DAG (skeleton
precision and recall, SHD, cost against the generating DAG scored with urlgpu_score_sets and summed in float32).

Size: discrete_bn(p=256, n=20000, seed=11), BIC at -p 2, pruned, no skeleton: one component of 256, four words per entry.
The card's name, power limit and SM clock are read in the same command."""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
pkg = importlib.import_module("urlearning-cpp_b200")
from measure_order_local_search import dag_compare, split, timed_calls  # noqa: E402

TABLE, SPARSE = "urlgpu_order_local_search", "urlgpu_order_local_search_sparse"


def search_entries(codes, card, cand, cap):
    """BIC caches with PRUNE_DOMINATED over the given candidate masks, scores negated into the search sign; masks as one uint64
    per entry up to 64 variables, as Python ints above"""
    p = len(card)
    eng = pkg.Engine(0)
    eng.set_discrete(codes, card)
    entries = []
    for v in range(p):
        res = eng.score_variable(v, cand[v], cap, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        m, s = res.fetch()
        res.free()
        masks = m[:, 0].copy() if p <= 64 else [pkg.words_to_mask(row) for row in m]
        entries.append((masks, (-s).astype(np.float32)))
    eng.close()
    return entries


def card_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                              check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}
    return dict(zip(q.split(","), [x.strip() for x in line.split(",")]))


def cand_bits(entries, comp):
    """c_v per variable of the component"""
    out = []
    for v, (m, _) in enumerate(entries):
        if not (comp >> v) & 1:
            continue
        u = 0
        for x in m:
            if int(x) & ~comp == 0:
                u |= int(x)
        out.append(bin(u).count("1"))
    return out


def same(a, b):
    return bool(a[0].view(np.uint32) == b[0].view(np.uint32) and a[1] == b[1] and np.array_equal(a[2], b[2]) and
                np.array_equal(a[3].view(np.uint32), b[3].view(np.uint32)) and np.array_equal(a[4], b[4]))


def crossover_one(eng, label, entries, p, edges, restarts=256):
    runs = []
    for comp in pkg.components(p, edges):
        cb = cand_bits(entries, comp)
        if len(cb) < 2:
            continue
        forms = {"table": TABLE, "sparse": SPARSE}
        res = {f: eng._order_local_search(s, entries, p, comp, edges, restarts, 0) for f, s in forms.items()}
        t = {f: [] for f in forms}
        for _ in range(3):                                          # alternating, after the warm-up calls above
            for f, s in forms.items():
                t0 = time.perf_counter()
                r = eng._order_local_search(s, entries, p, comp, edges, restarts, 0)
                t[f].append(time.perf_counter() - t0)
                assert same(r, res[f])
        run = {"cache": label, "k": len(cb), "restarts": restarts, "max_candidates": max(cb), "mean_candidates": float(np.mean(cb)),
               "entries": int(sum(len(entries[v][0]) for v in range(p) if (comp >> v) & 1)), "bit_equal": same(res["table"], res["sparse"]),
               "moves_mean": float(res["table"][4].mean())}
        for f, s in forms.items():
            run[f"{f}_call_s_mean3"] = float(np.mean(t[f]))
            sp = split(eng, lambda: eng._order_local_search(s, entries, p, comp, edges, restarts, 0))
            run[f"{f}_ms_tables"], run[f"{f}_ms_climb"] = sp["ms_tables"], sp["ms_climb"]
        print(json.dumps(run), flush=True)
        runs.append(run)
    return runs


def hepatitis_entries():
    S = importlib.import_module("urlearning-cpp_b200.search")
    path = os.path.join("/tmp", f"hep_r07_{os.getpid()}.pss")
    subprocess.check_call([os.path.join(ROOT, "urlearning-cpp_b200", "score"), os.path.join(ROOT, "tests", "data", "hepatitis.clean.csv"), path,
                           "-s", "-f", "BIC", "--quiet", "--prune"], stdout=subprocess.DEVNULL)
    cache = S.ScoreCache(path)
    entries = [cache.entries(v) for v in range(cache.p)]
    os.remove(path)
    return entries, cache.p


def crossover(eng, sizes):
    runs = []
    for k in sizes:
        codes, card, edges, _ = pkg.datagen.discrete_bn(p=k, n=20000, seed=40 + k, window=4, max_indegree=3)
        hop = [pkg.two_hop_neighbors(edges, k, v) & ~(1 << v) for v in range(k)]
        for skel_name, nb in (("none", None), ("2-hop", hop)):
            entries = search_entries(codes, card, [pkg.two_hop_neighbors(nb, k, v) for v in range(k)], 3)
            runs += crossover_one(eng, f"r04 recipe k={k} skeleton {skel_name}", entries, k, nb)
    entries, p = hepatitis_entries()
    runs += crossover_one(eng, "hepatitis, BIC, pruned", entries, p, None)
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=60, n=1_000_000, seed=4)
    cap = pkg.effective_max_parents(12, 60, 1_000_000, True)
    entries = search_entries(codes, card, [pkg.two_hop_neighbors(edges, 60, v) for v in range(60)], cap)
    runs += crossover_one(eng, f"configs[3], BIC cap {cap}, 2-hop candidates, generating skeleton", entries, 60, [int(e) for e in edges])
    return runs


def pair_gain(codes, card):
    """n MI(v; u) - (r_v - 1)(r_u - 1) ln(n) / 2 for every pair, from 2-D counts (codes [p, n])"""
    p, n = codes.shape
    g = np.full((p, p), -np.inf)
    for v in range(p):
        for u in range(v + 1, p):
            joint = np.bincount(codes[v].astype(np.int64) * card[u] + codes[u], minlength=card[v] * card[u]).reshape(card[v], card[u])
            pv, pu = joint.sum(1, keepdims=True), joint.sum(0, keepdims=True)
            nz = joint > 0
            mi = float((joint[nz] * np.log(joint[nz] * n / (pv @ pu)[nz])).sum())
            g[v, u] = g[u, v] = mi - (card[v] - 1) * (card[u] - 1) * np.log(n) / 2
    return g


def crossover_by_table_size(eng, ks, restarts=256):
    p, n = 60, 1_000_000
    codes, card, _, _ = pkg.datagen.discrete_bn(p=p, n=n, seed=4)
    g = pair_gain(np.asarray(codes), np.asarray(card))
    comp = (1 << p) - 1
    runs = []
    for K in ks:
        cand = [sum(1 << int(u) for u in np.argsort(-g[v])[:K]) | (1 << v) for v in range(p)]
        entries = search_entries(codes, card, cand, 3)
        cb = cand_bits(entries, comp)
        run = {"cache": f"configs[3] data, BIC -p 3, top {K} pairwise candidates, no skeleton", "K": K, "k": p, "restarts": restarts,
               "max_candidates": max(cb), "median_candidates": float(np.median(cb)), "table_bytes": int(sum(4 << c for c in cb)),
               "entries": int(sum(len(m) for m, _ in entries))}
        try:
            table = eng._order_local_search(TABLE, entries, p, comp, None, restarts, 0)
        except pkg.UrlGpuError as e:
            table = None
            run["table_form"] = str(e)
        sparse = eng._order_local_search(SPARSE, entries, p, comp, None, restarts, 0)
        forms = {"sparse": SPARSE} if table is None else {"table": TABLE, "sparse": SPARSE}
        if table is not None:
            run["bit_equal"] = same(table, sparse)
        t = {f: [] for f in forms}
        for _ in range(3):                                          # alternating, after the warm-up calls above
            for f, s in forms.items():
                t0 = time.perf_counter()
                eng._order_local_search(s, entries, p, comp, None, restarts, 0)
                t[f].append(time.perf_counter() - t0)
        for f, s in forms.items():
            run[f"{f}_call_s_mean3"] = float(np.mean(t[f]))
            sp = split(eng, lambda: eng._order_local_search(s, entries, p, comp, None, restarts, 0))
            run[f"{f}_ms_tables"], run[f"{f}_ms_climb"] = sp["ms_tables"], sp["ms_climb"]
        print(json.dumps(run), flush=True)
        runs.append(run)
    return runs


def scan_lengths(entries, order, comp):
    """entries tested by the list look-up for each of the order's k look-ups (the hit's position + 1, or the whole list)"""
    out = []
    U = 0
    for v in order:
        m, s = entries[v]
        q = sorted((float(s[i]), bin(int(m[i])).count("1"), int(m[i])) for i in range(len(m)) if int(m[i]) & ~comp == 0)
        n = next((i + 1 for i, e in enumerate(q) if e[2] & ~U == 0), len(q))
        out.append(n)
        U |= 1 << v
    return out


def past_limit(eng, restarts_list):
    p, n, cap = 60, 1_000_000, 3
    codes, card, _, gen_parents = pkg.datagen.discrete_bn(p=p, n=n, seed=4)
    t0 = time.perf_counter()
    entries = search_entries(codes, card, [(1 << p) - 1] * p, cap)
    score_s = time.perf_counter() - t0
    comp = (1 << p) - 1
    cb = cand_bits(entries, comp)
    per_var = [len(m) for m, _ in entries]
    truth = [sum(1 << u for u in pa) for pa in gen_parents]
    scorer = pkg.Engine(0)
    scorer.set_discrete(codes, card)
    fam, _ = scorer.score_sets(list(range(p)), truth, pkg.BIC)
    scorer.close()
    gen_cost = np.float32(0)
    for v in range(p):
        gen_cost = np.float32(gen_cost - fam[v])
    out = {"workload": f"discrete_bn(p=60, n=1e6, seed=4), BIC -p {cap} over all variables, PRUNE_DOMINATED, no skeleton",
           "scoring_s": score_s, "entries": int(sum(per_var)), "entries_per_variable": {"min": min(per_var), "median": float(np.median(per_var)),
                                                                                        "max": max(per_var)},
           "candidates": {"min": min(cb), "median": float(np.median(cb)), "max": max(cb), "above_32": int(sum(c > 32 for c in cb)),
                          "histogram": {str(c): cb.count(c) for c in sorted(set(cb))}},
           "table_form": None, "generating_dag_cost": float(gen_cost), "runs": []}
    try:
        eng._order_local_search(TABLE, entries, p, comp, None, 8, 0)
    except pkg.UrlGpuError as e:
        out["table_form"] = str(e)
    for restarts in restarts_list:
        def call():
            return eng._order_local_search(SPARSE, entries, p, comp, None, restarts, 0)
        cost, order, parents, rc, rm = call()
        times = timed_calls(call)
        sl = scan_lengths(entries, order, comp)
        run = {"restarts": restarts, "call_s": times, "call_s_mean3": float(np.mean(times)), **split(eng, call),
               "moves_mean": float(rm.mean()), "moves_max": int(rm.max()), "best_cost": float(cost), "restart_cost_median": float(np.median(rc)),
               "restarts_at_best": int((rc == cost).sum()), "scan_length_mean": float(np.mean(sl)), "scan_length_max": int(max(sl)),
               "best_minus_generating_dag_cost": float(cost) - float(gen_cost), "vs_generating_dag": dag_compare(parents, truth, p)}
        print(json.dumps(run), flush=True)
        out["runs"].append(run)
    return out


def size256(eng, restarts=256):
    p, cap = 256, 2
    codes, card, _, _ = pkg.datagen.discrete_bn(p=p, n=20000, seed=11)
    entries = search_entries(codes, card, [(1 << p) - 1] * p, cap)
    comp = (1 << p) - 1
    cb = cand_bits(entries, comp)

    def call():
        return eng._order_local_search(SPARSE, entries, p, comp, None, restarts, 0)
    cost, order, parents, rc, rm = call()
    times = timed_calls(call)
    sl = scan_lengths(entries, order, comp)
    run = {"workload": f"discrete_bn(p=256, n=20000, seed=11), BIC -p {cap} over all variables, PRUNE_DOMINATED, no skeleton",
           "restarts": restarts, "entries": int(sum(len(m) for m, _ in entries)), "max_candidates": max(cb), "median_candidates": float(np.median(cb)),
           "call_s_mean3": float(np.mean(times)), **split(eng, call), "moves_mean": float(rm.mean()), "moves_max": int(rm.max()),
           "scan_length_mean": float(np.mean(sl)), "best_cost": float(cost)}
    print(json.dumps(run), flush=True)
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--restarts", default="256,4096")
    ap.add_argument("--sizes", default="20,24,28,32")
    ap.add_argument("--top", default="22,24,26,28,30")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_order_local_search_sparse.json"))
    args = ap.parse_args()
    result = {"card": card_info(), "timing": "host clock around warmed synchronous calls, mean of 3; tables and climb by CUDA events",
              "scan": "warp-cooperative scan of the sorted list"}
    print(result["card"], flush=True)
    eng = pkg.Engine(0)
    result["crossover"] = crossover(eng, [int(x) for x in args.sizes.split(",") if x])
    result["crossover_by_table_size"] = crossover_by_table_size(eng, [int(x) for x in args.top.split(",") if x])
    result["past_limit"] = past_limit(eng, [int(x) for x in args.restarts.split(",") if x])
    result["size_256"] = size256(eng)
    result["card_after"] = card_info()
    eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
