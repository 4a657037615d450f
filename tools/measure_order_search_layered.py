"""The layered order-graph search (urlgpu_order_search_layered) next to the dense one (urlgpu_order_search) and the host
A* -> profiles/r05_order_search_layered.json.

Inputs: the recipe of tools/measure_order_search.py (datagen.discrete_bn data, window 4, at most 3 parents, BIC at -p 3
with PRUNE_DOMINATED, written as a .pss and read back by search.ScoreCache), with no skeleton and with the data's 2-hop
skeleton.  At k = 24, 28, 30 and 32 both forms run on the same caches, alternating call by call, and their cost, order and
parents are compared bit for bit; at k = 33..36 only the layered form runs, and a refusal for want of free device memory
is recorded as such.

Per form and run: the call's time (host clock around the synchronous search, warmed, mean of 3), the split between the
best-parent tables and the layer sweeps (urlgpu_stats ms_order_tables / ms_order_layers, a separate timed call), the
algorithmic bytes of the sweep (8 k 2^(k-1): a 4-byte cost and a 4-byte table entry per (S, v) pair) over the sweep time,
and the device bytes the call asks for.  The host A* (list) runs on the same cache in a child process under an
address-space limit and a wall-clock budget.  The card's name, power limit and free memory are read in the same command."""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
pkg = importlib.import_module("urlearning-cpp_b200")
search = importlib.import_module("urlearning-cpp_b200.search")
from measure_order_search import card_info, run_astar  # noqa: E402

DENSE, LAYERED = "urlgpu_order_search", "urlgpu_order_search_layered"


def free_memory():
    out = subprocess.run(["nvidia-smi", "--query-gpu=memory.free,memory.total", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def device_bytes(form, k, cand_bits, n_ent):
    """what the call asks for (include/urlgpu.h); the entries are the ones inside the component"""
    tables = sum(4 << c for c in cand_bits)
    if form == DENSE:
        return 5 * 2 ** k + tables + 16 * n_ent + k * 24 + k * 1024 + 33 * 33 * 4 + (2 + 2 * k) * 4
    return 2 ** k + 8 * math.comb(k, k // 2) + tables + 16 * n_ent + 1328 * k + 10960


def timed(eng, form, entries, k, comp, nb):
    eng.reset_stats()
    eng.enable_timing(True)
    eng._order_search(form, entries, k, comp, nb)
    st = eng.stats()
    eng.enable_timing(False)
    alg = 8.0 * k * 2 ** (k - 1)
    return {"ms_tables": st["ms_order_tables"], "ms_layers": st["ms_order_layers"], "algorithmic_bytes": alg,
            "algorithmic_GBps": alg / (st["ms_order_layers"] / 1e3) / 1e9 if st["ms_order_layers"] > 0 else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--both", default="24,28,30,32", help="sizes run with both forms")
    ap.add_argument("--layered", default="33,34,35,36", help="sizes run with the layered form only")
    ap.add_argument("--skeletons", default="none,2-hop")
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--astar-budget", type=float, default=30.0)
    ap.add_argument("--astar-mem-gb", type=float, default=64.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_order_search_layered.json"))
    args = ap.parse_args()
    result = {"card": card_info(), "memory_free_total": free_memory(), "astar_budget_s": args.astar_budget, "runs": []}
    print(result["card"], result["memory_free_total"], flush=True)
    both = [int(x) for x in args.both.split(",") if x]
    only = [int(x) for x in args.layered.split(",") if x]
    eng = pkg.Engine(0)
    tmp = tempfile.mkdtemp(prefix="order_search_layered_")
    for k in both + only:
        forms = [DENSE, LAYERED] if k in both else [LAYERED]
        codes, card, edges, _ = pkg.datagen.discrete_bn(p=k, n=args.n, seed=40 + k, window=4, max_indegree=3)
        hop = [pkg.two_hop_neighbors(edges, k, v) & ~(1 << v) for v in range(k)]
        for skel_name in args.skeletons.split(","):
            skeleton = skel_name == "2-hop"
            nb = hop if skeleton else None
            scorer = pkg.Engine(0)
            scorer.set_discrete(codes, card)
            caches = {}
            for v in range(k):
                res = scorer.score_variable(v, pkg.two_hop_neighbors(nb, k, v), 3, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
                caches[v] = res.fetch()
                res.free()
            scorer.close()
            path = os.path.join(tmp, f"k{k}_{int(skeleton)}.pss")
            pkg.pss.write_pss(path, "bn.csv", args.n, 3, "BIC", [f"X{v}" for v in range(k)], card, caches)
            skel_file = None
            if skeleton:
                skel_file = os.path.join(tmp, f"k{k}.skel.csv")
                pkg.datagen.write_skeleton_matrix(skel_file, hop, k)
            cache = search.ScoreCache(path)
            entries = [cache.entries(v) for v in range(k)]
            comp = (1 << k) - 1
            assert pkg.components(k, nb) == [comp], f"k={k}: the skeleton is not connected"
            cand_bits = [bin(int(np.bitwise_or.reduce(m)) if len(m) else 0).count("1") for m, _ in entries]
            n_ent = int(sum(len(m) for m, _ in entries))
            run = {"k": k, "skeleton": skel_name, "entries": n_ent, "max_candidates": max(cand_bits),
                   "table_bytes": int(sum(4 << c for c in cand_bits)), "forms": {}}
            out, times = {}, {f: [] for f in forms}
            try:
                for f in forms:                                        # warm-up
                    out[f] = eng._order_search(f, entries, k, comp, nb)
                for _ in range(3):                                     # alternating
                    for f in forms:
                        t0 = time.perf_counter()
                        eng._order_search(f, entries, k, comp, nb)
                        times[f].append(time.perf_counter() - t0)
                for f in forms:
                    run["forms"][f] = {"device_bytes": device_bytes(f, k, cand_bits, n_ent), "call_s_mean3": float(np.mean(times[f])),
                                       "call_s": times[f], **timed(eng, f, entries, k, comp, nb)}
            except pkg.UrlGpuError as e:
                run["refused"] = str(e)
                run["device_bytes"] = device_bytes(LAYERED, k, cand_bits, n_ent)
                run["memory_free_total"] = free_memory()
            if out:
                c, o, par = out[forms[-1]]
                run["cost"] = float(c)
                if len(forms) == 2:
                    cd, od, pd = out[DENSE]
                    run["bit_equal"] = bool(c.view(np.uint32) == cd.view(np.uint32) and o == od and np.array_equal(par, pd))
                run["astar"] = run_astar(path, skel_file, args.astar_budget, int(args.astar_mem_gb * (1 << 30)))
                if "cost" in run["astar"]:
                    run["astar"]["cost_minus_order_search"] = run["astar"]["cost"] - float(c)
            print(json.dumps(run), flush=True)
            result["runs"].append(run)
    eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    for name in os.listdir(tmp):
        os.remove(os.path.join(tmp, name))
    os.rmdir(tmp)


if __name__ == "__main__":
    main()
