"""Order-graph search on the device (urlgpu_order_search) against the host A* (urlsearch_astar) on components of k = 20, 24,
28 and 30 variables -> profiles/r04_order_search.json.

Inputs: datagen.discrete_bn data (window 4, at most 3 parents), scored by the engine with BIC at -p 3 and PRUNE_DOMINATED,
written as a .pss and read back by search.ScoreCache (scores negated into the search side's sign).  Each size runs once with
no skeleton (every variable a candidate of every other) and once with the data's 2-hop skeleton (skeleton row v = the 2-hop
neighbourhood of v in the generating graph, which is also the candidate set the scores were computed over).

Per run: the call's time (host clock around the synchronous Engine.order_search, warmed, mean of 3); the split between the
best-parent tables and the layer sweeps (CUDA events, urlgpu_stats ms_order_tables / ms_order_layers, a separate timed
call); the algorithmic bytes of the sweep, sum over nodes S of |S| gathers of a 4-byte cost and a 4-byte table entry =
8 k 2^(k-1) bytes, over the layer time, next to the HBM bandwidth a device-to-device copy reaches in the same process; and
the host A* (list) in a child process under an address-space limit and a wall-clock budget, killed and reaped when it
overruns.  The card's name and power limit are read in the same command."""
from __future__ import annotations

import argparse
import importlib
import json
import multiprocessing as mp
import os
import resource
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("urlearning-cpp_b200")
search = importlib.import_module("urlearning-cpp_b200.search")


def card_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def hbm_copy_gbs():
    """device-to-device copy of 8 GiB, best of 5, read + write bytes over time (the L2 cannot hold it)"""
    import torch
    a = torch.empty(1 << 31, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * a.numel() * 4 / (e0.elapsed_time(e1) / 1e3) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


def astar_child(path, skel, conn, limit_bytes):
    resource.setrlimit(resource.RLIMIT_AS, (limit_bytes, limit_bytes))
    try:
        c = search.ScoreCache(path)
        t0 = time.perf_counter()
        cost, _, nodes, _ = c.astar("list", 2, skel)
        conn.send({"seconds": time.perf_counter() - t0, "cost": cost, "nodes_expanded": nodes})
    except BaseException as e:  # noqa: BLE001 (MemoryError, bad_alloc as RuntimeError)
        conn.send({"error": f"{type(e).__name__}: {e}"})


def run_astar(path, skel, budget_s, limit_bytes):
    ctx = mp.get_context("spawn")   # a fresh interpreter: no CUDA address-space reservations under the limit
    rd, wr = ctx.Pipe(duplex=False)
    proc = ctx.Process(target=astar_child, args=(path, skel, wr, limit_bytes))
    proc.start()
    wr.close()
    got = rd.poll(budget_s)
    res = rd.recv() if got else None
    if proc.is_alive():
        proc.kill()
    proc.join()
    if res is None:
        return {"did_not_finish_within_s": budget_s, "address_space_limit_bytes": limit_bytes}
    res["address_space_limit_bytes"] = limit_bytes
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20,24,28,30")
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--astar-budget", type=float, default=30.0)
    ap.add_argument("--astar-mem-gb", type=float, default=64.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_order_search.json"))
    args = ap.parse_args()
    result = {"card": card_info(), "hbm_copy_GBps": hbm_copy_gbs(), "astar_budget_s": args.astar_budget, "runs": []}
    print(result["card"], "HBM copy", result["hbm_copy_GBps"], "GB/s", flush=True)
    eng = pkg.Engine(0)
    tmp = tempfile.mkdtemp(prefix="order_search_")
    for k in [int(x) for x in args.sizes.split(",")]:
        codes, card, edges, _ = pkg.datagen.discrete_bn(p=k, n=args.n, seed=40 + k, window=4, max_indegree=3)
        hop = [pkg.two_hop_neighbors(edges, k, v) & ~(1 << v) for v in range(k)]
        for skeleton in (False, True):
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
            comps = pkg.components(k, nb)
            assert comps == [(1 << k) - 1], f"k={k}: the skeleton is not connected"
            comp = comps[0]
            cand_bits = [bin(int(np.bitwise_or.reduce(m)) if len(m) else 0).count("1") for m, _ in entries]
            eng.order_search(entries, k, comp, nb)                     # warm-up
            times = []
            for _ in range(3):
                t0 = time.perf_counter()
                cost, order, parents = eng.order_search(entries, k, comp, nb)
                times.append(time.perf_counter() - t0)
            eng.reset_stats()
            eng.enable_timing(True)
            eng.order_search(entries, k, comp, nb)
            st = eng.stats()
            eng.enable_timing(False)
            alg = 8.0 * k * 2 ** (k - 1)
            run = {"k": k, "skeleton": "2-hop" if skeleton else "none", "entries": int(sum(len(m) for m, _ in entries)),
                   "max_candidates": max(cand_bits), "table_bytes": int(sum(4 << c for c in cand_bits)), "node_bytes": 5 * 2 ** k,
                   "cost": float(cost), "call_s_mean3": float(np.mean(times)), "call_s": times,
                   "ms_tables": st["ms_order_tables"], "ms_layers": st["ms_order_layers"],
                   "algorithmic_bytes": alg, "algorithmic_GBps": alg / (st["ms_order_layers"] / 1e3) / 1e9 if st["ms_order_layers"] > 0 else None}
            run["astar"] = run_astar(path, skel_file, args.astar_budget, int(args.astar_mem_gb * (1 << 30)))
            if "cost" in run["astar"]:
                run["astar"]["cost_minus_order_search"] = run["astar"]["cost"] - float(cost)
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
