#!/usr/bin/env python
"""Throughput of urlgpu_score_sets (a list of arbitrary parent sets in one call) against a loop of urlgpu_score_one, one GPU:
  discrete — configs[3]-shaped data (datagen.discrete_bn(p=60, n=1e6, seed=4)), 100 000 random sets of 0 to 8 parents drawn
             from each child's 2-hop neighbourhood of the generating skeleton, under BIC, fNML and BDeu (ess = 1)
  cBIC     — datagen.linear_gaussian_sem(p=200, n=2e5), 100 000 random sets of 0 to 16 parents, lambda = 2
Both calls are synchronous (outputs in host memory on return), so a host clock around warmed calls times them whole.  The
score_one loop runs over the first 1 000 sets of the same list, which it must reproduce bit for bit.  Prints the card's name
and power limit, then one JSON line per workload; --out also writes all of it as one JSON file.
Usage: python tools/measure_score_sets.py [--sets 100000] [--one 1000] [--steps 3] [--out FILE]"""
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


def random_sets(rng, p, n_sets, kmax, pools):
    """n_sets (child, parent mask words) pairs: the child uniform, 0..kmax parents drawn from pools[child]"""
    words = (p + 63) // 64
    variables = rng.integers(0, p, size=n_sets).astype(np.int32)
    masks = np.zeros((n_sets, words), dtype=np.uint64)
    for i, v in enumerate(variables):
        pool = pools[v]
        k = int(rng.integers(0, min(kmax, len(pool)) + 1))
        for q in rng.choice(pool, size=k, replace=False):
            masks[i, q >> 6] |= np.uint64(1 << int(q & 63))
    return variables, masks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", type=int, default=100_000)
    ap.add_argument("--one", type=int, default=1000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    pkg = importlib.import_module("urlearning-cpp_b200")
    card_info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True, check=True).stdout
    print(card_info.strip())
    eng = pkg.Engine(0)
    rng = np.random.default_rng(2026)
    results = []

    def run(name, variables, masks, st, lam, note):
        eng.score_sets(variables, masks, st, lam)                                     # warm-up
        eng.reset_stats()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            s, x = eng.score_sets(variables, masks, st, lam)
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        launches = eng.stats()["launches_total"] // args.steps
        m = args.one
        for i in range(min(m, 50)):                                                   # warm-up
            eng.score_one(int(variables[i]), pkg.words_to_mask(masks[i]), st, lam)
        t0 = time.perf_counter()
        one = [eng.score_one(int(variables[i]), pkg.words_to_mask(masks[i]), st, lam)[0] for i in range(m)]
        one_ms = (time.perf_counter() - t0) * 1e3
        same = bool(np.array_equal(np.array(one, dtype=np.float32).view(np.uint32), s[:m].view(np.uint32)))
        r = {"score": name, "workload": note, "n_sets": len(variables), "score_sets_ms": round(ms, 3),
             "score_sets_sets_per_s": round(len(variables) / ms * 1e3), "score_sets_launches": int(launches),
             "score_one_sets": m, "score_one_ms": round(one_ms, 3), "score_one_sets_per_s": round(m / one_ms * 1e3),
             "speedup": round((len(variables) / ms) / (m / one_ms), 1), "score_one_bit_equal": same}
        print(json.dumps(r), flush=True)
        results.append(r)

    codes, card, edges, _ = pkg.datagen.discrete_bn(p=60, n=1_000_000, seed=4)
    p = codes.shape[0]
    pools = [[q for q in range(p) if q != v and (pkg.two_hop_neighbors(edges, p, v) >> q) & 1] for v in range(p)]
    variables, masks = random_sets(rng, p, args.sets, 8, pools)
    eng.set_discrete(codes, card)
    note = "discrete_bn(p=60, n=1e6, seed=4); sets of 0-8 parents from 2-hop neighbourhoods"
    run("BIC", variables, masks, pkg.BIC, 0.0, note)
    run("fNML", variables, masks, pkg.FNML, 0.0, note)
    run("BDeu", variables, masks, pkg.BDEU, 1.0, note + "; ess = 1")

    x, _ = pkg.datagen.linear_gaussian_sem(p=200, n=200_000)
    p = x.shape[0]
    pools = [[q for q in range(p) if q != v] for v in range(p)]
    variables, masks = random_sets(rng, p, args.sets, 16, pools)
    eng.set_continuous(x)
    run("cBIC", variables, masks, pkg.CBIC, 2.0, "linear_gaussian_sem(p=200, n=2e5); sets of 0-16 parents; lambda = 2")
    eng.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"nvidia_smi": card_info.strip().splitlines(), "steps": args.steps, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
