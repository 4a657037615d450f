"""randomised parity sweep of the BIC / fNML path against the oracle (development aid): random shapes, arities (incl. arity-1
columns), skeletons, parent limits, all K1 modes and root-kernel budgets, warps, segment caps and the slice switch; prints the first mismatch and exits non-zero"""
import importlib, os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
pkg = importlib.import_module("urlearning-cpp_b200")
import oracle_lib as orc
seed = int(sys.argv[1]) if len(sys.argv) > 1 else 0
budget_s = float(sys.argv[2]) if len(sys.argv) > 2 else 60.0
rng = np.random.default_rng(seed)
t_end = time.time() + budget_s
cases = 0
while time.time() < t_end:
    mode = str(rng.choice(["cube", "cube", "direct"]))
    env = {"URLGPU_BIC_MODE": mode, "URLGPU_FUSE_ROOTS": str(rng.integers(0, 2)),
           "URLGPU_ROOT_BUDGET": str(int(rng.choice([1024, 4096, 24576, 40000]))),
           "URLGPU_ROOT_WARPS": str(int(rng.choice([8, 12, 16]))),
           "URLGPU_ROOT_SEGS": str(int(rng.choice([32, 256, 1024, 8192]))),
           "URLGPU_SLICE_COUNT": str(int(rng.random() < 0.85))}
    os.environ.update(env)
    eng = pkg.Engine(0)
    p = int(rng.integers(3, 15))
    n = int(rng.choice([17, 1000, 65536, 70001, 131072, 200003]))
    ar = tuple(int(x) for x in rng.choice([2, 3, 4, 5, 7], size=int(rng.integers(1, 4))))
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=p, n=n, seed=int(rng.integers(1 << 30)), arities=ar, window=int(rng.integers(1, p + 1)),
                                                   max_indegree=int(rng.integers(1, 4)))
    if rng.random() < 0.3:  # a constant column
        j = int(rng.integers(p)); codes[j] = 0; card[j] = 1
    eng.set_discrete(codes, card)
    for _ in range(3):
        v = int(rng.integers(p))
        K = int(rng.integers(0, p))
        use_skel = rng.random() < 0.5
        nb = pkg.two_hop_neighbors(edges if use_skel else None, p, v)
        flags = pkg.PRUNE_DOMINATED if rng.random() < 0.5 else 0
        cells = int(card[v]) * int(np.prod(sorted(card[[i for i in range(p) if i != v and (nb >> i) & 1]])[::-1][:K])) if K else 1
        if cells > (1 << 24):
            continue
        fnml = rng.random() < 0.35 and int(card[v]) <= 7   # fNML on the same kernels (regret tables of wide children overflow float32)
        res = eng.score_variable(v, nb, K, pkg.FNML if fnml else pkg.BIC, flags=flags)
        masks, scores = res.fetch(); res.free()
        om = orc.enumerate_sets(v, nb, p, K)
        osc = orc.fnml_score_many(codes, card, v, om) if fnml else orc.bic_score_many(codes, card, v, om)
        stored = np.array([(s < 1) if m == 0 else (s < 0) for m, s in zip(om, osc)])
        om, osc = om[stored], osc[stored]
        if flags:
            keep = orc.prune(om, osc, K); om, osc = om[keep], osc[keep]
        order = orc.canonical_order(om)
        ok = [int(m[0]) for m in masks] == [int(om[i]) for i in order] and np.array_equal(scores.view(np.uint32), osc[order].view(np.uint32))
        cases += 1
        if not ok:
            print("MISMATCH", env, dict(p=p, n=n, ar=ar, v=v, K=K, skel=use_skel, flags=flags, fnml=fnml, card=card.tolist()))
            sys.exit(1)
    eng.close()
print(f"stress OK: {cases} (variable, family) cases, seed {seed}")
