"""quick timing of the BIC path on config-4-like data (development aid, not the bench)."""
import importlib, sys, time, os
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
pkg = importlib.import_module("urlearning-cpp_b200")
n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
p = int(sys.argv[2]) if len(sys.argv) > 2 else 60
vars_ = [int(v) for v in sys.argv[3].split(",")] if len(sys.argv) > 3 else [0, 5, 30]
t0 = time.time()
codes, card, edges, _ = pkg.datagen.discrete_bn(p=p, n=n, seed=4)
print(f"datagen {time.time()-t0:.1f}s card={card.tolist()}")
eng = pkg.Engine(0)
eng.set_discrete(codes, card)
K = pkg.effective_max_parents(12, p, n, True)
eng.enable_timing(True)
for rep in range(2):
    for v in vars_:
        nb = pkg.two_hop_neighbors(edges, p, v)
        c = bin(nb & ~(1 << v)).count("1")
        eng.reset_stats()
        t0 = time.time()
        res = eng.score_variable(v, nb, K, pkg.BIC)
        eng.synchronize()
        dt = time.time() - t0
        st = eng.stats()
        print(f"v={v} c={c} K={K} sets={res.scored()} wall={dt*1e3:.1f} ms  count_ms={st['ms_count']:.2f} cube_ms={st['ms_cube']:.2f} "
              f"launches={st['launches_total']} sets/s={res.scored()/dt:.3e} alg_GB/s={st['algorithmic_bytes']/dt/1e9:.1f}")
        res.free()
