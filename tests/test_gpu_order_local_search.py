"""urlgpu_order_local_search / Engine.order_local_search / Engine.local_search_dag: insertion hill climbing over the admissible
orders of a skeleton component, with the objective of the exact order-graph search.  Checked bit for bit against a direct
restatement of the contract (include/urlgpu.h), never below the exact search's cost, at the exact optimum on the pinned caches,
locally optimal on a 60-variable component the exact search cannot take, and for every refusal."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

from test_gpu_order_search import bn_cache, family_score, markov_class, random_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "tests", "data")
EXE = os.path.join(ROOT, "urlearning-cpp_b200", "score")
FLT_MAX = np.float32(np.finfo(np.float32).max)
ERR_ARG, ERR_LIMIT = -1, -3
M64 = (1 << 64) - 1
VALUES = np.array([0.1, 0.7, 1.3, 2.0, 2.5, 3.0], dtype=np.float32)


@pytest.fixture(scope="module")
def S():
    return importlib.import_module("urlearning-cpp_b200.search")


# ------------------------------------------------------------------------------------------------ restatement
class Restated:
    """the contract of urlgpu_order_local_search, transliterated: best(v, U) by a scan of v's sorted list, the cost of an order
    by its full float32 path sum, every neighbour of every iteration evaluated from scratch"""

    def __init__(self, entries, p, comp, edges=None):
        self.vs = [v for v in range(p) if (comp >> v) & 1]
        self.comp = comp
        self.lists = {}
        for v in self.vs:
            m, s = entries[v]
            q = [(np.float32(s[i]), bin(int(m[i])).count("1"), int(m[i]), i) for i in range(len(m)) if int(m[i]) & ~comp == 0]
            q.sort()
            self.lists[v] = [(e[0], e[2]) for e in q]
        self.adj = {v: (int(edges[v]) if edges is not None else comp) for v in self.vs}
        self.memo = {}

    def best(self, v, U):
        key = (v, U)
        if key not in self.memo:
            self.memo[key] = next(((s, m) for s, m in self.lists[v] if m & ~U == 0), (FLT_MAX, 0))
        return self.memo[key]

    def admissible(self, order):
        U = 0
        for m, v in enumerate(order):
            if m and not (self.adj[v] & U & ~(1 << v)):
                return False
            U |= 1 << v
        return True

    def cost(self, order):
        g, U = np.float32(0), 0
        with np.errstate(over="ignore"):
            for v in order:
                g = np.float32(g + self.best(v, U)[0])
                U |= 1 << v
        return g

    def start(self, seed, r):
        x = (seed + 0xD1B54A32D192ED03 * (r + 1)) & M64

        def draw():
            nonlocal x
            x = (x + 0x9E3779B97F4A7C15) & M64
            z = x
            z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
            z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
            return z ^ (z >> 31)
        order = [self.vs[draw() % len(self.vs)]]
        placed = 1 << order[0]
        while len(order) < len(self.vs):
            F = [v for v in self.vs if not (placed >> v) & 1 and any((self.adj[u] >> v) & 1 for u in order)]
            if not F:
                return None
            order.append(F[draw() % len(F)])
            placed |= 1 << order[-1]
        return order

    def climb(self, seed, r):
        order = self.start(seed, r)
        if order is None:
            return np.float32(np.inf), 0, None
        moves, k = 0, len(order)
        while True:
            cur = self.cost(order)
            best = None
            for i in range(k):
                for j in range(k):
                    if i == j:
                        continue
                    new = order[:i] + order[i + 1:]
                    new.insert(j, order[i])
                    if not self.admissible(new):
                        continue
                    c = self.cost(new)
                    if best is None or c < best[0]:
                        best = (c, new)
            if best is None or not best[0] < cur:
                return cur, moves, order
            order = best[1]
            moves += 1

    def run(self, restarts, seed):
        """-> (cost, order, parents {v: mask}, restart costs, restart moves) or None ("No solution found.")"""
        res = [self.climb(seed, r) for r in range(restarts)]
        b = 0
        for r in range(1, restarts):
            if res[r][0] < res[b][0]:
                b = r
        cost, _, order = res[b]
        if order is None or not cost < np.inf:
            return None
        parents, U = {}, 0
        for v in order:
            parents[v] = self.best(v, U)[1]
            U |= 1 << v
        return cost, order, parents, np.array([x[0] for x in res], dtype=np.float32), np.array([x[1] for x in res], dtype=np.uint32)


def wide_case(rng, skeleton):
    """random_case at k = 24, its variables moved to 13 of 60..75 and all of 130..140 in p = 200 (masks over four words)"""
    entries24, _, comp24, edges24 = random_case(rng, 24, 0, VALUES, skeleton)
    where = sorted(rng.choice(np.arange(60, 76), size=13, replace=False).tolist()) + list(range(130, 141))

    def move(m):
        return sum(1 << where[u] for u in range(24) if (int(m) >> u) & 1)
    p = 200
    entries = [([], []) for _ in range(p)]
    for u in range(24):
        m, s = entries24[u]
        entries[where[u]] = ([move(x) for x in m], s)
    entries = [(m if len(m) else np.zeros(0, dtype=np.uint64), np.asarray(s, dtype=np.float32)) for m, s in entries]
    edges = None
    if edges24 is not None:
        edges = [0] * p
        for u in range(24):
            edges[where[u]] = move(edges24[u])
    return entries, p, move(comp24), edges


def cases():
    out = []
    for k in (1, 2, 5, 9, 12):
        for skeleton in (False, True):
            rng = np.random.default_rng(7000 + 10 * k + skeleton)
            out += [(f"k{k}_{'skel' if skeleton else 'none'}_{t}", random_case(rng, k, 2, VALUES, skeleton)) for t in range(3)]
    for skeleton in (False, True):
        out.append((f"wide24_{'skel' if skeleton else 'none'}", wide_case(np.random.default_rng(7500 + skeleton), skeleton)))
    return out


CASES = cases()


def as_int(parents, v):
    row = parents[v]
    return int(row) if np.ndim(row) == 0 else sum(int(x) << (64 * w) for w, x in enumerate(row))


def check_local(lookup, entries, p, comp, edges, cost, order, parents):
    """the DAG is valid: the order is an admissible order of C, every parent placed earlier, every parent set best(v, pred) and
    a cache entry with that score, the float32 path sum equal to cost bit for bit"""
    vs = [v for v in range(p) if (comp >> v) & 1]
    assert sorted(order) == vs
    U, g = 0, np.float32(0)
    for m, v in enumerate(order):
        if edges is not None and m:
            assert int(edges[v]) & U & ~(1 << v), f"variable {v} at position {m} touches none of its predecessors"
        par = as_int(parents, v)
        assert par & ~U == 0, "the DAG has a cycle or disagrees with the order"
        s, want = lookup(v, U)
        assert par == want
        if s != FLT_MAX:
            assert family_score(entries, v, par) == s
        with np.errstate(over="ignore"):
            g = np.float32(g + s)
        U |= 1 << v
    assert g.view(np.uint32) == np.float32(cost).view(np.uint32)
    for v in range(p):
        if not (comp >> v) & 1:
            assert as_int(parents, v) == 0


# ------------------------------------------------------------------------------------------------ 1. the restatement
@pytest.mark.parametrize("name,case", CASES, ids=[c[0] for c in CASES])
def test_bit_equal_to_restatement(engine, name, case):
    entries, p, comp, edges = case
    want = Restated(entries, p, comp, edges).run(8, 12345)
    if want is None:
        with pytest.raises(Exception, match="No solution found."):
            engine.order_local_search(entries, p, comp, edges, restarts=8, seed=12345)
        return
    cost, order, parents, rc, rm = engine.order_local_search(entries, p, comp, edges, restarts=8, seed=12345)
    assert np.float32(cost).view(np.uint32) == want[0].view(np.uint32)
    assert order == want[1]
    for v in range(p):
        assert as_int(parents, v) == (want[2][v] if (comp >> v) & 1 else 0)
    assert np.array_equal(rc.view(np.uint32), want[3].view(np.uint32))
    assert np.array_equal(rm, want[4])


# ------------------------------------------------------------------------------------------------ 2. never below the exact optimum
@pytest.mark.parametrize("name,case", CASES, ids=[c[0] for c in CASES])
def test_random_cases_never_below_exact(engine, name, case):
    entries, p, comp, edges = case
    try:
        exact = engine.order_search(entries, p, comp, edges)[0]
    except Exception as e:
        assert "No solution found." in str(e)
        return
    cost, order, parents, _, _ = engine.order_local_search(entries, p, comp, edges, restarts=64, seed=3)
    assert np.float32(cost) >= np.float32(exact)
    R = Restated(entries, p, comp, edges)
    check_local(R.best, entries, p, comp, edges, cost, order, parents)


def cache_lookup(cache):
    def lookup(v, U):
        s, par = cache.best_scores(v, np.array([U], dtype=np.uint64), "list")
        return s[0], int(par[0])
    return lookup


def compare_on_cache(pkg, engine, cache, edges, restarts=256, seed=0):
    """per component: local >= exact and a valid DAG; the totals summed as local_search_dag does -> (local total, exact total)"""
    p = cache.p
    entries = [cache.entries(v) for v in range(p)]
    total, parents = engine.local_search_dag(cache, edges, restarts, seed)
    exact_total, _ = engine.optimal_dag(cache, edges)
    acc = np.float32(0)
    for comp in pkg.components(p, edges):
        cost, order, par, _, _ = engine.order_local_search(entries, p, comp, edges, restarts, seed)
        exact = engine.order_search(entries, p, comp, edges)[0]
        assert np.float32(cost) >= np.float32(exact)
        check_local(cache_lookup(cache), entries, p, comp, edges, cost, order, par)
        for v in range(p):
            if (comp >> v) & 1:
                assert int(parents[v]) == int(par[v])
        acc = np.float32(acc + cost)
    assert np.float32(total).view(np.uint32) == acc.view(np.uint32)
    return np.float32(total), np.float32(exact_total), parents


def hepatitis(S, tmp_path, prune):
    path = str(tmp_path / f"hep{int(prune)}.pss")
    subprocess.check_call([EXE, os.path.join(DATA, "hepatitis.clean.csv"), path, "-s", "-f", "BIC", "--quiet"] + (["--prune"] if prune else []),
                          stdout=subprocess.DEVNULL)
    return S.ScoreCache(path)


def figure(S, tmp_path, fig, fn):
    skel = os.path.join(DATA, "skeleton4_ones.csv")
    path = str(tmp_path / f"{fig}.pss")
    subprocess.check_call([EXE, os.path.join(DATA, fig, fn), path, "-k", skel, "-f", "cBIC", "--lambda=2", "--quiet"], stdout=subprocess.DEVNULL)
    m = np.loadtxt(skel, delimiter=",").astype(int)
    return S.ScoreCache(path), [sum(1 << j for j in range(4) if m[i, j]) for i in range(4)]


def p24_two_hop(pkg, engine, S, tmp_path):
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=24, n=4000, seed=5, window=3, max_indegree=2)
    path, (rows, _) = bn_cache(pkg, engine, tmp_path, codes, card, edges, True)
    return S.ScoreCache(path), rows


@pytest.mark.parametrize("prune", [False, True])
def test_hepatitis_reaches_exact_dag(pkg, engine, S, tmp_path, prune):
    """256 restarts find the exact search's DAG, but the best of them places it in another order, whose float32 path sum is one
    ulp above the exact search's (962.4949 against 962.4948; the float64 sums of the two are equal).  4096 restarts from the
    same seed, a superset of those 256, reach the exact cost bit for bit."""
    cache = hepatitis(S, tmp_path, prune)
    local, exact, parents = compare_on_cache(pkg, engine, cache, None)
    assert np.array_equal(parents, engine.optimal_dag(cache)[1])
    assert local.view(np.int32) - exact.view(np.int32) <= 1, f"gap {float(local) - float(exact)!r}"
    entries = [cache.entries(v) for v in range(cache.p)]
    wide = engine.order_local_search(entries, cache.p, (1 << cache.p) - 1, None, restarts=4096, seed=0)[0]
    assert np.float32(wide).view(np.uint32) == exact.view(np.uint32)


def test_p24_two_hop_reaches_exact(pkg, engine, S, tmp_path):
    cache, rows = p24_two_hop(pkg, engine, S, tmp_path)
    local, exact, _ = compare_on_cache(pkg, engine, cache, rows)
    assert local.view(np.uint32) == exact.view(np.uint32), f"gap {float(local) - float(exact)!r}"


def test_two_networks_side_by_side_never_below_exact(pkg, engine, S, tmp_path):
    c1, k1, e1, _ = pkg.datagen.discrete_bn(p=10, n=3000, seed=6, window=3, max_indegree=2)
    c2, k2, e2, _ = pkg.datagen.discrete_bn(p=9, n=3000, seed=7, window=3, max_indegree=2)
    edges = list(e1) + [int(e) << 10 for e in e2]
    path, _ = bn_cache(pkg, engine, tmp_path, np.concatenate([c1, c2]), np.concatenate([k1, k2]), edges, False)
    cache = S.ScoreCache(path)
    assert len(pkg.components(cache.p, edges)) >= 2
    compare_on_cache(pkg, engine, cache, edges)


@pytest.mark.parametrize("fig,fn,dag", [("Figure_1", "raw_data_8000.csv", "astar_dag_8000.csv"), ("Figure_2", "raw_data_5000.csv", "astar_dag_5000.csv")])
def test_figures_reach_exact_and_published_class(pkg, engine, S, tmp_path, fig, fn, dag):
    cache, rows = figure(S, tmp_path, fig, fn)
    local, exact, parents = compare_on_cache(pkg, engine, cache, rows)
    assert local.view(np.uint32) == exact.view(np.uint32)
    want = np.loadtxt(os.path.join(DATA, fig, dag), delimiter=",").astype(int)
    published = [sum(1 << i for i in range(4) if want[v, i]) for v in range(4)]
    assert markov_class(parents, 4) == markov_class(published, 4)


# ------------------------------------------------------------------------------------------------ 4. beyond the exact search
@pytest.fixture(scope="module")
def cfg3_shaped(pkg, tmp_path_factory):
    """discrete_bn(p=60, seed=4) at n = 20000, BIC over the 2-hop candidates at the bench's cap of 11, pruned, read back from a
    .pss; the generating skeleton makes it one component of 60 variables"""
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=60, n=20000, seed=4)
    eng = pkg.Engine(0)
    eng.set_discrete(codes, card)
    caches = {}
    for v in range(60):
        res = eng.score_variable(v, pkg.two_hop_neighbors(edges, 60, v), 11, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        caches[v] = res.fetch()
        res.free()
    eng.close()
    path = str(tmp_path_factory.mktemp("cfg3") / "cfg3.pss")
    pkg.pss.write_pss(path, "cfg3.csv", 20000, 11, "BIC", [f"X{v}" for v in range(60)], card, caches)
    S = importlib.import_module("urlearning-cpp_b200.search")
    cache = S.ScoreCache(path)
    assert pkg.components(60, edges) == [(1 << 60) - 1]
    return cache, [int(e) for e in edges]


def insertion_neighbours_lower(cache, order, edges, cost):
    """every admissible insertion move's path sum from batched best_scores look-ups -> the moves strictly below cost"""
    k = len(order)
    moves = []
    for i in range(k):
        for j in range(k):
            if i != j:
                new = order[:i] + order[i + 1:]
                new.insert(j, order[i])
                moves.append(new)
    queries = {}
    for new in moves:
        U = 0
        for v in new:
            queries.setdefault(v, set()).add(U)
            U |= 1 << v
    score = {}
    for v, qs in queries.items():
        qs = sorted(qs)
        s, _ = cache.best_scores(v, np.array(qs, dtype=np.uint64), "list")
        score.update({(v, U): x for U, x in zip(qs, s)})
    lower = []
    for new in moves:
        U, g, ok = 0, np.float32(0), True
        for m, v in enumerate(new):
            if m and not (edges[v] & U):
                ok = False
                break
            g = np.float32(g + score[(v, U)])
            U |= 1 << v
        if ok and g < np.float32(cost):
            lower.append((new, g))
    return lower


def test_cfg3_shaped_component_of_60(pkg, engine, cfg3_shaped):
    cache, edges = cfg3_shaped
    p, comp = 60, (1 << 60) - 1
    entries = [cache.entries(v) for v in range(p)]
    with pytest.raises(Exception, match="at most 36"):
        engine.order_search(entries, p, comp, edges)
    a = engine.order_local_search(entries, p, comp, edges, restarts=256, seed=0)
    cost, order, parents, rc, rm = a
    check_local(cache_lookup(cache), entries, p, comp, edges, cost, order, parents)
    assert insertion_neighbours_lower(cache, order, edges, cost) == []
    b = engine.order_local_search(entries, p, comp, edges, restarts=256, seed=0)
    assert np.float32(cost).view(np.uint32) == np.float32(b[0]).view(np.uint32) and order == b[1]
    assert np.array_equal(parents, b[2]) and np.array_equal(rc.view(np.uint32), b[3].view(np.uint32)) and np.array_equal(rm, b[4])
    c = engine.order_local_search(entries, p, comp, edges, restarts=64, seed=0)
    assert np.array_equal(c[3].view(np.uint32), rc[:64].view(np.uint32)) and np.array_equal(c[4], rm[:64])
    assert np.float32(cost) == rc.min()
    total, dag = engine.local_search_dag(cache, edges, restarts=256, seed=0)
    assert np.float32(total).view(np.uint32) == np.float32(cost).view(np.uint32) and np.array_equal(dag, parents)
    print(f"cost {cost!r}, restart costs {rc.min()!r}..{rc.max()!r}, moves mean {rm.mean():.1f} max {rm.max()}")


# ------------------------------------------------------------------------------------------------ 5. refusals
def raw(engine, p, words, offsets, masks, scores, comp, edges=None, restarts=8, symbol="urlgpu_order_local_search"):
    lib = engine.lib
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    m = np.ascontiguousarray(masks, dtype=np.uint64).reshape(-1)
    s = np.ascontiguousarray(scores, dtype=np.float32)
    cw = np.ascontiguousarray(comp, dtype=np.uint64)
    ed = None if edges is None else np.ascontiguousarray(edges, dtype=np.uint64)
    cost = C.c_float()
    order = np.zeros(256, dtype=np.int32)
    parents = np.zeros(max(1, p) * max(1, words) + 8, dtype=np.uint64)
    args = [engine._h, p, words, off.ctypes.data, m.ctypes.data if len(m) else None, s.ctypes.data if len(s) else None,
            None if ed is None else ed.ctypes.data, cw.ctypes.data]
    if symbol == "urlgpu_order_local_search":
        args += [restarts, 0, C.byref(cost), order.ctypes.data, parents.ctypes.data, None, None]
    else:
        args += [C.byref(cost), order.ctypes.data, parents.ctypes.data]
    rc = getattr(lib, symbol)(*args)
    return rc, lib.urlgpu_last_error(engine._h).decode()


def test_every_refusal(engine):
    def works():
        assert raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b11])[0] == 0

    works()
    same_as_exact = [
        (0, 1, [0], [], [], [0]),
        (2, 0, [0, 1, 2], [0, 1], [1, 2], [0b11]),
        (2, 5, [0, 1, 2], np.zeros(10), [1, 2], np.full(5, 3)),
        (70, 1, np.arange(71), np.zeros(70), np.ones(70), [1]),
        (2, 1, [0, 2, 1], [0, 1], [1, 2], [0b11]),
        (2, 1, [0, 1, 2], [0, 1], [1, 2], [0]),
        (2, 1, [0, 1, 2], [0, 1], [1, 2], [0b111]),
        (2, 1, [0, 1, 3], [0, 0, 1], [1, 2, np.nan], [0b11]),
        (2, 1, [0, 1, 3], [0, 0, 2], [1, 2, 3], [0b11]),
    ]
    for args in same_as_exact:
        rc, msg = raw(engine, *args)
        erc, emsg = raw(engine, *args, symbol="urlgpu_order_search")
        assert rc == erc == ERR_ARG
        assert msg.startswith("order_local_search: ") and emsg.startswith("order_search: ")
        assert msg[len("order_local_search: "):] == emsg[len("order_search: "):]
        works()
    for restarts in (0, (1 << 20) + 1):
        rc, msg = raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b11], restarts=restarts)
        assert rc == ERR_ARG and "restarts" in msg
        works()
    assert raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b11], restarts=1 << 20)[0] == 0
    # c_v = 33: variable 0 with every other variable of a 34-variable component
    p = 34
    masks = [((1 << p) - 1) & ~1] + [0] * (p - 1)
    rc, msg = raw(engine, p, 1, np.arange(p + 1), masks, np.ones(p), [(1 << p) - 1])
    assert rc == ERR_LIMIT and msg == "order_local_search: variable 0 has 33 candidate parents inside the component; at most 32 are supported"
    works()
    masks[0] &= ~2                                               # c_v = 32 is accepted
    assert raw(engine, p, 1, np.arange(p + 1), masks, np.ones(p), [(1 << p) - 1])[0] == 0
    # twelve variables with c_v = 32 need 12 tables of 2^32 entries, 206 GB
    p, restarts = 33, 8
    full = (1 << p) - 1
    masks = [full & ~(1 << v) for v in range(12)] + [0] * (p - 12)
    rc, msg = raw(engine, p, 1, np.arange(p + 1), masks, np.ones(p), [full], restarts=restarts)
    tables, ents, state = 4 * (12 * (1 << 32) + (p - 12)), 16 * p, restarts * (8 + 5 * p)
    need = tables + ents + state + 80 * p
    assert rc == ERR_LIMIT
    assert msg.startswith(f"order_local_search: the search needs {need} bytes of device memory ({tables} for the best-parent tables, "
                          f"{ents} for the entries, {state} for the state of {restarts} restarts), ")
    works()
    # no admissible order (the skeleton splits the component), and a best cost of +inf
    rc, msg = raw(engine, 2, 1, [0, 1, 2], [0, 0], [1, 2], [0b11], edges=[0, 0])
    assert rc == ERR_ARG and msg == "No solution found."
    works()
    rc, msg = raw(engine, 3, 1, [0, 0, 0, 1], [0], [1], [0b111])     # FLT_MAX + FLT_MAX in every order
    assert rc == ERR_ARG and msg == "No solution found."
    works()
