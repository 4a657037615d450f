"""urlgpu_order_search / Engine.order_search / Engine.optimal_dag: exact structure search over the order graph of each skeleton
component on the device.  Checked bit for bit against a numpy restatement of the contract (include/urlgpu.h), against the
host A* (ScoreCache.astar, list and bitwise) on real caches, against the published Figure_1/2 DAGs up to Markov
equivalence, at the limits (2^32 nodes, one variable, no cached subset) and for every refusal."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "tests", "data")
EXE = os.path.join(ROOT, "urlearning-cpp_b200", "score")
FLT_MAX = np.float32(np.finfo(np.float32).max)
ERR_ARG, ERR_LIMIT = -1, -3


@pytest.fixture(scope="module")
def S():
    return importlib.import_module("urlearning-cpp_b200.search")


# ------------------------------------------------------------------------------------------------ numpy restatement
def restate(entries, p, comp, edges=None):
    """the contract of urlgpu_order_search in numpy -> (cost float32, order, parents {v: mask}) or None (no solution)"""
    vs = [v for v in range(p) if (comp >> v) & 1]
    k, N = len(vs), 1 << len(vs)
    idx = np.arange(N, dtype=np.int64)
    popc = np.array([bin(i).count("1") for i in range(N)])

    def compact(m):
        return sum(1 << j for j, v in enumerate(vs) if (int(m) >> v) & 1)
    tabs = []
    for v in vs:
        m, s = entries[v]
        q = [(np.float32(s[i]), bin(int(m[i])).count("1"), int(m[i]), i) for i in range(len(m)) if int(m[i]) & ~comp == 0]
        q.sort()
        t = np.full(N, 1 << 40, dtype=np.int64)
        for r, e in enumerate(q):
            c = compact(e[2])
            t[c] = min(t[c], r)
        for b in range(k):
            sel = idx[(idx >> b) & 1 == 1]
            t[sel] = np.minimum(t[sel], t[sel ^ (1 << b)])
        sc = np.array([e[0] for e in q] + [FLT_MAX], dtype=np.float32)
        tabs.append((t, sc, [e[2] for e in q]))
    adj = [compact(edges[v]) if edges is not None else (1 << k) - 1 for v in vs]
    cost = np.full(N, np.inf, dtype=np.float32)
    cost[0] = 0
    leaf = np.full(N, 255, dtype=np.int64)
    with np.errstate(over="ignore", invalid="ignore"):
        for layer in range(1, k + 1):
            Sl = idx[popc == layer]
            best = np.full(len(Sl), np.inf, dtype=np.float32)
            bl = np.full(len(Sl), 255, dtype=np.int64)
            for j in range(k):
                prev = Sl ^ (1 << j)
                ok = ((Sl >> j) & 1 == 1) & (cost[prev] != np.inf)
                ok &= (prev == 0) | ((prev & adj[j]) != 0)
                t, sc, _ = tabs[j]
                pos = np.minimum(t[prev], len(sc) - 1)
                g = (cost[prev] + sc[pos]).astype(np.float32)
                ok &= g != np.inf
                upd = ok & (g < best)
                best[upd] = g[upd]
                bl[upd] = j
            cost[Sl] = best
            leaf[Sl] = bl
    full = N - 1
    if leaf[full] == 255 or cost[full] == np.inf:
        return None
    order, parents, s_ = [], {}, full
    for _ in range(k):
        j = int(leaf[s_])
        prev = s_ ^ (1 << j)
        t, sc, ms = tabs[j]
        parents[vs[j]] = ms[t[prev]] if t[prev] < len(ms) else 0
        order.append(vs[j])
        s_ = prev
    return cost[full], order[::-1], parents


def random_case(rng, k, outside, values, skeleton):
    p = k + outside
    comp_vars = sorted(rng.choice(p, size=k, replace=False).tolist())
    comp = sum(1 << v for v in comp_vars)
    entries = []
    for v in range(p):
        ms, ss = [], []
        if rng.random() < 0.9:
            ms.append(0)
            ss.append(rng.choice(values))
        for _ in range(int(rng.integers(0, 10))):
            others = [u for u in range(p) if u != v]
            m = sum(1 << int(u) for u in rng.choice(others, size=min(int(rng.integers(1, 4)), p - 1), replace=False))
            ms.append(m)
            ss.append(rng.choice(values))
        entries.append((np.array(ms, dtype=np.uint64), np.array(ss, dtype=np.float32)))
    edges = None
    if skeleton:
        edges = [0] * p
        perm = rng.permutation(comp_vars).tolist()
        for a, b in zip(perm, perm[1:]):                      # a spanning path keeps C connected
            edges[a] |= 1 << b
            edges[b] |= 1 << a
        for a in comp_vars:
            for b in comp_vars:
                if a < b and rng.random() < 0.2:
                    edges[a] |= 1 << b
                    edges[b] |= 1 << a
            if rng.random() < 0.3:
                edges[a] |= 1 << a                            # a diagonal changes nothing
    return entries, p, comp, edges


@pytest.mark.parametrize("k", [1, 2, 5, 9, 12, 14])
@pytest.mark.parametrize("skeleton", [False, True])
def test_bit_equal_to_numpy_restatement(engine, k, skeleton):
    """scores from a handful of values so that ties occur in the best-subset choice and in the leaf choice: cost, order and
    parents bit-equal to the restatement, with and without a skeleton, with entries that reach outside the component"""
    rng = np.random.default_rng(1000 * k + skeleton)
    values = np.array([0.1, 0.7, 1.3, 2.0, 2.5, 3.0], dtype=np.float32)
    for _ in range(4):
        entries, p, comp, edges = random_case(rng, k, 2, values, skeleton)
        want = restate(entries, p, comp, edges)
        if want is None:
            with pytest.raises(Exception, match="No solution found."):
                engine.order_search(entries, p, comp, edges)
            continue
        cost, order, parents = engine.order_search(entries, p, comp, edges)
        assert np.float32(cost).view(np.uint32) == want[0].view(np.uint32)
        assert order == want[1]
        for v in range(p):
            assert int(parents[v]) == (want[2][v] if (comp >> v) & 1 else 0)


# ------------------------------------------------------------------------------------------------ against A*
def family_score(entries, v, mask):
    m, s = entries[v]
    hit = [np.float32(s[i]) for i in range(len(m)) if int(m[i]) == int(mask)]
    assert hit, f"parent set {int(mask):#x} of variable {v} is not a cache entry"
    return min(hit)


def check_dag(engine, entries, p, comps, edges, parents, cost):
    """per component, the order order_search returns: acyclic (every parent placed earlier), every parent set a cache entry,
    the float32 sum of the families in that order equal to the component's cost bit for bit; the components' costs summed
    in float32 equal to the total"""
    total = np.float32(0)
    for comp in comps:
        c, order, par = engine.order_search(entries, p, comp, edges)
        assert sorted(order) == [v for v in range(p) if (comp >> v) & 1]
        placed, acc = 0, np.float32(0)
        for v in order:
            assert int(par[v]) == int(parents[v])
            assert int(par[v]) & ~placed == 0, "the DAG has a cycle"
            placed |= 1 << v
            acc = np.float32(acc + family_score(entries, v, par[v]))
        assert acc.view(np.uint32) == np.float32(c).view(np.uint32)
        total = np.float32(total + c)
    assert total.view(np.uint32) == np.float32(cost).view(np.uint32)


def compare_with_astar(engine, cache, edges, skel_file, label):
    pkg = importlib.import_module("urlearning-cpp_b200")
    p = cache.p
    entries = [cache.entries(v) for v in range(p)]
    cost, parents = engine.optimal_dag(cache, edges)
    assert isinstance(cost, float) and parents.dtype == np.uint64 and parents.shape == (p,)
    comps = pkg.components(p, edges)
    check_dag(engine, entries, p, comps, edges, parents, cost)
    for kind in ("list", "bitwise"):
        ac, ap, _, ncomp = cache.astar(kind, 2, skel_file)
        assert ncomp == len(comps)
        if np.float32(cost) != np.float32(ac):
            print(f"{label} {kind}: order search {cost!r}, A* {ac!r}, difference {ac - cost:.3g}")
        assert np.float32(cost) <= np.float32(ac)
        assert abs(ac - cost) <= 1e-4 * abs(ac)
        if not np.array_equal(ap, parents):
            other = np.float32(0)
            for v in range(p):
                other = np.float32(other + family_score(entries, v, ap[v]))
            print(f"{label} {kind}: the DAGs differ; A*'s scores {other!r}")
            assert abs(other - cost) <= 1e-4 * abs(cost)
    return cost


def test_hepatitis_against_astar_pruned_and_unpruned(engine, S, tmp_path):
    inp = os.path.join(DATA, "hepatitis.clean.csv")
    full, pruned = str(tmp_path / "full.pss"), str(tmp_path / "pruned.pss")
    subprocess.check_call([EXE, inp, full, "-s", "-f", "BIC", "--quiet"], stdout=subprocess.DEVNULL)
    subprocess.check_call([EXE, inp, pruned, "-s", "-f", "BIC", "--prune", "--quiet"], stdout=subprocess.DEVNULL)
    a = compare_with_astar(engine, S.ScoreCache(full), None, None, "hepatitis")
    b = compare_with_astar(engine, S.ScoreCache(pruned), None, None, "hepatitis --prune")
    assert np.float32(a).view(np.uint32) == np.float32(b).view(np.uint32)


def bn_cache(pkg, engine, tmp_path, codes, card, edges, two_hop_skeleton):
    """BIC at -p 3 with PRUNE_DOMINATED over the 2-hop candidates of `edges`, written as a .pss and read back (search sign)"""
    p, n = codes.shape
    eng = pkg.Engine(0)
    eng.set_discrete(codes, card)
    caches = {}
    for v in range(p):
        nb = pkg.two_hop_neighbors(edges, p, v)
        res = eng.score_variable(v, nb, 3, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        caches[v] = res.fetch()
        res.free()
    eng.close()
    path = str(tmp_path / "bn.pss")
    pkg.pss.write_pss(path, "bn.csv", n, 3, "BIC", [f"X{v}" for v in range(p)], card, caches)
    skel = None
    if two_hop_skeleton:
        skel_rows = [pkg.two_hop_neighbors(edges, p, v) & ~(1 << v) for v in range(p)]
        skel = (skel_rows, str(tmp_path / "skel.csv"))
        pkg.datagen.write_skeleton_matrix(skel[1], skel_rows, p)
    return path, skel


@pytest.mark.parametrize("case", ["p24_two_hop_skeleton", "two_networks_side_by_side", "p18_no_skeleton"])
def test_discrete_bn_against_astar(pkg, engine, S, tmp_path, case):
    if case == "p24_two_hop_skeleton":
        codes, card, edges, _ = pkg.datagen.discrete_bn(p=24, n=4000, seed=5, window=3, max_indegree=2)
        path, skel = bn_cache(pkg, engine, tmp_path, codes, card, edges, True)
        rows, skel_file = skel
    elif case == "two_networks_side_by_side":
        c1, k1, e1, _ = pkg.datagen.discrete_bn(p=10, n=3000, seed=6, window=3, max_indegree=2)
        c2, k2, e2, _ = pkg.datagen.discrete_bn(p=9, n=3000, seed=7, window=3, max_indegree=2)
        codes, card = np.concatenate([c1, c2]), np.concatenate([k1, k2])
        edges = list(e1) + [int(e) << 10 for e in e2]
        path, _ = bn_cache(pkg, engine, tmp_path, codes, card, edges, False)
        rows, skel_file = edges, str(tmp_path / "skel.csv")
        pkg.datagen.write_skeleton_matrix(skel_file, rows, 19)
    else:
        codes, card, edges, _ = pkg.datagen.discrete_bn(p=18, n=3000, seed=8, window=4, max_indegree=3)
        path, _ = bn_cache(pkg, engine, tmp_path, codes, card, None, False)
        rows, skel_file = None, None
    cache = S.ScoreCache(path)
    comps = pkg.components(cache.p, rows)
    if case == "two_networks_side_by_side":
        assert len(comps) >= 2
    compare_with_astar(engine, cache, rows, skel_file, case)


def markov_class(parents, p):
    skel = {frozenset((a, b)) for b in range(p) for a in range(p) if (int(parents[b]) >> a) & 1}
    vstruct = set()
    for c in range(p):
        pa = [a for a in range(p) if (int(parents[c]) >> a) & 1]
        for i, a in enumerate(pa):
            for b in pa[i + 1:]:
                if frozenset((a, b)) not in skel:
                    vstruct.add((min(a, b), c, max(a, b)))
    return skel, vstruct


@pytest.mark.parametrize("fig,fn,dag", [("Figure_1", "raw_data_8000.csv", "astar_dag_8000.csv"), ("Figure_2", "raw_data_5000.csv", "astar_dag_5000.csv")])
def test_figures_markov_equivalent_to_published_dag(engine, S, tmp_path, fig, fn, dag):
    skel = os.path.join(DATA, "skeleton4_ones.csv")
    path = str(tmp_path / "gpu.pss")
    subprocess.check_call([EXE, os.path.join(DATA, fig, fn), path, "-k", skel, "-f", "cBIC", "--lambda=2", "--quiet"], stdout=subprocess.DEVNULL)
    m = np.loadtxt(skel, delimiter=",").astype(int)
    rows = [sum(1 << j for j in range(4) if m[i, j]) for i in range(4)]
    cost, parents = engine.optimal_dag(S.ScoreCache(path), rows)
    for kind in ("list", "bitwise"):
        ac = S.ScoreCache(path).astar(kind, 2, skel)[0]
        assert np.float32(cost) <= np.float32(ac) and abs(ac - cost) <= 1e-4 * abs(ac)
    want = np.loadtxt(os.path.join(DATA, fig, dag), delimiter=",").astype(int)
    published = [sum(1 << i for i in range(4) if want[v, i]) for v in range(4)]
    assert markov_class(parents, 4) == markov_class(published, 4)


# ------------------------------------------------------------------------------------------------ limits
@pytest.mark.parametrize("k", [30, 32])
def test_sparse_component_with_closed_form_optimum(engine, k):
    """variable 0: {} 7; variable 1: {} 10, {0} 3; variable j >= 2: {} 10, {j-1} 3, {j-1, j-2} 2.  Integer scores make every
    path sum exact; the only order that gives every variable its best set is 0, 1, ..., k-1, cost 7 + 3 + 2 (k - 2).  At
    k = 32 the graph has 2^32 nodes and node indices cross 32 bits."""
    entries = [(np.array([0], dtype=np.uint64), np.array([7], dtype=np.float32)),
               (np.array([0, 1], dtype=np.uint64), np.array([10, 3], dtype=np.float32))]
    for j in range(2, k):
        entries.append((np.array([0, 1 << (j - 1), (1 << (j - 1)) | (1 << (j - 2))], dtype=np.uint64), np.array([10, 3, 2], dtype=np.float32)))
    cost, order, parents = engine.order_search(entries, k, (1 << k) - 1)
    assert cost == np.float32(7 + 3 + 2 * (k - 2))
    assert order == list(range(k))
    assert [int(x) for x in parents] == [0, 1] + [(1 << (j - 1)) | (1 << (j - 2)) for j in range(2, k)]


def test_one_variable_component(engine):
    entries = [(np.array([0, 2], dtype=np.uint64), np.array([5, 1], dtype=np.float32)),
               (np.array([0], dtype=np.uint64), np.array([4], dtype=np.float32))]
    cost, order, parents = engine.order_search(entries, 2, 0b01)
    assert cost == np.float32(5) and order == [0] and int(parents[0]) == 0 and int(parents[1]) == 0
    cost, order, parents = engine.order_search(entries, 2, 0b10)
    assert cost == np.float32(4) and order == [1]


def write_pss(path, blocks):
    with open(path, "w") as f:
        f.write("META pss_version = 0.1\n\n")
        for name, lines in blocks:
            f.write(f"VAR {name}\nMETA arity=2\n" + "".join(line + "\n" for line in lines) + "\n")


def test_variable_without_cached_subset_like_astar(engine, S, tmp_path):
    """one such variable adds FLT_MAX and the search ends at FLT_MAX, as A* does (every order then costs FLT_MAX, so the DAGs may
    differ); two overflow to +inf: "No solution found.\""""
    one, two = str(tmp_path / "one.pss"), str(tmp_path / "two.pss")
    write_pss(one, [("A", ["-10.0"]), ("B", []), ("C", ["-5.0", "-1.0 A"])])
    write_pss(two, [("A", []), ("B", []), ("C", ["-5.0"])])
    c1 = S.ScoreCache(one)
    cost, parents = engine.optimal_dag(c1)
    ac, ap, _, _ = c1.astar("list")
    assert np.float32(cost) == np.float32(ac) == FLT_MAX and int(parents[1]) == 0 and int(parents[2]) in (0, 1)
    c2 = S.ScoreCache(two)
    with pytest.raises(RuntimeError, match="No solution found."):
        c2.astar("list")
    with pytest.raises(Exception, match="No solution found."):
        engine.optimal_dag(c2)


# ------------------------------------------------------------------------------------------------ refusals
def raw(engine, p, words, offsets, masks, scores, comp, edges=None):
    lib = engine.lib
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    m = np.ascontiguousarray(masks, dtype=np.uint64).reshape(-1)
    s = np.ascontiguousarray(scores, dtype=np.float32)
    cw = np.ascontiguousarray(comp, dtype=np.uint64)
    cost = C.c_float()
    order = np.zeros(64, dtype=np.int32)
    parents = np.zeros(max(1, p) * max(1, words) + 8, dtype=np.uint64)
    rc = lib.urlgpu_order_search(engine._h, p, words, off.ctypes.data, m.ctypes.data if len(m) else None, s.ctypes.data if len(s) else None,
                                 None if edges is None else np.ascontiguousarray(edges, dtype=np.uint64).ctypes.data, cw.ctypes.data,
                                 C.byref(cost), order.ctypes.data, parents.ctypes.data)
    return rc, lib.urlgpu_last_error(engine._h).decode()


def test_every_refusal(engine):
    ok = raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b11])
    assert ok[0] == 0
    assert raw(engine, 0, 1, [0], [], [], [0])[0] == ERR_ARG
    assert raw(engine, 2, 0, [0, 1, 2], [0, 1], [1, 2], [0b11])[0] == ERR_ARG
    assert raw(engine, 2, 5, [0, 1, 2], np.zeros(10), [1, 2], np.full(5, 3))[0] == ERR_ARG
    assert raw(engine, 2, 1, [0, 2, 1], [0, 1], [1, 2], [0b11])[0] == ERR_ARG
    assert raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0])[0] == ERR_ARG
    assert raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b111])[0] == ERR_ARG
    rc, msg = raw(engine, 2, 1, [0, 1, 3], [0, 0, 1], [1, 2, np.nan], [0b11])
    assert rc == ERR_ARG and "variable 1" in msg and "entry 1" in msg and "NaN" in msg
    rc, msg = raw(engine, 2, 1, [0, 1, 3], [0, 0, 2], [1, 2, 3], [0b11])
    assert rc == ERR_ARG and "variable 1" in msg and "entry 1" in msg
    p = 40
    rc, msg = raw(engine, p, 1, np.arange(p + 1), np.zeros(p), np.ones(p), [(1 << 33) - 1])
    assert rc == ERR_LIMIT and "33" in msg
    # a complete candidate set at k = 32: 32 tables of 2^31 entries, 275 GB with the nodes
    full = (1 << 32) - 1
    rc, msg = raw(engine, 32, 1, np.arange(33), [full & ~(1 << v) for v in range(32)], np.ones(32), [full])
    assert rc == ERR_LIMIT and "bytes" in msg
    print(msg)
    # the context still works afterwards
    assert raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b11])[0] == 0
