"""urlgpu_order_local_search_sparse and Engine.order_local_search's choice of form: the climb of urlgpu_order_local_search with
best(v, U) scanned from v's sorted list, so a variable may have any number of candidate parents.  Checked bit for bit against
the table form wherever both run, against the restatement where only the sparse form runs, on real data past the table
form's limit, for the Engine's choice of form, and for every refusal."""
import ctypes as C
import functools
import importlib
import operator

import numpy as np
import pytest

from test_gpu_order_local_search import (CASES, VALUES, Restated, as_int, cache_lookup, cfg3_shaped, check_local, figure,  # noqa: F401
                                         hepatitis, insertion_neighbours_lower, p24_two_hop)
from test_gpu_order_search import bn_cache, random_case

pytestmark = pytest.mark.gpu
ERR_ARG, ERR_LIMIT = -1, -3
TABLE, SPARSE = "urlgpu_order_local_search", "urlgpu_order_local_search_sparse"


@pytest.fixture(scope="module")
def S():
    return importlib.import_module("urlearning-cpp_b200.search")


def assert_same(a, b):
    """two order_local_search results: cost and restart costs as uint32 bits, order, parents, restart moves"""
    assert np.float32(a[0]).view(np.uint32) == np.float32(b[0]).view(np.uint32)
    assert a[1] == b[1]
    assert np.array_equal(a[2], b[2])
    assert np.array_equal(a[3].view(np.uint32), b[3].view(np.uint32))
    assert np.array_equal(a[4], b[4])


def both(engine, entries, p, comp, edges, restarts, seed):
    """the table and sparse forms on one input: equal results, or both "No solution found." -> the result or None"""
    try:
        a = engine._order_local_search(TABLE, entries, p, comp, edges, restarts, seed)
    except Exception as e:
        assert "No solution found." in str(e)
        with pytest.raises(Exception, match="No solution found."):
            engine._order_local_search(SPARSE, entries, p, comp, edges, restarts, seed)
        return None
    b = engine._order_local_search(SPARSE, entries, p, comp, edges, restarts, seed)
    assert_same(a, b)
    return b


def both_on_cache(pkg, engine, cache, edges, restarts=256, seed=0):
    entries = [cache.entries(v) for v in range(cache.p)]
    for comp in pkg.components(cache.p, edges):
        both(engine, entries, cache.p, comp, edges, restarts, seed)


def max_cv(entries, p, comp):
    """the largest c_v over C, counted from the restatement's lists"""
    R = Restated(entries, p, comp)
    return max(bin(functools.reduce(operator.or_, (m for _, m in R.lists[v]), 0)).count("1") for v in R.vs)


# ------------------------------------------------------------------------------------------------ 1. the table form's bits
@pytest.mark.parametrize("name,case", CASES, ids=[c[0] for c in CASES])
def test_same_bits_as_table_form(engine, name, case):
    both(engine, *case, restarts=8, seed=12345)


@pytest.mark.parametrize("prune", [False, True])
def test_hepatitis_same_bits_as_table_form(pkg, engine, S, tmp_path, prune):
    cache = hepatitis(S, tmp_path, prune)
    both_on_cache(pkg, engine, cache, None)
    entries = [cache.entries(v) for v in range(cache.p)]
    comp = (1 << cache.p) - 1
    wide = both(engine, entries, cache.p, comp, None, 4096, 0)
    exact = engine.order_search(entries, cache.p, comp)[0]
    assert np.float32(wide[0]).view(np.uint32) == np.float32(exact).view(np.uint32)


def test_p24_two_hop_same_bits_as_table_form(pkg, engine, S, tmp_path):
    cache, rows = p24_two_hop(pkg, engine, S, tmp_path)
    both_on_cache(pkg, engine, cache, rows)


def test_two_networks_side_by_side_same_bits_as_table_form(pkg, engine, S, tmp_path):
    c1, k1, e1, _ = pkg.datagen.discrete_bn(p=10, n=3000, seed=6, window=3, max_indegree=2)
    c2, k2, e2, _ = pkg.datagen.discrete_bn(p=9, n=3000, seed=7, window=3, max_indegree=2)
    edges = list(e1) + [int(e) << 10 for e in e2]
    path, _ = bn_cache(pkg, engine, tmp_path, np.concatenate([c1, c2]), np.concatenate([k1, k2]), edges, False)
    cache = S.ScoreCache(path)
    assert len(pkg.components(cache.p, edges)) >= 2
    both_on_cache(pkg, engine, cache, edges)


@pytest.mark.parametrize("fig,fn", [("Figure_1", "raw_data_8000.csv"), ("Figure_2", "raw_data_5000.csv")])
def test_figures_same_bits_as_table_form(pkg, engine, S, tmp_path, fig, fn):
    cache, rows = figure(S, tmp_path, fig, fn)
    both_on_cache(pkg, engine, cache, rows)


def test_cfg3_shaped_same_bits_as_table_form(pkg, engine, cfg3_shaped):
    cache, edges = cfg3_shaped
    both_on_cache(pkg, engine, cache, edges)


def spread(entries, p, comp, edges, where, p_new):
    """a case moved to the variables `where` of p_new (masks as ints)"""
    def move(m):
        return sum(1 << where[u] for u in range(p) if (int(m) >> u) & 1)
    out = [([], np.zeros(0, dtype=np.float32)) for _ in range(p_new)]
    for u in range(p):
        out[where[u]] = ([move(x) for x in entries[u][0]], np.asarray(entries[u][1], dtype=np.float32))
    moved = None
    if edges is not None:
        moved = [0] * p_new
        for u in range(p):
            moved[where[u]] = move(edges[u])
    return out, p_new, move(comp), moved


def test_three_mask_words_of_the_component_same_bits_as_table_form(engine):
    """140 variables in p = 200: the sparse form's entries take three words over C"""
    rng = np.random.default_rng(7700)
    k = 140
    where = sorted(rng.choice(200, size=k, replace=False).tolist())
    ent = [([], np.zeros(0, dtype=np.float32)) for _ in range(200)]
    for u in range(k):
        ms, ss = [0], [rng.choice(VALUES)]
        for _ in range(int(rng.integers(0, 8))):
            others = rng.choice([x for x in range(k) if x != u], size=int(rng.integers(1, 4)), replace=False)
            ms.append(sum(1 << where[int(x)] for x in others))
            ss.append(rng.choice(VALUES))
        ent[where[u]] = (ms, np.array(ss, dtype=np.float32))
    cm = sum(1 << w for w in where)
    assert max_cv(ent, 200, cm) <= 32
    assert both(engine, ent, 200, cm, None, 16, 5) is not None


# ------------------------------------------------------------------------------------------------ 2. the restatement past c_v = 32
def heavy_case(rng, k, outside, skeleton, heavy=3):
    """random_case with an empty-set entry for every variable, and `heavy` variables of C given 33..60 candidate parents in
    entries of 1-3 parents"""
    entries, p, comp, edges = random_case(rng, k, outside, VALUES, skeleton)
    vs = [v for v in range(p) if (comp >> v) & 1]
    out = []
    for v in range(p):
        ms, ss = [int(m) for m in entries[v][0]], list(entries[v][1])
        if 0 not in ms:
            ms.append(0)
            ss.append(VALUES[-1])
        out.append((ms, ss))
    for v in rng.choice(vs, size=heavy, replace=False).tolist():
        others = [u for u in vs if u != v]
        pick = rng.choice(others, size=int(rng.integers(33, min(len(others), 60) + 1)), replace=False).tolist()
        while pick:
            n = int(rng.integers(1, 4))
            out[v][0].append(sum(1 << u for u in pick[:n]))
            out[v][1].append(rng.choice(VALUES))
            pick = pick[n:]
    return [(np.array(m, dtype=np.uint64), np.array(s, dtype=np.float32)) for m, s in out], p, comp, edges


def heavy_two_block_case(rng):
    """two 36-variable heavy cases with skeletons, moved to 72 variables of p = 200 and joined by one skeleton edge, and one
    variable given 40..60 candidate parents across both: over C's 72 positions the entries take two words"""
    blocks = [heavy_case(rng, 36, 0, True, heavy=1) for _ in range(2)]
    pos = rng.choice(200, size=72, replace=False).tolist()
    where = [pos[:36], pos[36:]]
    entries = [([], np.zeros(0, dtype=np.float32)) for _ in range(200)]
    edges = [0] * 200

    def move(b, m):
        return sum(1 << where[b][u] for u in range(36) if (int(m) >> u) & 1)
    for b, (ent, _, _, ed) in enumerate(blocks):
        for u in range(36):
            entries[where[b][u]] = ([move(b, x) for x in ent[u][0]], np.asarray(ent[u][1], dtype=np.float32))
            edges[where[b][u]] = move(b, ed[u])
    a, c = where[0][0], where[1][0]
    edges[a] |= 1 << c
    edges[c] |= 1 << a
    v = where[0][1]
    pick = rng.choice([u for u in pos if u != v], size=int(rng.integers(40, 61)), replace=False).tolist()
    ms, ss = list(entries[v][0]), list(entries[v][1])
    while pick:
        n = int(rng.integers(1, 4))
        ms.append(sum(1 << u for u in pick[:n]))
        ss.append(rng.choice(VALUES))
        pick = pick[n:]
    entries[v] = (ms, np.array(ss, dtype=np.float32))
    return entries, 200, sum(1 << u for u in pos), edges


def heavy_cases():
    out = []
    for k, outside in ((40, 6), (48, 0)):
        for skeleton in (False, True):
            out.append((f"k{k}_{'skel' if skeleton else 'none'}", heavy_case(np.random.default_rng(7800 + k + skeleton), k, outside, skeleton)))
    rng = np.random.default_rng(7900)
    case = heavy_case(rng, 44, 0, True)
    where = sorted(rng.choice(np.arange(0, 64), size=8, replace=False).tolist() + rng.choice(np.arange(64, 128), size=12, replace=False).tolist() +
                   rng.choice(np.arange(128, 192), size=16, replace=False).tolist() + list(range(192, 200)))
    out.append(("k44_p200_four_words", spread(*case, where, 200)))
    out.append(("k72_p200_two_words_over_C", heavy_two_block_case(np.random.default_rng(7950))))
    return out


HEAVY = heavy_cases()


@pytest.mark.parametrize("name,case", HEAVY, ids=[c[0] for c in HEAVY])
def test_bit_equal_to_restatement_past_32_candidates(engine, name, case):
    entries, p, comp, edges = case
    assert max_cv(entries, p, comp) > 32
    vs = [v for v in range(p) if (comp >> v) & 1]
    if len(vs) > 64:                                  # some qualifying entry has a parent at a position of C >= 64
        high = sum(1 << v for v in vs[64:])
        assert any(m & high for v in vs for _, m in Restated(entries, p, comp).lists[v])
    with pytest.raises(Exception, match="candidate parents inside the component; at most 32 are supported"):
        engine._order_local_search(TABLE, entries, p, comp, edges, 8, 12345)
    want = Restated(entries, p, comp, edges).run(8, 12345)
    assert want is not None
    cost, order, parents, rc, rm = engine._order_local_search(SPARSE, entries, p, comp, edges, 8, 12345)
    assert np.float32(cost).view(np.uint32) == want[0].view(np.uint32)
    assert order == want[1]
    for v in range(p):
        assert as_int(parents, v) == (want[2][v] if (comp >> v) & 1 else 0)
    assert np.array_equal(rc.view(np.uint32), want[3].view(np.uint32))
    assert np.array_equal(rm, want[4])


# ------------------------------------------------------------------------------------------------ 3. real data past the limit
@pytest.fixture(scope="module")
def cfg3_data_no_skeleton(pkg, tmp_path_factory):
    """configs[3]'s generator, discrete_bn(p=60, n=1e6, seed=4), BIC over all variables at a parent limit of 3, pruned, read back
    from a .pss: one component of 60 whose variables have up to 33 or more candidate parents"""
    n = 1_000_000
    codes, card, _, _ = pkg.datagen.discrete_bn(p=60, n=n, seed=4)
    eng = pkg.Engine(0)
    eng.set_discrete(codes, card)
    caches = {}
    for v in range(60):
        res = eng.score_variable(v, (1 << 60) - 1, 3, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        caches[v] = res.fetch()
        res.free()
    eng.close()
    path = str(tmp_path_factory.mktemp("cfg3n") / "cfg3n.pss")
    pkg.pss.write_pss(path, "cfg3.csv", n, 3, "BIC", [f"X{v}" for v in range(60)], card, caches)
    S = importlib.import_module("urlearning-cpp_b200.search")
    return S.ScoreCache(path)


def test_cfg3_data_without_skeleton(pkg, engine, cfg3_data_no_skeleton):
    cache = cfg3_data_no_skeleton
    p, comp = 60, (1 << 60) - 1
    entries = [cache.entries(v) for v in range(p)]
    cv = max_cv(entries, p, comp)
    assert cv > 32
    with pytest.raises(Exception, match="candidate parents inside the component; at most 32 are supported"):
        engine._order_local_search(TABLE, entries, p, comp, None, 8, 0)
    a = engine._order_local_search(SPARSE, entries, p, comp, None, 256, 0)
    cost, order, parents, rc, rm = a
    check_local(cache_lookup(cache), entries, p, comp, None, cost, order, parents)
    assert insertion_neighbours_lower(cache, order, [comp] * p, cost) == []
    assert_same(a, engine._order_local_search(SPARSE, entries, p, comp, None, 256, 0))
    c = engine._order_local_search(SPARSE, entries, p, comp, None, 64, 0)
    assert np.array_equal(c[3].view(np.uint32), rc[:64].view(np.uint32)) and np.array_equal(c[4], rm[:64])
    assert np.float32(cost) == rc.min()
    total, dag = engine.local_search_dag(cache, None, restarts=256, seed=0)
    assert np.float32(total).view(np.uint32) == np.float32(cost).view(np.uint32) and np.array_equal(dag, parents)
    print(f"max c_v {cv}, cost {cost!r}, restart costs {rc.min()!r}..{rc.max()!r}, moves mean {rm.mean():.1f} max {rm.max()}")


# ------------------------------------------------------------------------------------------------ 4. the Engine's choice
def test_engine_chooses_the_form_by_table_bytes(pkg, engine, monkeypatch):
    called = []
    direct = engine._order_local_search

    def spy(symbol, *a, **kw):
        called.append(symbol)
        return direct(symbol, *a, **kw)
    monkeypatch.setattr(engine, "_order_local_search", spy)
    small = next(c for n, c in CASES if n.startswith("wide24_skel"))
    large = HEAVY[0][1]
    # every c_v <= 32, but twelve variables with c_v = 32 need 12 tables of 2^32 entries, 206 GB, which the table form refuses
    # (their empty set, at a worse score, keeps every order finite)
    p = 33
    full = (1 << p) - 1
    fits_not = ([(np.array([full & ~(1 << v), 0], dtype=np.uint64), np.array([1, 2], dtype=np.float32)) for v in range(12)] +
                [(np.zeros(1, dtype=np.uint64), np.ones(1, dtype=np.float32)) for _ in range(p - 12)], p, full, None)
    assert max_cv(*fits_not[:3]) == 32
    with pytest.raises(Exception, match="the search needs"):
        direct(TABLE, *fits_not, 8, 9)
    for case, want in ((small, TABLE), (large, SPARSE), (fits_not, SPARSE)):
        args = engine._order_args(*case)
        assert (pkg.table_bytes(args[1], args[2], args[4]) <= pkg.TABLE_MAX_BYTES) == (want == TABLE)
        called.clear()
        got = engine.order_local_search(*case, restarts=8, seed=9)
        assert called == [want]
        assert_same(got, direct(want, *case, 8, 9))


# ------------------------------------------------------------------------------------------------ 5. refusals
def raw(engine, p, words, offsets, masks, scores, comp, edges=None, restarts=8, symbol=SPARSE):
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    m = np.ascontiguousarray(masks, dtype=np.uint64).reshape(-1)
    s = np.ascontiguousarray(scores, dtype=np.float32)
    cw = np.ascontiguousarray(comp, dtype=np.uint64)
    ed = None if edges is None else np.ascontiguousarray(edges, dtype=np.uint64)
    cost = C.c_float()
    order = np.zeros(512, dtype=np.int32)
    parents = np.zeros(max(1, p) * max(1, words) + 8, dtype=np.uint64)
    rc = getattr(engine.lib, symbol)(engine._h, p, words, off.ctypes.data, m.ctypes.data if len(m) else None, s.ctypes.data if len(s) else None,
                                     None if ed is None else ed.ctypes.data, cw.ctypes.data, restarts, 0, C.byref(cost), order.ctypes.data,
                                     parents.ctypes.data, None, None)
    return rc, engine.lib.urlgpu_last_error(engine._h).decode()


def test_every_refusal(engine):
    def works():
        assert raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b11])[0] == 0

    works()
    same_as_table = [
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
    for args in same_as_table:
        rc, msg = raw(engine, *args)
        trc, tmsg = raw(engine, *args, symbol=TABLE)
        assert rc == trc == ERR_ARG
        assert msg.startswith("order_local_search_sparse: ") and tmsg.startswith("order_local_search: ")
        assert msg[len("order_local_search_sparse: "):] == tmsg[len("order_local_search: "):]
        works()
    for restarts in (0, (1 << 20) + 1):
        rc, msg = raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b11], restarts=restarts)
        assert rc == ERR_ARG and msg == "order_local_search_sparse: restarts must be in 1..2^20"
        works()
    assert raw(engine, 2, 1, [0, 1, 2], [0, 1], [1, 2], [0b11], restarts=1 << 20)[0] == 0
    # a component of 257 variables needs a fifth mask word, which both forms refuse; 256 are accepted
    p = 257
    args = (p, 5, np.arange(p + 1), np.zeros((p, 5)), np.ones(p), [(1 << 64) - 1] * 4 + [1])
    rc, msg = raw(engine, *args)
    trc, tmsg = raw(engine, *args, symbol=TABLE)
    assert rc == trc == ERR_ARG and msg == "order_local_search_sparse: mask_words must be in 1..4" and tmsg == "order_local_search: mask_words must be in 1..4"
    works()
    assert raw(engine, 256, 4, np.arange(257), np.zeros((256, 4)), np.ones(256), [(1 << 64) - 1] * 4)[0] == 0
    # c_v = 33, which the table form refuses, and c_v = 255
    p = 34
    masks = [((1 << p) - 1) & ~1] + [0] * (p - 1)
    assert raw(engine, p, 1, np.arange(p + 1), masks, np.ones(p), [(1 << p) - 1], symbol=TABLE)[0] == ERR_LIMIT
    assert raw(engine, p, 1, np.arange(p + 1), masks, np.ones(p), [(1 << p) - 1])[0] == 0
    full = [(1 << 64) - 1] * 4
    masks = np.zeros((256, 4), dtype=np.uint64)
    masks[0] = full
    masks[0, 0] ^= np.uint64(1)
    assert raw(engine, 256, 4, np.arange(257), masks, np.ones(256), full)[0] == 0
    # no admissible order (the skeleton splits the component), and a best cost of +inf
    rc, msg = raw(engine, 2, 1, [0, 1, 2], [0, 0], [1, 2], [0b11], edges=[0, 0])
    assert rc == ERR_ARG and msg == "No solution found."
    works()
    rc, msg = raw(engine, 3, 1, [0, 0, 0, 1], [0], [1], [0b111])     # FLT_MAX + FLT_MAX in every order
    assert rc == ERR_ARG and msg == "No solution found."
    works()
