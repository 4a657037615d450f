"""urlgpu_order_search_layered: the order-graph search with two cost layers in colex rank and one leaf byte per node, for
components of up to 36 variables.  Checked bit for bit against urlgpu_order_search (and the numpy restatement) wherever
both run, against closed-form optima above 32 variables (leaf offsets past 2^32 at 33, ranks inside one layer past 2^32 at
35), at 36 variables against the device's free memory, against the host A* through Engine.optimal_dag, and for every
refusal."""
import ctypes as C
import importlib
import math
import os
import subprocess

import numpy as np
import pytest

from test_gpu_order_search import DATA, ERR_ARG, ERR_LIMIT, EXE, bn_cache, check_dag, compare_with_astar, random_case, raw, restate

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def S():
    return importlib.import_module("urlearning-cpp_b200.search")


def pack(entries, p, comp, edges=None):
    """entries as Engine.order_search takes them (int or uint64 masks) -> the arrays of the C ABI"""
    words = max(1, (p + 63) // 64)

    def w(x):
        return [(int(x) >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(words)]
    offsets = np.zeros(p + 1, dtype=np.uint64)
    masks, scores = [], []
    for v, (m, s) in enumerate(entries):
        masks += [w(x) for x in m]
        scores += [float(x) for x in np.asarray(s, dtype=np.float32).reshape(-1)]
        offsets[v + 1] = offsets[v] + len(m)
    return (p, words, offsets, np.array(masks, dtype=np.uint64).reshape(-1, words), np.array(scores, dtype=np.float32), w(comp),
            None if edges is None else [w(e) for e in edges])


def call(engine, fn, p, words, offsets, masks, scores, comp, edges=None):
    """one call of urlgpu_order_search{,_layered} -> (rc, message, cost bits, order, parents [p, words])"""
    lib = engine.lib
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    m = np.ascontiguousarray(masks, dtype=np.uint64).reshape(-1)
    s = np.ascontiguousarray(scores, dtype=np.float32)
    cw = np.ascontiguousarray(comp, dtype=np.uint64)
    ed = None if edges is None else np.ascontiguousarray(edges, dtype=np.uint64)
    cost = C.c_float()
    order = np.zeros(64, dtype=np.int32)
    parents = np.zeros((max(1, p), max(1, words)), dtype=np.uint64)
    rc = getattr(lib, fn)(engine._h, p, words, off.ctypes.data, m.ctypes.data if len(m) else None, s.ctypes.data if len(s) else None,
                          None if ed is None else ed.ctypes.data, cw.ctypes.data, C.byref(cost), order.ctypes.data, parents.ctypes.data)
    k = sum(bin(int(x)).count("1") for x in cw)
    return rc, lib.urlgpu_last_error(engine._h).decode(), np.float32(cost.value).view(np.uint32), [int(x) for x in order[:k]], parents


def assert_same_as_dense(engine, entries, p, comp, edges=None):
    """both entry points on one input: the same return code and, on success, the same cost bits, order and parents"""
    args = pack(entries, p, comp, edges)
    d = call(engine, "urlgpu_order_search", *args)
    l = call(engine, "urlgpu_order_search_layered", *args)
    assert l[0] == d[0], (d[1], l[1])
    if d[0] == 0:
        assert l[2] == d[2] and l[3] == d[3] and np.array_equal(l[4], d[4])
    else:
        assert l[1] == d[1] == "No solution found."
    return d


# ------------------------------------------------------------------------------------------------ closed-form caches
def chain(k):
    """test_sparse_component_with_closed_form_optimum's cache: the only optimal order is 0, 1, ..., k-1, cost 7 + 3 + 2 (k - 2)"""
    entries = [(np.array([0], dtype=np.uint64), np.array([7], dtype=np.float32)),
               (np.array([0, 1], dtype=np.uint64), np.array([10, 3], dtype=np.float32))]
    for j in range(2, k):
        entries.append((np.array([0, 1 << (j - 1), (1 << (j - 1)) | (1 << (j - 2))], dtype=np.uint64), np.array([10, 3, 2], dtype=np.float32)))
    return entries


def planted(p, vs, rng):
    """the chain over the variables vs in a random order q (q[0] {} 7; q[1] {} 10, {q[0]} 3; q[j] {} 10, {q[j-1]} 3,
    {q[j-1], q[j-2]} 2), with a decoy {q[j+1]} 1 for every third j: a decoy saves 1 but puts q[j+1] before q[j], which then
    pays 10 instead of 2, so the chain order q, cost 7 + 3 + 2 (k - 2), is the only optimum.  Where p > |vs|, every fourth
    q[j] also gets a best entry {u} with u outside vs, which never qualifies.  -> (entries, q, parents {v: mask})"""
    q = [int(x) for x in rng.permutation(vs)]
    k = len(q)
    entries = [([0], [1]) for _ in range(p)]
    want = {q[0]: 0, q[1]: 1 << q[0]}
    entries[q[0]] = ([0], [7])
    entries[q[1]] = ([0, 1 << q[0]], [10, 3])
    for j in range(2, k):
        ms, ss = [0, 1 << q[j - 1], (1 << q[j - 1]) | (1 << q[j - 2])], [10, 3, 2]
        if j % 3 == 2 and j + 1 < k:
            ms.append(1 << q[j + 1])
            ss.append(1)
        entries[q[j]] = (ms, ss)
        want[q[j]] = (1 << q[j - 1]) | (1 << q[j - 2])
    outside = [v for v in range(p) if v not in want]
    for v in outside:
        entries[v] = ([0, 1 << q[0]], [1, 0.5])
    for j in range(0, k, 4) if outside else ():              # the best entry of q[j], never inside the component
        entries[q[j]][0].append(1 << outside[j % len(outside)])
        entries[q[j]][1].append(0)
    entries = [(np.array(m, dtype=object), np.array(s, dtype=np.float32)) for m, s in entries]
    return entries, q, want


def closed_form(k):
    return np.float32(7 + 3 + 2 * (k - 2))


# ------------------------------------------------------------------------------------------------ same bits as urlgpu_order_search
@pytest.mark.parametrize("k", [1, 2, 5, 9, 12, 14, 20, 24])
@pytest.mark.parametrize("skeleton", [False, True])
def test_bit_equal_to_dense_form(engine, k, skeleton):
    """tie-heavy random caches with entries reaching outside the component: cost, order and parents of
    urlgpu_order_search_layered equal urlgpu_order_search's bit for bit, and the numpy restatement's where k <= 14"""
    rng = np.random.default_rng(7000 + 100 * k + skeleton)
    values = np.array([0.1, 0.7, 1.3, 2.0, 2.5, 3.0], dtype=np.float32)
    for _ in range(4 if k <= 14 else 2):
        entries, p, comp, edges = random_case(rng, k, 2, values, skeleton)
        d = assert_same_as_dense(engine, entries, p, comp, edges)
        if k > 14:
            continue
        want = restate(entries, p, comp, edges)
        assert (want is None) == (d[0] != 0)
        if want is not None:
            assert d[2] == want[0].view(np.uint32) and d[3] == want[1]
            for v in range(p):
                assert int(d[4][v, 0]) == (want[2][v] if (comp >> v) & 1 else 0)


def test_hepatitis_bit_equal_to_dense_form(engine, S, tmp_path):
    path = str(tmp_path / "hepatitis.pss")
    subprocess.check_call([EXE, os.path.join(DATA, "hepatitis.clean.csv"), path, "-s", "-f", "BIC", "--quiet"], stdout=subprocess.DEVNULL)
    cache = S.ScoreCache(path)
    d = assert_same_as_dense(engine, [cache.entries(v) for v in range(cache.p)], cache.p, (1 << cache.p) - 1)
    assert d[0] == 0


@pytest.mark.parametrize("k", [30, 32])
def test_closed_form_bit_equal_to_dense_form(engine, k):
    d = assert_same_as_dense(engine, chain(k), k, (1 << k) - 1)
    assert d[0] == 0 and d[2] == closed_form(k).view(np.uint32) and d[3] == list(range(k))


# ------------------------------------------------------------------------------------------------ above 32 variables
@pytest.mark.parametrize("k", [33, 34, 35])
def test_chain_above_32(engine, k):
    """33: leaf offsets pass 2^32; 35: C(35, 17) = 4 537 567 650 ranks inside one layer"""
    cost, order, parents = engine.order_search(chain(k), k, (1 << k) - 1)
    assert cost.view(np.uint32) == closed_form(k).view(np.uint32)
    assert order == list(range(k))
    assert [int(x) for x in parents] == [0, 1] + [(1 << (j - 1)) | (1 << (j - 2)) for j in range(2, k)]


def test_planted_optimum_with_decoys(engine):
    k = 33
    entries, q, want = planted(k, list(range(k)), np.random.default_rng(33))
    assert q != list(range(k))
    cost, order, parents = engine.order_search(entries, k, (1 << k) - 1)
    assert cost.view(np.uint32) == closed_form(k).view(np.uint32)
    assert order == q
    assert {v: int(parents[v]) for v in range(k)} == want


def test_two_mask_words_equal_one(engine):
    """a 34-variable component spread over p = 70 (variables on both sides of 64) gives what the same component
    renumbered into one word gives"""
    rng = np.random.default_rng(70)
    vs = sorted(int(x) for x in rng.choice(70, size=34, replace=False))
    assert vs[0] < 64 <= vs[-1]
    entries, q, want = planted(70, vs, rng)
    comp = sum(1 << v for v in vs)
    cost, order, parents = engine.order_search(entries, 70, comp)
    assert parents.shape == (70, 2)
    assert cost.view(np.uint32) == closed_form(34).view(np.uint32) and order == q
    for v in range(70):
        got = int(parents[v, 0]) | (int(parents[v, 1]) << 64)
        assert got == (want[v] if v in want else 0)
    new = {v: i for i, v in enumerate(vs)}

    def renum(m):
        return sum(1 << new[v] for v in range(70) if (int(m) >> v) & 1)
    inside = [[i for i, m in enumerate(entries[v][0]) if int(m) & ~comp == 0] for v in vs]   # the others never qualify
    one = [(np.array([renum(entries[v][0][i]) for i in ix], dtype=np.uint64), entries[v][1][ix]) for v, ix in zip(vs, inside)]
    c1, o1, p1 = engine.order_search(one, 34, (1 << 34) - 1)
    assert c1.view(np.uint32) == cost.view(np.uint32)
    assert o1 == [new[v] for v in order]
    assert [int(x) for x in p1] == [renum(want[v]) for v in vs]


def layered_bytes(k, cand_bits, n_ent):
    """the device memory urlgpu_order_search_layered asks for (include/urlgpu.h)"""
    return (1 << k) + 8 * math.comb(k, k // 2) + sum(4 << c for c in cand_bits) + 16 * n_ent + 1328 * k + 10960


def test_36_variables_fit_or_refused_with_their_bytes(engine):
    k = 36
    need = layered_bytes(k, [0, 1] + [2] * (k - 2), 1 + 2 + 3 * (k - 2))
    rc, msg, cost, order, parents = call(engine, "urlgpu_order_search_layered", *pack(chain(k), k, (1 << k) - 1))
    print(f"k = 36: {need} bytes: rc {rc} {msg}")
    if rc == 0:
        assert cost == closed_form(k).view(np.uint32) and order == list(range(k))
        assert [int(x) for x in parents[:, 0]] == [0, 1] + [(1 << (j - 1)) | (1 << (j - 2)) for j in range(2, k)]
    else:
        assert rc == ERR_LIMIT and f"{need} bytes of device memory" in msg


# ------------------------------------------------------------------------------------------------ against A*
class CountingLib:
    """engine.lib with a count of the order-search calls per entry point"""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        f = getattr(self._lib, name)
        if not name.startswith("urlgpu_order_search"):
            return f

        def counted(h, p, words, offsets, masks, scores, edges, comp, *rest):
            k = sum(bin(int(x)).count("1") for x in np.ctypeslib.as_array(C.cast(comp, C.POINTER(C.c_uint64)), (words,)))
            self.calls.append((name, k))
            return f(h, p, words, offsets, masks, scores, edges, comp, *rest)
        return counted


@pytest.mark.parametrize("p,skeleton,seed", [(34, False, 1), (34, True, 1), (36, False, 2), (36, True, 2)])
def test_discrete_bn_against_astar(pkg, engine, S, tmp_path, p, skeleton, seed):
    """BIC at -p 3, pruned; seeds where A*'s pattern-database heuristic lets the host finish within seconds"""
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=p, n=4000, seed=seed, window=3, max_indegree=2)
    path, skel = bn_cache(pkg, engine, tmp_path, codes, card, edges if skeleton else None, skeleton)
    rows, skel_file = skel if skeleton else (None, None)
    assert pkg.components(p, rows) == [(1 << p) - 1]
    cache = S.ScoreCache(path)
    try:
        compare_with_astar(engine, cache, rows, skel_file, f"p{p}")
    except pkg.UrlGpuError as e:
        if "bytes of device memory" not in str(e):
            raise
        pytest.skip(f"the device has too little free memory: {e}")


def test_components_reach_their_own_form(pkg, engine, S, tmp_path):
    """one 34-variable component and three small ones in one skeleton: the large one through urlgpu_order_search_layered,
    the small ones through urlgpu_order_search, each once per search; the result agrees with A*"""
    parts = [pkg.datagen.discrete_bn(p=n, n=4000, seed=s, window=3, max_indegree=2) for n, s in ((34, 1), (5, 3), (4, 4), (3, 5))]
    codes = np.concatenate([c for c, _, _, _ in parts])
    card = np.concatenate([k for _, k, _, _ in parts])
    edges, at = [], 0
    for c, _, e, _ in parts:
        edges += [int(x) << at for x in e]
        at += len(c)
    path, skel = bn_cache(pkg, engine, tmp_path, codes, card, edges, True)
    rows, skel_file = skel
    comps = pkg.components(at, rows)
    sizes = sorted(bin(c).count("1") for c in comps)
    assert sizes[-1] == 34 and len(sizes) >= 4
    eng = pkg.Engine(0)
    try:
        eng.lib = CountingLib(eng.lib)
        eng.optimal_dag(S.ScoreCache(path), rows)
        assert sorted(eng.lib.calls, key=lambda c: c[1]) == sorted(
            [("urlgpu_order_search_layered" if n > 32 else "urlgpu_order_search", n) for n in sizes], key=lambda c: c[1])
    finally:
        eng.lib = eng.lib._lib if isinstance(eng.lib, CountingLib) else eng.lib
        eng.close()
    compare_with_astar(engine, S.ScoreCache(path), rows, skel_file, "p46 components")


# ------------------------------------------------------------------------------------------------ refusals
def works(engine):
    args = pack(chain(5), 5, 0b11111)
    rc, _, cost, order, _ = call(engine, "urlgpu_order_search_layered", *args)
    return rc == 0 and cost == closed_form(5).view(np.uint32) and order == list(range(5))


ARG_CASES = [   # the refusals of test_every_refusal in tests/test_gpu_order_search.py
    (0, 1, [0], [], [], [0]),
    (2, 0, [0, 1, 2], [0, 1], [1, 2], [0b11]),
    (2, 5, [0, 1, 2], np.zeros(10), [1, 2], np.full(5, 3)),
    (2, 1, [0, 2, 1], [0, 1], [1, 2], [0b11]),
    (2, 1, [0, 1, 2], [0, 1], [1, 2], [0]),
    (2, 1, [0, 1, 2], [0, 1], [1, 2], [0b111]),
    (2, 1, [0, 1, 3], [0, 0, 1], [1, 2, np.nan], [0b11]),
    (2, 1, [0, 1, 3], [0, 0, 2], [1, 2, 3], [0b11]),
]


def test_arg_refusals_as_dense(engine):
    for case in ARG_CASES:
        rc_d, msg_d = raw(engine, *case)
        rc, msg = call(engine, "urlgpu_order_search_layered", *case)[:2]
        assert rc_d == rc == ERR_ARG
        assert msg_d.startswith("order_search: ") and msg == "order_search_layered: " + msg_d[len("order_search: "):]
        assert works(engine)


def test_limit_refusals(engine):
    p = 40
    rc, msg = call(engine, "urlgpu_order_search_layered", p, 1, np.arange(p + 1), np.zeros(p), np.ones(p), [(1 << 37) - 1])[:2]
    assert rc == ERR_LIMIT and "37 variables" in msg and "at most 36" in msg
    assert works(engine)
    # complete candidate sets at k = 36: 36 tables of 2^35 entries
    full = (1 << 36) - 1
    rc, msg = call(engine, "urlgpu_order_search_layered", 36, 1, np.arange(37), [full & ~(1 << v) for v in range(36)], np.ones(36), [full])[:2]
    need = layered_bytes(36, [35] * 36, 36)
    print(msg)
    assert rc == ERR_LIMIT
    assert f"needs {need} bytes of device memory ({1 << 36} for the leaves of the 2^36 nodes, {8 * math.comb(36, 18)} for two cost " \
           f"layers of C(36, 18) nodes, {36 * (4 << 35)} for the best-parent tables)" in msg
    assert works(engine)


def test_no_solution_found(engine):
    # no admissible order: the skeleton has no edge inside the component
    rc, msg = call(engine, "urlgpu_order_search_layered", 2, 1, [0, 1, 2], [0, 0], [1, 2], [0b11], [0b01, 0b10])[:2]
    assert rc == ERR_ARG and msg == "No solution found."
    assert works(engine)
    # every order costs +inf: two variables without a cached subset, FLT_MAX + FLT_MAX
    rc, msg = call(engine, "urlgpu_order_search_layered", 3, 1, [0, 0, 0, 1], [0], [5], [0b111])[:2]
    assert rc == ERR_ARG and msg == "No solution found."
    assert works(engine)
