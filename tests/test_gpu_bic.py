"""GPU parity: discrete BIC through the C ABI vs the CPU oracle (bit-exact counts, scores and stored lists)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check_variable(pkg, orc, eng, codes, card, edges, v, K, flags=0):
    p = codes.shape[0]
    nb = pkg.two_hop_neighbors(edges, p, v)
    res = eng.score_variable(v, nb, K, pkg.BIC, flags=flags)
    masks, scores = res.fetch()
    om = orc.enumerate_sets(v, nb, p, K)
    osc = orc.bic_score_many(codes, card, v, om)
    stored = np.array([(s < 1) if m == 0 else (s < 0) for m, s in zip(om, osc)])
    om, osc = om[stored], osc[stored]
    if flags & pkg.PRUNE_DOMINATED:
        keep = orc.prune(om, osc, K)
        om, osc = om[keep], osc[keep]
    order = orc.canonical_order(om)
    assert res.scored() == len(stored)
    assert [int(m[0]) for m in masks] == [int(om[i]) for i in order]
    assert np.array_equal(scores.view(np.uint32), osc[order].view(np.uint32))
    res.free()
    return len(order)


def test_hepatitis_all_variables(pkg, orc, bic_engine, data_dir):
    engine = bic_engine
    t = orc.Table(os.path.join(data_dir, "hepatitis.clean.csv"), has_header=True)
    codes = t.codes()
    engine.set_discrete(codes, t.card)
    K = pkg.effective_max_parents(0, t.p, t.n, True)
    assert K == 3
    total = sum(_check_variable(pkg, orc, engine, codes, t.card, None, v, K) for v in range(t.p))
    assert total == 23200  # SURVEY.md §4


def test_contingency_counts_ragged_rows(pkg, orc, engine):
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=12, n=10007, seed=11, arities=(2, 3, 4))
    engine.set_discrete(codes, card)
    rng = np.random.default_rng(0)
    for _ in range(25):
        v = int(rng.integers(12))
        k = int(rng.integers(0, 8))
        others = [i for i in range(12) if i != v]
        parents = sum(1 << int(i) for i in rng.choice(others, size=k, replace=False))
        ref = orc.bic_counts(codes, card, v, parents)
        got = engine.contingency(v, parents, len(ref))
        assert got.sum() == 10007
        assert np.array_equal(got, ref)
        s, ll = engine.score_one(v, parents, pkg.BIC)
        rs, rll = orc.bic_score(codes, card, v, parents)
        assert s.view(np.uint32) == rs.view(np.uint32) and ll == rll


@pytest.mark.parametrize("n", [1, 15, 16, 17, 4097])
def test_tiny_and_edge_row_counts(pkg, orc, bic_engine, n):
    engine = bic_engine
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=6, n=max(n, 2), seed=n, arities=(2, 3))
    codes = codes[:, :n].copy()
    if n < 3:  # N=1: log(1)=0 -> the reference's BIC parent cap divides by zero; use N=2 instead
        codes = np.array([[0, 1], [0, 0], [1, 0], [0, 1], [0, 0], [1, 1]], dtype=np.uint8)
        card = np.array([2, 1, 2, 2, 1, 2], dtype=np.int32)
    else:
        card = np.array([max(1, int(c.max()) + 1) for c in codes], dtype=np.int32)
    engine.set_discrete(codes, card)
    for v in range(6):
        _check_variable(pkg, orc, engine, codes, card, None, v, 5)


def test_all_tiers_arity4(pkg, orc, bic_engine):
    engine = bic_engine
    """tables from 4 cells to 4^10 = 1M cells: small shared tier, one-CTA-per-SM shared tier and the global tier"""
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=11, n=20011, seed=5, arities=(4,), window=10, max_indegree=3)
    engine.set_discrete(codes, card)
    for v in (0, 5, 10):
        _check_variable(pkg, orc, engine, codes, card, None, v, 9)


@pytest.mark.parametrize("fuse,budget", [("1", 22528), ("1", 2048), ("0", 22528), ("1", 40000), ("0", 2048)])
def test_cube_roots_counted_in_slices_and_fused(pkg, orc, fuse, budget):
    """the cube path's big roots: counted in shared-memory slices of the packed rows; ancestor-only roots (layer K+1) hand
    their children straight to the next layer (fused) or, with URLGPU_FUSE_ROOTS=0 / a run that does not fit the slice
    budget, are written out and marginalised through HBM.  Edge shapes: every set a root's descendant (K = c - 1), a
    single parent, the empty set alone.  All variants bit-exact against the oracle."""
    keys = {"URLGPU_BIC_MODE": "cube", "URLGPU_FUSE_ROOTS": fuse, "URLGPU_ROOT_BUDGET": str(budget)}
    old = {k: os.environ.get(k) for k in keys}
    os.environ.update(keys)
    try:
        eng = pkg.Engine(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=14, n=70003, seed=31, arities=(2, 3, 4), window=6, max_indegree=3)
    eng.set_discrete(codes, card)
    for v, K in ((2, 9), (11, 8), (5, 10), (0, 13), (9, 1), (3, 0)):
        _check_variable(pkg, orc, eng, codes, card, None, v, K)
    _check_variable(pkg, orc, eng, codes, card, None, 7, 9, flags=pkg.PRUNE_DOMINATED)
    eng.close()


def test_skeleton_two_hop_and_prune(pkg, orc, bic_engine):
    engine = bic_engine
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=24, n=30000, seed=7, window=3, max_indegree=2)
    engine.set_discrete(codes, card)
    K = pkg.effective_max_parents(12, 24, 30000, True)
    for v in (0, 3, 11, 23):
        _check_variable(pkg, orc, engine, codes, card, edges, v, K)
        _check_variable(pkg, orc, engine, codes, card, edges, v, K, flags=pkg.PRUNE_DOMINATED)


def test_row_permutation_invariance_and_counts_sum(pkg, orc, bic_engine):
    engine = bic_engine
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=10, n=50000, seed=9)
    perm = np.random.default_rng(1).permutation(50000)
    engine.set_discrete(codes, card)
    a = engine.score_variable(4, (1 << 10) - 1, 6, pkg.BIC).fetch()
    engine.set_discrete(codes[:, perm], card)
    b = engine.score_variable(4, (1 << 10) - 1, 6, pkg.BIC).fetch()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))


def test_score_binary_matches_oracle_pss(pkg, orc, data_dir, tmp_path):
    """the product `score` binary vs the oracle's restatement of score_main.cpp: identical bytes"""
    exe = os.path.join(ROOT, "urlearning-cpp_b200", "score")
    inp = os.path.join(data_dir, "hepatitis.clean.csv")
    out = str(tmp_path / "gpu.pss")
    ref = str(tmp_path / "ref.pss")
    subprocess.check_call([exe, inp, out, "-s", "-f", "BIC", "--quiet"], stdout=subprocess.DEVNULL)
    orc.score_file(inp, ref, "BIC", has_header=True)
    gb, rb = open(out, "rb").read(), open(ref, "rb").read()
    assert gb == rb
    meta, variables = orc.parse_pss(out)
    assert meta["num_records"] == "80" and meta["parent_limit"] == "3" and len(variables) == 20
    # with pruning and 2 worker threads
    subprocess.check_call([exe, inp, out, "-s", "--prune", "-t", "2", "--quiet"], stdout=subprocess.DEVNULL)
    orc.score_file(inp, ref, "BIC", has_header=True, prune=True)
    assert open(out, "rb").read() == open(ref, "rb").read()


@pytest.mark.parametrize("arities", [(2, 5, 9), (3, 16), (6, 18)])
def test_wide_arities_packed_rows(pkg, orc, bic_engine, arities):
    """arities above 4 switch the packed rows to 4- and 8-bit fields; big root tables (9^6 cells and more) go through the
    shared-memory root kernel (fused and plain), smaller ones through the other tiers"""
    engine = bic_engine
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=9, n=70001, seed=41, arities=arities, window=8, max_indegree=2)
    engine.set_discrete(codes, card)
    for v, K in ((0, 5), (4, 6), (8, 4)):
        _check_variable(pkg, orc, engine, codes, card, None, v, K)


def test_bic_wide_masks_p_above_64(pkg, orc, engine):
    """p = 130 variables (three 64-bit words per varset), the shape of bench.py's weak-scaling data set (60 N variables):
    checked bit for bit against the oracle on the relabelled sub-problem of the variable's 2-hop candidates"""
    p = 130
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=p, n=20011, seed=23, window=3, max_indegree=2)
    engine.set_discrete(codes, card)
    for v in (1, 64, 129):
        nb = pkg.two_hop_neighbors(edges, p, v)
        res = engine.score_variable(v, nb, 6, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        masks, scores = res.fetch()
        res.free()
        assert masks.shape[1] == 3
        sub = sorted({i for i in range(p) if (nb >> i) & 1} | {v})
        vs = sub.index(v)
        om = orc.enumerate_sets(vs, (1 << len(sub)) - 1, len(sub), 6)
        osc = orc.bic_score_many(codes[sub], card[sub], vs, om)
        stored = np.array([(s < 1) if m == 0 else (s < 0) for m, s in zip(om, osc)])
        om, osc = om[stored], osc[stored]
        keep = orc.prune(om, osc, 6)
        om, osc = om[keep], osc[keep]
        order = orc.canonical_order(om)
        want = [sum(1 << sub[i] for i in range(len(sub)) if (int(om[j]) >> i) & 1) for j in order]
        assert [pkg.words_to_mask(row) for row in masks] == want
        assert np.array_equal(scores.view(np.uint32), osc[order].view(np.uint32))


def test_pipelined_prefetch_matches_plain_fetch(pkg, engine):
    """prefetch(v) / score(v+1) / fetch(v): the compaction is enqueued behind the scoring kernels and the payload is copied
    on a second stream while the next variable runs; results must equal the unpipelined ones, in canonical order"""
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=20, n=70001, seed=13, window=4, max_indegree=3)
    engine.set_discrete(codes, card)
    K = 6
    nbs = [pkg.two_hop_neighbors(edges, 20, v) for v in range(20)]
    plain = []
    for v in range(20):
        r = engine.score_variable(v, nbs[v], K, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        plain.append(r.fetch())
        r.free()
    for rep in range(2):
        got, prev = [], None
        for v in range(20):
            r = engine.score_variable(v, nbs[v], K, pkg.BIC, flags=pkg.PRUNE_DOMINATED).prefetch()
            if prev is not None:
                got.append(prev.fetch())
                prev.free()
            prev = r
        got.append(prev.fetch())
        prev.free()
        for (m0, s0), (m1, s1) in zip(plain, got):
            assert np.array_equal(m0, m1) and np.array_equal(s0.view(np.uint32), s1.view(np.uint32))
            pc = [bin(int(x)).count("1") for x in m1[:, 0]]
            assert pc == sorted(pc)  # canonical order: layer by layer


def test_pinned_fetch_equals_plain_fetch(pkg, engine):
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=16, n=30011, seed=19, window=4, max_indegree=3)
    engine.set_discrete(codes, card)
    for v in (0, 7, 15):
        r = engine.score_variable(v, pkg.two_hop_neighbors(edges, 16, v), 6, pkg.BIC)
        m0, s0 = r.fetch()
        m1, s1 = r.fetch(pinned=True)
        assert np.array_equal(m0, m1) and np.array_equal(s0.view(np.uint32), s1.view(np.uint32))
        r.free()
    pool = pkg.EnginePool(0, 2)
    pool.set_discrete(codes, card)
    items = [(v, pkg.two_hop_neighbors(edges, 16, v)) for v in range(16)]
    full = pool.run(items, 6, pkg.BIC, fetch=True)
    counts = pool.run(items, 6, pkg.BIC, fetch="pinned")
    assert {v: len(x[1]) for v, x in full.items()} == counts
    pool.close()


def test_engine_pool_matches_single_engine(pkg, engine):
    """three contexts on one device driven by three host threads (the reference's -t workers on one GPU): same caches"""
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=18, n=50021, seed=17, window=4, max_indegree=3)
    nbs = [pkg.two_hop_neighbors(edges, 18, v) for v in range(18)]
    engine.set_discrete(codes, card)
    want = {}
    for v in range(18):
        r = engine.score_variable(v, nbs[v], 7, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        want[v] = r.fetch()
        r.free()
    pool = pkg.EnginePool(0, 3)
    pool.set_discrete(codes, card)
    items = [(v, nbs[v]) for v in range(18)]
    for costs in (None, [float(bin(nb).count("1")) for _, nb in items]):
        got = pool.run(items, 7, pkg.BIC, flags=pkg.PRUNE_DOMINATED, fetch=True, costs=costs)
        assert sorted(got) == list(range(18))
        for v in range(18):
            assert np.array_equal(got[v][0], want[v][0]) and np.array_equal(got[v][1].view(np.uint32), want[v][1].view(np.uint32))
    scored = pool.run(items, 7, pkg.BIC, fetch=False)
    assert all(scored[v] > 0 for v in range(18))
    pool.close()


def test_randomised_parity_sweep():
    """tools/stress_bic.py: random shapes, arities (incl. constant columns), skeletons, parent limits, K1 modes and kernel
    budgets, BIC and fNML, against the oracle for ~10 s; 1854 cases of the same sweep passed during development (seeds 1, 2, 3, 7)"""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stress_bic.py"), "7", "10"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "stress OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_errors_are_loud(pkg, engine):
    with pytest.raises(pkg.UrlGpuError):
        engine.score_variable(99, 1, 1, pkg.BIC)
    codes = np.zeros((40, 100), dtype=np.uint8)
    engine.set_discrete(codes, [1] * 40)
    with pytest.raises(pkg.UrlGpuError, match="2\\^32 parent sets"):
        engine.score_variable(0, (1 << 40) - 1, 20, pkg.BIC)  # 39 candidates, sets of up to 20: beyond 32-bit ranks


def test_speculative_16bit_tables_and_their_fallback(pkg, orc):
    """cube path: tables of the deep layers are written with uint16 cells; a count that does not fit raises a flag and the
    variable is recomputed with 32-bit tables.  (a) skewed data whose modal configuration holds > 65535 records: the fallback
    runs and the cache is still exact; (b) 16-bit cells forced down to layer 1 on ordinary data: exact either way;
    (c) ordinary data at the default setting: no fallback."""
    from conftest import engine_with_env
    rng = np.random.default_rng(8)
    p, n = 12, 200_003
    skew = (rng.random((p, n)) < 0.04).astype(np.uint8)            # every column ~96 % zeros: the all-zero configuration is huge
    skew[:, :3] = np.array([[0, 1, 0]] * p, dtype=np.uint8)        # value 0 appears first in every column
    card = np.full(p, 2, dtype=np.int32)
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_LAYOUT": "dense"})
    eng.set_discrete(skew, card)
    eng.reset_stats()
    for v in (0, 11):
        _check_variable(pkg, orc, eng, skew, card, None, v, 10)
        _check_variable(pkg, orc, eng, skew, card, None, v, 10, flags=pkg.PRUNE_DOMINATED)
    assert eng.stats()["table16_fallbacks"] == 2   # once per variable: its later scorings go straight to 32-bit tables
    eng.close()
    codes, card2, edges, _ = pkg.datagen.discrete_bn(p=14, n=90001, seed=31, arities=(2, 3, 4), window=6, max_indegree=3)
    forced = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_TABLE16_MINLAYER": "1"})
    forced.set_discrete(codes, card2)
    for v, K in ((2, 9), (11, 8), (5, 10)):
        _check_variable(pkg, orc, forced, codes, card2, None, v, K)
    forced.close()
    plain = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube"})
    plain.set_discrete(codes, card2)
    plain.reset_stats()
    for v, K in ((2, 9), (7, 11)):
        _check_variable(pkg, orc, plain, codes, card2, None, v, K, flags=pkg.PRUNE_DOMINATED)
    assert plain.stats()["table16_fallbacks"] == 0
    off = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_TABLE16": "0"})
    off.set_discrete(codes, card2)
    _check_variable(pkg, orc, off, codes, card2, None, 2, 9)
    off.close()
    plain.close()
