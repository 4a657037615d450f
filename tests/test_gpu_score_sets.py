"""urlgpu_score_sets: a list of arbitrary (variable, parent set) pairs scored in one call.

Every entry must equal urlgpu_score_one on the same pair bit for bit, and through it the oracle (BIC and fNML bit-exact, BDeu
within one float32 ulp, cBIC within 1e-9 relative on the FP64 value) and the family caches.  The list path sends discrete
entries to the direct-counting tiers by table size (``bic_count_smem_kernel<ListSets>``, the global tier) in groups of one
child arity, and cBIC entries to ``cbic_sets_kernel`` in groups of one set size: the tests below put entries on every tier
edge, on every lane stride of the warp sweep, and on both sides of the shared-memory opt-in, in shuffled lists.
"""
import importlib
import os
import subprocess

import numpy as np
import pytest

from conftest import engine_with_env

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-9
LAM = 2.0
T0_CELLS = 12 * 1024              # tier 0 of the direct path (48 KB of shared memory)
BATCH_CELLS = 12 << 20            # the global tier's scratch batch, int32 cells


@pytest.fixture(scope="module")
def eng(pkg):
    e = pkg.Engine(0)
    yield e
    e.close()


def _bits(idx):
    return sum(1 << int(i) for i in idx)


def _u32(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def _ulps(a, b):
    a = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a)
    b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)


def _one_loop(eng, variables, masks, st, lam):
    out = [eng.score_one(int(v), int(m), st, lam) for v, m in zip(variables, masks)]
    return np.array([s for s, _ in out], dtype=np.float32), np.array([x for _, x in out], dtype=np.float64)


def _oracle(orc, pkg, codes, card, variables, masks, st, ess=1.0):
    """the oracle's score of every entry (the child's own bit removed), grouped by child"""
    variables = np.asarray(variables)
    out = np.zeros(len(variables), dtype=np.float32)
    for v in np.unique(variables):
        idx = np.nonzero(variables == v)[0]
        mv = np.array([int(masks[i]) & ~(1 << int(v)) for i in idx], dtype=np.uint64)
        if st == pkg.BIC:
            out[idx] = orc.bic_score_many(codes, card, int(v), mv)
        elif st == pkg.FNML:
            out[idx] = orc.fnml_score_many(codes, card, int(v), mv)
        else:
            out[idx] = orc.bdeu_score_many(codes, card, int(v), mv, ess=ess)
    return out


def _random_list(rng, p, n, kmax, child_bit_every=0):
    variables, masks = [], []
    for i in range(n):
        v = int(rng.integers(p))
        k = int(rng.integers(0, kmax + 1))
        others = [j for j in range(p) if j != v]
        m = _bits(rng.choice(others, size=k, replace=False))
        if child_bit_every and i % child_bit_every == 0:
            m |= 1 << v
        variables.append(v)
        masks.append(m)
    return variables, masks


# ------------------------------------------------------------------------------------------------ 1. equal to score_one
@pytest.fixture(scope="module")
def disc(pkg):
    codes, card, _, _ = pkg.datagen.discrete_bn(p=20, n=10_007, seed=5, arities=(2, 3, 4))
    rng = np.random.default_rng(7)
    c7 = rng.integers(0, 7, size=codes.shape[1]).astype(np.uint8)
    c7[:7] = np.arange(7)
    codes = np.vstack([codes, c7[None, :]])
    card = np.concatenate([card, [7]]).astype(np.int32)
    return codes, card


def test_equal_to_score_one_and_the_oracle(pkg, orc, eng, disc):
    """2 000 shuffled entries over all 21 variables (arities 2, 3, 4 and 7): empty sets, up to 8 parents, duplicates and masks
    naming the child.  Scores and values64 equal a score_one loop bit for bit; BIC and fNML bit-exact against the oracle,
    BDeu within one ulp"""
    codes, card = disc
    p = codes.shape[0]
    eng.set_discrete(codes, card)
    rng = np.random.default_rng(11)
    variables, masks = _random_list(rng, p, 1800, 8, child_bit_every=9)
    dup = rng.integers(0, 1800, size=200)
    variables += [variables[i] for i in dup]
    masks += [masks[i] for i in dup]
    variables += list(range(p))            # every child with the empty set
    masks += [0] * p
    perm = rng.permutation(len(variables))
    variables = [variables[i] for i in perm]
    masks = [masks[i] for i in perm]
    for st in (pkg.BIC, pkg.FNML, pkg.BDEU):
        lam = 1.0 if st == pkg.BDEU else 0.0
        s, x = eng.score_sets(variables, masks, st, lam)
        s1, x1 = _one_loop(eng, variables, masks, st, lam)
        assert np.array_equal(_u32(s), _u32(s1)), st
        assert np.array_equal(x.view(np.uint64), x1.view(np.uint64)), st
        want = _oracle(orc, pkg, codes, card, variables, masks, st)
        if st == pkg.BDEU:
            assert _ulps(s, want).max() <= 1
        else:
            assert np.array_equal(_u32(s), _u32(want)), st


# ------------------------------------------------------------------------------------------------ 2. tier edges
def _tier1_cells():
    import torch
    return (torch.cuda.get_device_properties(0).shared_memory_per_block_optin - 2048) // 4


def _split(cells, limit=64):
    """arities (each <= limit) whose product is `cells`: its prime factors packed first-fit, largest first"""
    f, x, q = [], cells, 2
    while q * q <= x:
        while x % q == 0:
            f.append(q)
            x //= q
        q += 1
    if x > 1:
        f.append(x)
    bins = []
    for q in sorted(f, reverse=True):
        for i, b in enumerate(bins):
            if b * q <= limit:
                bins[i] = b * q
                break
        else:
            bins.append(q)
    return sorted(bins, reverse=True)


def test_tier_edges_in_one_list(pkg, orc, eng):
    """one table exactly on each tier bound and one just above it (tier 0: 3 * 4^6 and 4^7; tier 1: the opt-in less 2 KB read
    from the device, and the next product above), and a 4 * 4^11 = 16.8M-cell table above the global tier's 12M-cell batch,
    each mixed into small sets: every output at its input index, bit-exact against the oracle (BIC, fNML)"""
    t1 = _tier1_cells()
    t1_par = _split(t1 // 4)
    assert 4 * int(np.prod(t1_par)) == t1
    card = [3, 4] + [4] * 11 + t1_par + [t1_par[0] + 1]
    a4 = list(range(2, 13))
    tp = list(range(13, 13 + len(t1_par)))
    above = [len(card) - 1] + tp[1:]
    rng = np.random.default_rng(3)
    n = 30_011
    codes = np.zeros((len(card), n), dtype=np.uint8)
    for i, r in enumerate(card):
        col = rng.integers(0, r, size=n)
        if i >= 2:
            col = np.where(rng.random(n) < 0.4, (codes[i - 1].astype(np.int64) * 7 + codes[i - 2]) % r, col)
        codes[i] = col
    edges = [(0, a4[:6], T0_CELLS), (1, a4[:6], 4 * 4 ** 6), (1, tp, t1), (1, above, 4 * (t1_par[0] + 1) * int(np.prod(t1_par[1:]))),
             (1, a4, 4 * 4 ** 11)]
    assert 4 * 4 ** 11 > BATCH_CELLS
    eng.set_discrete(codes, card)
    variables, masks = _random_list(rng, 13, 60, 3)
    for v, par, cells in edges:
        assert int(card[v]) * int(np.prod([card[i] for i in par])) == cells
        at = int(rng.integers(len(variables) + 1))
        variables.insert(at, v)
        masks.insert(at, _bits(par))
    for st in (pkg.BIC, pkg.FNML):
        s, x = eng.score_sets(variables, masks, st)
        want = _oracle(orc, pkg, codes, card, variables, masks, st)
        assert np.array_equal(_u32(s), _u32(want)), st
        s1, x1 = _one_loop(eng, variables, masks, st, 0.0)
        assert np.array_equal(x.view(np.uint64), x1.view(np.uint64)), st


# ------------------------------------------------------------------------------------------------ 3. wide masks
def test_wide_masks(pkg, eng):
    """150 variables (three mask words): parents above bits 64 and 128, children in every word, equal to score_one"""
    codes, card, _, _ = pkg.datagen.discrete_bn(p=150, n=5003, seed=15, arities=(2, 3))
    eng.set_discrete(codes, card)
    rng = np.random.default_rng(15)
    variables, masks = _random_list(rng, 150, 300, 5)
    variables += [0, 70, 149, 130, 64]
    masks += [_bits([63, 64, 127, 128]), _bits([1, 129, 149]), _bits([0, 64, 128]), _bits([65, 128, 130]), _bits([64])]
    for st in (pkg.BIC, pkg.BDEU):
        lam = 1.0 if st == pkg.BDEU else 0.0
        s, x = eng.score_sets(variables, masks, st, lam)
        s1, x1 = _one_loop(eng, variables, masks, st, lam)
        assert np.array_equal(_u32(s), _u32(s1)) and np.array_equal(x.view(np.uint64), x1.view(np.uint64)), st
    words = np.zeros((len(masks), 3), dtype=np.uint64)       # the array form of the same list
    for i, m in enumerate(masks):
        words[i] = pkg.mask_to_words(m, 3)
    s2, _ = eng.score_sets(np.array(variables), words, pkg.BDEU, 1.0)
    assert np.array_equal(_u32(s2), _u32(s))


# ------------------------------------------------------------------------------------------------ 4. cBIC
def _sub_residual(orc, x, v, members, lam=LAM):
    """the oracle's the_score of (v, members) on the relabelled sub-problem of those columns (at most 63 parents)"""
    sub = sorted(list(members) + [v])
    zs = orc.standardise(x[sub])
    return orc.cbic_residual(zs, sub.index(v), sum(1 << sub.index(i) for i in members), lam)


def _gram_score(orc, g, n, v, members, lam=LAM):
    """the oracle's the_score of (v, members) from the Gram g, on the relabelled sub-Gram of those columns: the oracle reads a
    parent set as one 64-bit mask, so with more than 64 variables the columns are renumbered first (at most 63 parents)"""
    sub = sorted(list(members) + [v])
    return orc.cbic_gram(np.ascontiguousarray(g[np.ix_(sub, sub)]), n, sub.index(v), sum(1 << sub.index(i) for i in members), lam)


def _lstsq_the_score(z, v, members, lam=LAM):
    n = z.shape[1]
    a = z[list(members)].T
    coef = np.linalg.lstsq(a, z[v], rcond=None)[0]
    r = z[v] - a @ coef
    return n * np.log(float(r @ r) / n) + lam * len(members) * np.log(n)


def test_cbic_set_sizes_pivot_guard_and_gram_refresh(pkg, orc, eng):
    """k = 0, 1, 32, 33, 64, 65 and 200 in one list (the empty set is -0.0f), bit-equal to score_one, within 1e-9 of the oracle
    (numpy least squares above 63 parents); a duplicated column takes the pivot guard as score_one does; after set_gram the next
    list reads the new Gram"""
    p, n = 202, 3000
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=8)
    x[201] = x[5]                      # a duplicated column
    z = orc.standardise(x)
    eng.set_continuous(x)
    rng = np.random.default_rng(4)
    variables, members = [], []
    for k in (0, 1, 32, 33, 64, 65, 200, 3, 0, 33):
        v = int(rng.choice([i for i in range(201) if i != 5]))
        others = [i for i in range(201) if i != v]           # column 201 only where asked for below
        variables.append(v)
        members.append(sorted(int(i) for i in rng.choice(others, size=k, replace=False)))
    variables += [7, 9]
    members += [[5, 201], [1, 5, 100, 201]]    # both copies of the column
    masks = [_bits(m) for m in members]
    s, ts = eng.score_sets(variables, masks, pkg.CBIC, LAM)
    s1, ts1 = _one_loop(eng, variables, masks, pkg.CBIC, LAM)
    assert np.array_equal(_u32(s), _u32(s1)) and np.array_equal(ts.view(np.uint64), ts1.view(np.uint64))
    assert _u32(s[0]) == 0x80000000 and ts[0] == 0.0
    for i, (v, mem) in enumerate(zip(variables, members)):
        if not mem or 201 in mem:
            continue
        ref = _sub_residual(orc, x, v, mem) if len(mem) <= 63 else _lstsq_the_score(z, v, mem)
        assert abs(ts[i] - ref) <= TOL * max(1.0, abs(ref)), (i, len(mem), ts[i], ref)
        assert _u32(s[i]) == _u32(-np.float32(ts[i]))
    # a different Gram through set_gram: the list follows it (oracle from the Gram itself), and so does the family cache
    x2, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=9)
    g2 = orc.gram(orc.standardise(x2))
    vs, mem2 = [3, 60, 40], [[1, 2], [0, 33, 63, 150, 201], list(range(10))]
    ms = [_bits(m) for m in mem2]
    before = eng.score_sets(vs, ms, pkg.CBIC, LAM)[1]
    eng.set_gram(g2, n)
    s2, ts2 = eng.score_sets(vs, ms, pkg.CBIC, LAM)
    for i in range(3):
        ref = _gram_score(orc, g2, n, vs[i], mem2[i])
        assert abs(ts2[i] - ref) <= TOL * max(1.0, abs(ref)) and ts2[i] != before[i]
    res = eng.score_variable(3, _bits([1, 2, 3]), 2, pkg.CBIC, lam=LAM, flags=pkg.CBIC_NO_ACCEPT)
    m, sc = res.fetch()
    res.free()
    assert pkg.words_to_mask(m[-1]) == ms[0] and _u32(sc[-1]) == _u32(s2[0])


# ------------------------------------------------------------------------------------------------ 5. family caches
@pytest.mark.parametrize("layout", ["dense", "rank"])
def test_equal_to_the_family_caches(pkg, orc, disc, layout):
    """the raw scores of score_range (BIC; cBIC: the_score, i.e. -score) and the cBIC cache without acceptance equal
    score_sets over the same masks, bit for bit, in both cache layouts"""
    codes, card = disc
    p = codes.shape[0]
    e = engine_with_env(pkg, {"URLGPU_LAYOUT": layout})
    e.set_discrete(codes, card)
    v, nb, K = 20, (1 << 20) - 1 - (1 << 3), 3
    total = e.family_size(v, nb, K, pkg.BIC)
    om = orc.enumerate_sets(v, nb, p, K)
    om = om[orc.canonical_order(om)]
    assert total == len(om)
    raw = e.score_range(v, nb, K, pkg.BIC, 0, total)
    s, _ = e.score_sets([v] * total, [int(m) for m in om], pkg.BIC)
    assert np.array_equal(_u32(raw), _u32(s))
    x, _ = pkg.datagen.linear_gaussian_sem(p=24, n=4000, seed=2)
    e.set_continuous(x)
    v, nb, K = 11, (1 << 24) - 1, 4
    res = e.score_variable(v, nb, K, pkg.CBIC, lam=LAM, flags=pkg.CBIC_NO_ACCEPT)
    m, sc = res.fetch()
    res.free()
    s, _ = e.score_sets(np.full(len(m), v), m, pkg.CBIC, LAM)
    assert len(m) > 1000 and np.array_equal(_u32(sc), _u32(s))
    om = orc.enumerate_sets(v, nb, 24, K)
    om = om[orc.canonical_order(om)]
    total = e.family_size(v, nb, K, pkg.CBIC)
    raw = e.score_range(v, nb, K, pkg.CBIC, 0, total, lam=LAM)
    s, _ = e.score_sets([v] * len(om), [int(q) for q in om], pkg.CBIC, LAM)
    assert total == len(om) and np.array_equal(_u32(raw), _u32(-s))
    e.close()


# ------------------------------------------------------------------------------------------------ 6. launches
def test_launches_do_not_grow_with_the_list(pkg, eng, disc):
    """1 000 and 20 000 entries drawn from the same shapes (every child arity and, for cBIC, every set size in both lists)
    take the same number of kernel launches"""
    codes, card = disc
    p = codes.shape[0]
    eng.set_discrete(codes, card)
    rng = np.random.default_rng(6)
    counts = {}
    for n in (1000, 20_000):
        variables, masks = _random_list(rng, p, n, 4)
        variables[:p] = range(p)
        eng.reset_stats()
        eng.score_sets(variables, masks, pkg.BIC)
        counts[("bic", n)] = eng.stats()["launches_total"]
    x, _ = pkg.datagen.linear_gaussian_sem(p=30, n=2000, seed=6)
    eng.set_continuous(x)
    for n in (1000, 20_000):
        variables, masks = _random_list(rng, 30, n, 6)
        masks[:7] = [_bits(range(1, 1 + k)) for k in range(7)]
        variables[:7] = [0] * 7
        eng.reset_stats()
        eng.score_sets(variables, masks, pkg.CBIC, LAM)
        counts[("cbic", n)] = eng.stats()["launches_total"]
    assert counts[("bic", 1000)] == counts[("bic", 20_000)] > 0, counts
    assert counts[("cbic", 1000)] == counts[("cbic", 20_000)] == 7, counts


# ------------------------------------------------------------------------------------------------ 7. interleaving
def test_interleaving_with_families_and_score_one(pkg, orc, eng, disc):
    """a BIC cache prefetched but not fetched, an fNML list, then the fetch: the BIC entries are unchanged.  A BDeu list followed
    by a BIC score_one gives BIC"""
    codes, card = disc
    p = codes.shape[0]
    eng.set_discrete(codes, card)
    v, nb, K = 4, (1 << p) - 1, 3
    want_m, want_s = eng.score_variable(v, nb, K, pkg.BIC).fetch()
    res = eng.score_variable(v, nb, K, pkg.BIC).prefetch()
    rng = np.random.default_rng(8)
    variables, masks = _random_list(rng, p, 500, 5)
    s, _ = eng.score_sets(variables, masks, pkg.FNML)
    m, sc = res.fetch()
    res.free()
    assert np.array_equal(m, want_m) and np.array_equal(_u32(sc), _u32(want_s))
    assert np.array_equal(_u32(s), _u32(_oracle(orc, pkg, codes, card, variables, masks, pkg.FNML)))
    eng.score_sets(variables, masks, pkg.BDEU, 1.0)
    b, _ = eng.score_one(6, _bits([1, 2]), pkg.BIC)
    assert _u32(b) == _u32(orc.bic_score(codes, card, 6, _bits([1, 2]))[0])


# ------------------------------------------------------------------------------------------------ 8. refusals
def test_refusals_name_the_entry_and_leave_the_context_usable(pkg, orc):
    e = pkg.Engine(0)
    s, x = e.score_sets([], [], pkg.BIC)                     # nothing to do: succeeds even before any data is installed
    assert len(s) == 0 and len(x) == 0
    with pytest.raises(pkg.UrlGpuError, match="need urlgpu_set_discrete first"):
        e.score_sets([0], [0], pkg.BIC)
    p, n = 40, 1000
    card = [4] * p
    codes = np.random.default_rng(1).integers(0, 4, size=(p, n)).astype(np.uint8)
    e.set_discrete(codes, card)
    ok_v, ok_m = [3, 5], [_bits([1, 2]), 0]

    def check_ok():
        got, _ = e.score_sets(ok_v, ok_m, pkg.BIC)
        assert np.array_equal(_u32(got), _u32(_oracle(orc, pkg, codes, card, ok_v, ok_m, pkg.BIC)))

    cases = [
        ([3, 5, 0], ok_m + [_bits(range(1, 32))], pkg.BIC, "entry 2: more than 30 parents"),
        ([3, 0, 5], [ok_m[0], _bits(range(1, 16)), 0], pkg.BIC, "entry 1: contingency table exceeds 2\\^30 cells"),
        ([3, 40], ok_m, pkg.BIC, "entry 1: variable out of range"),
        ([3, -1], ok_m, pkg.FNML, "entry 1: variable out of range"),
        ([3, 5, 6], ok_m + [1 << 40], pkg.BIC, "entry 2: mask names a variable >= p"),
        (ok_v, ok_m, 7, "unknown score type"),
        (ok_v, ok_m, pkg.BDEU, "equivalent sample size"),
    ]
    for variables, masks, st, msg in cases:
        with pytest.raises(pkg.UrlGpuError, match=msg):
            e.score_sets(variables, masks, st, 0.0)
        check_ok()
    # cBIC: 201 parents, and one mask word for 202 variables
    g = np.eye(202) * 999.0
    g[0, 1] = g[1, 0] = 100.0
    e.set_gram(g, 1000)
    with pytest.raises(pkg.UrlGpuError, match="entry 1: more than 200 parents"):
        e.score_sets([0, 201], [_bits([1]), (1 << 201) - 1], pkg.CBIC, LAM)
    with pytest.raises(pkg.UrlGpuError, match="mask_words too small"):
        e.score_sets([0], np.zeros((1, 1), dtype=np.uint64), pkg.CBIC, LAM)
    s, ts = e.score_sets([0, 201], [_bits([1]), _bits(range(200))], pkg.CBIC, LAM)
    assert abs(ts[0] - _gram_score(orc, g, 1000, 0, [1])) <= TOL * abs(ts[0])
    check_ok()
    e.close()


# ------------------------------------------------------------------------------------------------ 9. a learned DAG, rescored
def test_learned_dag_rescored(pkg, orc, eng, tmp_path):
    """hepatitis: `score` -> .pss -> A*; score_sets over the 20 (variable, parents) pairs of the optimal DAG equals the
    score_variable cache entries bit for bit, and minus their sum is the A* cost"""
    S = importlib.import_module("urlearning-cpp_b200.search")
    inp = os.path.join(ROOT, "tests", "data", "hepatitis.clean.csv")
    pss = str(tmp_path / "hep.pss")
    subprocess.check_call([os.path.join(ROOT, "urlearning-cpp_b200", "score"), inp, pss, "-s", "-f", "BIC", "--quiet"], stdout=subprocess.DEVNULL)
    cost, parents, _, _ = S.ScoreCache(pss).astar("list")
    t = orc.Table(inp, has_header=True)
    codes = t.codes()
    eng.set_discrete(codes, t.card)
    K = pkg.effective_max_parents(0, t.p, t.n, True)
    s, _ = eng.score_sets(list(range(t.p)), [int(m) for m in parents], pkg.BIC)
    for v in range(t.p):
        m, sc = eng.score_variable(v, pkg.two_hop_neighbors(None, t.p, v), K, pkg.BIC).fetch()
        hit = np.nonzero(m[:, 0] == np.uint64(parents[v]))[0]
        assert len(hit) == 1 and _u32(sc[hit[0]]) == _u32(s[v]), v
    total = -float(np.sum(s.astype(np.float64)))
    assert abs(total - cost) <= 1e-5 * abs(cost), (total, cost)
