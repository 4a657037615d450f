"""GPU parity of the continuous (cBIC) path at the limits its API admits, not only at comfortable shapes.

Each test names the kernel or route it reaches and checks it against the CPU oracle (tests/oracle_lib.py) or a plain
numpy reference, at the project's tolerances: the FP64 the_score within 1e-9 relative, the float32 score within one ulp,
``score_one`` bit-equal to the cache entry of the same set, both cache layouts bit-equal, acceptance and prune decisions
exact given the engine's own float32 scores, and the Gram within 1e-12 n of the long-double Gram of the oracle.

- K2 (``standardise_kernel``, ``gram_partial_kernel``, ``gram_combine_kernel``): partial 64-wide tiles, several tile
  pairs, fewer records than one 32-record chunk, row slices between the clamps with a short last slice, the device-input
  routes and row shards;
- ``cbic_one_kernel`` (``urlgpu_score_one``) up to its 200-parent limit: the second stride of the lane loop (k >= 33) and
  the shared-memory opt-in (k >= 110);
- ``rank_cbic_kernel<0>`` at layers 15 and 16, 16-parent ranges over 31 candidates, 255 candidates, and the refusals;
- ``accept_literal_kernel`` at 12 parents and at 62 candidates;
- the standalone ``urlgpu_prune`` with masks over up to 30 variables (several segment high bits).
"""
from math import comb

import numpy as np
import pytest

from conftest import engine_with_env

pytestmark = pytest.mark.gpu
TOL = 1e-9
LAM = 2.0


def ulp_diff(a, b):
    a = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a)
    b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)


def bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def colex_unrank(c, l, r):
    """rank r among the l-subsets of range(c) in colex order -> ascending positions (the engine's rank-space order)"""
    e = [0] * l
    hi = c - 1
    for i in range(l, 0, -1):
        b = hi
        while comb(b, i) > r:
            b -= 1
        e[i - 1] = b
        r -= comb(b, i)
        hi = b - 1
    return e


def family_set(c, K, idx):
    """index of the canonical (|S|, colex) numbering of all subsets of range(c) with at most K members -> positions"""
    for l in range(K + 1):
        if idx < comb(c, l):
            return colex_unrank(c, l, idx)
        idx -= comb(c, l)
    raise IndexError(idx)


def sub_residual(orc, x, v, members, lam=LAM):
    """the oracle's the_score of (v, members) on the relabelled sub-problem of those columns (any p, masks of <= 64 bits)"""
    sub = sorted(list(members) + [v])
    zs = orc.standardise(x[sub])
    return orc.cbic_residual(zs, sub.index(v), sum(1 << sub.index(i) for i in members), lam)


def lstsq_the_score(z, v, members, lam=LAM):
    """plain numpy reference of the_score for any number of parents: OLS without intercept on the standardised columns,
    n ln(RSS / n) + lam k ln(n) (oracle.cpp, orc_cbic_the_score_residual)"""
    n = z.shape[1]
    a = z[list(members)].T
    y = z[v]
    coef = np.linalg.lstsq(a, y, rcond=None)[0]
    r = y - a @ coef
    rss = float(r @ r)
    return n * np.log(rss / n) + lam * np.log(n) * len(members)


@pytest.fixture(scope="module")
def eng(pkg):
    e = pkg.Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def layouts(pkg):
    d = engine_with_env(pkg, {"URLGPU_LAYOUT": "dense"})
    r = engine_with_env(pkg, {"URLGPU_LAYOUT": "rank"})
    yield {"dense": d, "rank": r}
    d.close()
    r.close()


# ------------------------------------------------------------------------------------------------ 1. K2 shapes and routes

def gram_data(p, n, seed):
    """normal columns on a 2^-20 grid (so that the mean of two records is exact), every third column offset by 1e3 .. 1e6"""
    rng = np.random.default_rng(seed)
    x = np.round(rng.standard_normal((p, n)) * 2.0 ** 20) / 2.0 ** 20
    for j in range(0, p, 3):
        x[j] += 10.0 ** (3 + (j // 3) % 4)
    return x


GRAM_SHAPES = sorted({(p, n) for p in (1, 2, 31, 63, 64, 65, 127, 128, 129, 200) for n in (2, 33, 2049)}
                     | {(p, n) for p in (1, 65, 129) for n in (2, 3, 31, 32, 33, 1025, 2049)} | {(129, 300001)})


@pytest.mark.parametrize("p,n", GRAM_SHAPES)
def test_gram_shapes_against_long_double(pkg, orc, eng, p, n):
    """standardise_kernel + gram_partial_kernel + gram_combine_kernel: partial tiles (p = 65, 129, 200), several tile pairs,
    n below one chunk, and at (129, 300001) slices of 1536 records with a short last one"""
    x = gram_data(p, n, seed=p * 7 + n)
    eng.set_continuous(x)
    g = eng.gram()
    ref = orc.gram(orc.standardise(x))
    assert np.array_equal(g, g.T)
    assert np.allclose(np.diag(g), n - 1.0, rtol=1e-12, atol=0)
    assert np.max(np.abs(g - ref)) <= 1e-12 * n
    if n == 2:
        assert np.max(np.abs(np.abs(g) - 1.0)) <= 1e-15


def shard_gram(pkg, x, cuts, device=False):
    """the row-sharded protocol of include/urlgpu.h on one GPU: one context per shard, moments and partial Grams summed in
    shard order -> (Gram, contexts)"""
    import torch
    n = x.shape[1]
    engs = [pkg.Engine(0) for _ in cuts[:-1]]
    keep = []
    for e, a, b in zip(engs, cuts[:-1], cuts[1:]):
        if device:
            t = torch.from_numpy(np.ascontiguousarray(x[:, a:b])).cuda()
            keep.append(t)
            torch.cuda.synchronize()
            e.shard_begin(t.data_ptr(), b - a, x.shape[0])
        else:
            e.shard_begin(x[:, a:b].copy())
    s1 = engs[0].shard_moments(None)[0]
    for e in engs[1:]:
        s1 = s1 + e.shard_moments(None)[0]
    mean = s1 / n
    parts = [e.shard_moments(mean) for e in engs]
    S1, S2 = parts[0]
    for a, b in parts[1:]:
        S1, S2 = S1 + a, S2 + b
    dev = np.sqrt((S2 - S1 * S1 / n) / (n - 1.0))
    for e in engs:
        e.shard_finish(mean, dev, n)
    g = engs[0].gram()
    for e in engs[1:]:
        g = g + e.gram()
    del keep
    return g, engs


def test_gram_routes_are_bit_identical(pkg, orc):
    """one data set through every route into K2: two contexts, set_continuous_device (a torch CUDA tensor), and the one-shard
    protocol from a host array and from a device pointer (standardised into the cached z buffer) give the same bits"""
    import torch
    p, n = 129, 40001
    x = gram_data(p, n, seed=11)
    a, b, c = pkg.Engine(0), pkg.Engine(0), pkg.Engine(0)
    a.set_continuous(x)
    b.set_continuous(x)
    ga = a.gram()
    assert np.array_equal(ga, b.gram())
    xt = torch.from_numpy(x).cuda()
    torch.cuda.synchronize()
    c.set_continuous_device(xt.data_ptr(), n, p)
    assert np.array_equal(ga, c.gram())
    assert np.max(np.abs(ga - orc.gram(orc.standardise(x)))) <= 1e-12 * n
    for device in (False, True):
        g1, engs = shard_gram(pkg, x, [0, n], device=device)
        assert np.array_equal(ga, g1), f"one-shard protocol (device input: {device}) differs from set_continuous"
        for e in engs:
            e.close()
    # the contexts still score: the device route left a usable Gram behind
    s_a = a.score_one(5, (1 << 40) | (1 << 64) | (1 << 100), pkg.CBIC, LAM)
    s_c = c.score_one(5, (1 << 40) | (1 << 64) | (1 << 100), pkg.CBIC, LAM)
    assert bits(s_a[0]) == bits(s_c[0]) and s_a[1] == s_c[1]
    for e in (a, b, c):
        e.close()


def test_row_shards_agree_and_a_fixed_cut_is_bit_identical(pkg, orc):
    """2 and 3 row shards over cuts that are not multiples of 32 agree with the one-shard Gram within 1e-12 n; the bits
    differ (the cut moves the slice boundaries and the moment sums), but the same cut always gives the same bits"""
    p, n = 70, 50003
    x = gram_data(p, n, seed=5)
    ref = orc.gram(orc.standardise(x))
    g1, engs = shard_gram(pkg, x, [0, n])
    for e in engs:
        e.close()
    differs = {}
    for cuts in ([0, 16411, n], [0, 9001, 30017, n]):
        g, engs = shard_gram(pkg, x, cuts)
        for e in engs:
            e.close()
        assert np.array_equal(g, g.T)
        assert np.max(np.abs(g - g1)) <= 1e-12 * n
        assert np.max(np.abs(g - ref)) <= 1e-12 * n
        again, engs = shard_gram(pkg, x, cuts, device=True)
        for e in engs:
            e.close()
        assert np.array_equal(g, again), f"shard cut {cuts}: two runs differ"
        differs[len(cuts) - 1] = int(np.sum(g != g1))
    print(f"entries whose bits differ from the one-shard Gram: {differs} of {p * p}")


# ------------------------------------------------------------------------------------------------ 2. score_one up to 200 parents

ONE_K = (15, 16, 17, 31, 32, 33, 63, 64, 65, 109, 110, 111, 150, 199, 200)


@pytest.fixture(scope="module")
def wide(pkg, orc):
    p, n = 201, 6000
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=21, mean_indegree=2.0)
    return x, orc.standardise(x)


def one_parents(p, v, k, seed):
    """k parents of v among the other p - 1 variables, always including the word edges 63, 64, 127, 128 when k allows"""
    others = [i for i in range(p) if i != v]
    edges = [i for i in (63, 64, 127, 128) if i != v][: k]
    rest = [i for i in others if i not in edges]
    rng = np.random.default_rng(seed)
    pick = edges + [int(i) for i in rng.choice(rest, size=k - len(edges), replace=False)]
    return sorted(pick)


@pytest.mark.parametrize("v", [0, 200])
def test_score_one_up_to_200_parents(pkg, orc, eng, wide, v):
    """cbic_one_kernel with k = 15 .. 200 parents over 4-word masks: k >= 33 runs the second stride of the lane loop, k >= 110
    needs the shared-memory opt-in.  k <= 63 against the oracle on the relabelled sub-problem; above, against numpy's
    least squares, which is first held to the oracle on the k <= 63 sets"""
    x, z = wide
    p, n = x.shape
    eng.set_continuous(x)
    for k in ONE_K:
        members = one_parents(p, v, k, seed=1000 * v + k)
        mask = sum(1 << i for i in members)
        s, ts64 = eng.score_one(v, mask, pkg.CBIC, LAM)
        ref = lstsq_the_score(z, v, members)
        if k <= 63:
            r = sub_residual(orc, x, v, members)
            assert abs(ref - r) <= TOL * max(1.0, abs(r)), f"numpy reference off the oracle at k = {k}"
            ref = r
        assert abs(ts64 - ref) <= TOL * max(1.0, abs(ref)), (k, ts64, ref)
        assert ulp_diff(s, np.float32(-np.float32(ref))) <= 1, k
        assert bits(s) == bits(-np.float32(ts64))
        if k in (15, 16):   # the same set as the only k-set of its own family, through rank_cbic_kernel<0>: the same bits
            nb = mask | (1 << v)
            total = eng.family_size(v, nb, k, pkg.CBIC)
            raw = eng.score_range(v, nb, k, pkg.CBIC, total - 1, 1, lam=LAM)
            assert bits(raw[0]) == bits(-s)
    # a small set after the largest one: still bit-equal to its cache entry
    members = one_parents(p, v, 3, seed=7)
    mask = sum(1 << i for i in members)
    s, ts64 = eng.score_one(v, mask, pkg.CBIC, LAM)
    res = eng.score_variable(v, mask | (1 << v), 3, pkg.CBIC, lam=LAM, flags=pkg.CBIC_NO_ACCEPT)
    m, sc = res.fetch()
    res.free()
    assert pkg.words_to_mask(m[-1]) == mask and bits(sc[-1]) == bits(s)
    r = sub_residual(orc, x, v, members)
    assert abs(ts64 - r) <= TOL * max(1.0, abs(r))


def test_score_one_refuses_201_parents(pkg, orc, eng):
    p, n = 202, 3000
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=8)
    eng.set_continuous(x)
    with pytest.raises(pkg.UrlGpuError, match="more than 200 parents"):
        eng.score_one(201, (1 << 201) - 1, pkg.CBIC, LAM)
    members = [3, 64, 150, 200]
    s, ts64 = eng.score_one(201, sum(1 << i for i in members), pkg.CBIC, LAM)
    r = sub_residual(orc, x, 201, members)
    assert abs(ts64 - r) <= TOL * max(1.0, abs(r)) and ulp_diff(s, np.float32(-np.float32(r))) <= 1


# ------------------------------------------------------------------------------------------------ 3. rank-space sweeps

def no_accept(e, pkg, v, nb, K, flags=None):
    r = e.score_variable(v, nb, K, pkg.CBIC, lam=LAM, flags=pkg.CBIC_NO_ACCEPT if flags is None else flags)
    out = r.fetch()
    r.free()
    return out


@pytest.mark.parametrize("c,K", [(16, 15), (16, 16), (20, 15), (20, 16)])
def test_layers_15_and_16_layouts_agree(pkg, layouts, c, K):
    """rank_cbic_kernel<0> at layers 15 and 16 (URLGPU_LAYOUT=rank) against the dense DFS (URLGPU_LAYOUT=dense): the same
    cache bit for bit, under CBIC_NO_ACCEPT, the default acceptance and PRUNE_DOMINATED"""
    p = c + 1
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=3000, seed=c + K)
    for e in layouts.values():
        e.set_continuous(x)
    v = c // 2
    nb = (1 << p) - 1
    for flags in (pkg.CBIC_NO_ACCEPT, 0, pkg.PRUNE_DOMINATED):
        (md, sd), (mr, sr) = (no_accept(layouts[k], pkg, v, nb, K, flags) for k in ("dense", "rank"))
        if flags == pkg.CBIC_NO_ACCEPT:
            assert len(sr) == sum(comb(c, l) for l in range(K + 1))
        assert np.array_equal(md, mr) and np.array_equal(bits(sd), bits(sr)), flags


def test_layers_13_to_16_against_oracle_and_score_one(pkg, orc, layouts):
    """every set of layers 13 .. 16 at c = 16 (697 sets): the rank cache within one ulp of the oracle, score_one within 1e-9
    and bit-equal to the cache"""
    p, n, K = 17, 3000, 16
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=44)
    z = orc.standardise(x)
    e = layouts["rank"]
    e.set_continuous(x)
    for v in (0, 9):
        m, neg = no_accept(e, pkg, v, (1 << p) - 1, K)
        masks = m[:, 0]
        top = np.array([bin(int(q)).count("1") >= 13 for q in masks])
        assert top.sum() == 697
        for q, s_cache in zip(masks[top], neg[top]):
            r = orc.cbic_residual(z, v, int(q), LAM)
            assert ulp_diff(-s_cache, np.float32(r)) <= 1
            s, ts64 = e.score_one(v, int(q), pkg.CBIC, LAM)
            assert abs(ts64 - r) <= TOL * max(1.0, abs(r))
            assert bits(s) == bits(s_cache)


def test_17_parents_under_rank_policy_go_dense(pkg, layouts):
    """K = 17 at c = 18: URLGPU_LAYOUT=rank hands the family to the dense layout (the per-set sweeps hold 16 parents), and
    the result is the dense engine's"""
    p = 19
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=2500, seed=19)
    for e in layouts.values():
        e.set_continuous(x)
    for flags in (pkg.CBIC_NO_ACCEPT, 0, pkg.PRUNE_DOMINATED):
        (md, sd), (mr, sr) = (no_accept(layouts[k], pkg, 4, (1 << p) - 1, 17, flags) for k in ("dense", "rank"))
        assert np.array_equal(md, mr) and np.array_equal(bits(sd), bits(sr)), flags


def test_16_parents_over_31_candidates_by_range(pkg, orc, eng):
    """c = 31, K = 16: 1 374 282 019 sets, layer 16 starting at 2^30.  Ranges (counts not multiples of kRankRun = 4) at the
    start of layer 16, across layers 15 / 16 and at the end of the family, against the oracle and score_one"""
    p, n, K = 32, 2000, 16
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=31)
    eng.set_continuous(x)
    z = orc.standardise(x)
    v = 0
    nb = (1 << p) - 1
    total = eng.family_size(v, nb, K, pkg.CBIC)
    assert total == sum(comb(31, l) for l in range(K + 1)) == 1374282019
    assert sum(comb(31, l) for l in range(K)) == 1 << 30
    cand = list(range(1, p))
    for first, count in ((1 << 30, 301), ((1 << 30) - 203, 406), (total - 333, 333)):
        raw = eng.score_range(v, nb, K, pkg.CBIC, first, count, lam=LAM)
        for i in range(count):
            members = [cand[e] for e in family_set(31, K, first + i)]
            mask = sum(1 << q for q in members)
            r = orc.cbic_residual(z, v, mask, LAM)
            assert ulp_diff(raw[i], np.float32(r)) <= 1, (first + i, members)
            s, ts64 = eng.score_one(v, mask, pkg.CBIC, LAM)
            assert abs(ts64 - r) <= TOL * max(1.0, abs(r))
            assert bits(-s) == bits(raw[i])


def test_more_than_16_parents_refusals(pkg, orc, eng):
    """K = 17 over 31 candidates (score_variable, score_range) and over 18 candidates (score_range, score_part's range
    fallback) is refused with a message true for that family; the context scores correctly afterwards"""
    p = 32
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=2000, seed=31)
    eng.set_continuous(x)
    nb = (1 << p) - 1
    before = eng.score_range(0, nb, 16, pkg.CBIC, 1 << 30, 9, lam=LAM)
    with pytest.raises(pkg.UrlGpuError, match="at most 16 parents") as ex:
        eng.score_variable(0, nb, 17, pkg.CBIC, lam=LAM)
    assert "more than 30 candidates" in str(ex.value)
    with pytest.raises(pkg.UrlGpuError, match="at most 16 parents"):
        eng.score_range(0, nb, 17, pkg.CBIC, 1000, 10, lam=LAM)
    assert np.array_equal(bits(eng.score_range(0, nb, 16, pkg.CBIC, 1 << 30, 9, lam=LAM)), bits(before))
    # c = 18 <= 30: score_variable scores this family (dense), so the range routes must not blame the candidate count
    nb18 = (1 << 19) - 1
    for call in (lambda: eng.score_range(2, nb18, 17, pkg.CBIC, 5, 100, lam=LAM),
                 lambda: eng.score_part(2, nb18, 17, pkg.CBIC, 1, 3, lam=LAM)):
        with pytest.raises(pkg.UrlGpuError, match="at most 16 parents") as ex:
            call()
        assert "more than 30 candidates" not in str(ex.value)
    m, neg = no_accept(eng, pkg, 2, nb18, 17)
    assert len(m) == sum(comb(18, l) for l in range(18))
    z = orc.standardise(x)
    for i in (0, 1, 5000, len(m) - 1):
        r = orc.cbic_residual(z, 2, int(m[i, 0]), LAM)
        assert ulp_diff(-neg[i], np.float32(r)) <= 1


def test_255_candidates(pkg, orc, eng):
    """p = 256, v = 0, K = 2: 32 641 sets with 4-word masks, for cBIC and BIC.  The canonical (|S|, colex) order of the
    cache, sampled sets against the oracle on relabelled sub-problems (BIC bit-exact, cBIC within the tolerances and
    bit-equal to score_one), and the refusal of 256 candidates"""
    p, K, v = 256, 2, 0
    total = 1 + 255 + comb(255, 2)
    assert total == 32641
    want = [0] + [1 << j for j in range(1, p)] + [(1 << a) | (1 << b) for b in range(1, p) for a in range(1, b)]
    nb = (1 << p) - 1
    rng = np.random.default_rng(255)
    sample = np.unique(np.concatenate([rng.choice(total, size=330, replace=False), [0, 1, 255, 256, 257, total - 1]]))
    # cBIC
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=2000, seed=6, mean_indegree=2.0)
    eng.set_continuous(x)
    assert eng.family_size(v, nb, K, pkg.CBIC) == total
    res = eng.score_variable(v, nb, K, pkg.CBIC, lam=LAM, flags=pkg.CBIC_NO_ACCEPT)
    assert res.scored() == total and res.count() == total
    m, neg = res.fetch()
    res.free()
    assert m.shape == (total, 4)
    assert [pkg.words_to_mask(row) for row in m] == want
    for i in sample:
        members = [j for j in range(p) if (want[i] >> j) & 1]
        r = sub_residual(orc, x, v, members)
        assert ulp_diff(-neg[i], np.float32(r)) <= 1, members
        s, ts64 = eng.score_one(v, want[i], pkg.CBIC, LAM)
        assert abs(ts64 - r) <= TOL * max(1.0, abs(r))
        assert bits(s) == bits(neg[i])
    # BIC: raw scores of the whole family by range, the cache = those under the store rule
    codes, card, _, _ = pkg.datagen.discrete_bn(p=p, n=3000, seed=7, arities=(2, 3, 4), window=4, max_indegree=2)
    eng.set_discrete(codes, card)
    raw = eng.score_range(v, nb, K, pkg.BIC, 0, total)
    res = eng.score_variable(v, nb, K, pkg.BIC)
    assert res.scored() == total
    mb, sb = res.fetch()
    res.free()
    stored = np.array([raw[0] < 1] + [s < 0 for s in raw[1:]])
    assert [pkg.words_to_mask(row) for row in mb] == [w for w, st in zip(want, stored) if st]
    assert np.array_equal(bits(sb), bits(raw[stored]))
    for i in sample:
        members = [j for j in range(p) if (want[i] >> j) & 1]
        sub = sorted(members + [v])
        s_ref, _ = orc.bic_score(codes[sub], card[sub], sub.index(v), sum(1 << sub.index(j) for j in members))
        assert bits(raw[i]) == bits(s_ref), members
    # 256 candidates
    x2, _ = pkg.datagen.linear_gaussian_sem(p=257, n=500, seed=2)
    eng.set_continuous(x2)
    with pytest.raises(pkg.UrlGpuError, match="at most 255"):
        eng.score_variable(0, (1 << 257) - 1, 2, pkg.CBIC, lam=LAM)


# ------------------------------------------------------------------------------------------------ 4. literal-zero acceptance

def check_literal(pkg, orc, e, p, v, nb, K):
    nb &= ~(1 << v)    # the oracle's enumeration counts v among the neighbours when it is named (62 at most)
    om = orc.enumerate_sets(v, nb, p, K)
    om = om[orc.canonical_order(om)]
    m0, neg = no_accept(e, pkg, v, nb, K)
    assert np.array_equal(m0[:, 0], om)
    ts = -neg
    stored, val = orc.cbic_accept(v, p, om, ts, mode=1)
    m, s = no_accept(e, pkg, v, nb, K, pkg.CBIC_ACCEPT_LITERAL)
    assert np.array_equal(m[:, 0], om[stored]), (p, v, K)
    assert np.array_equal(bits(s), bits(val[stored]))
    keep = orc.prune(om[stored], val[stored], K)
    m, s = no_accept(e, pkg, v, nb, K, pkg.CBIC_ACCEPT_LITERAL | pkg.PRUNE_DOMINATED)
    assert np.array_equal(m[:, 0], om[stored][keep]) and np.array_equal(bits(s), bits(val[stored][keep]))


@pytest.mark.parametrize("layout", ["dense", "rank"])
@pytest.mark.parametrize("p", [13, 14])
def test_literal_acceptance_at_12_parents(pkg, orc, layouts, p, layout):
    """accept_literal_kernel with K = 12: all 13 LiteralFrames and all 256 words of the per-thread checked bitset; variable 0
    as the child, as a candidate (two launches per layer) and absent from the family"""
    e = layouts[layout]
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=2000, seed=200 + p)
    e.set_continuous(x)
    allb = (1 << p) - 1
    for v, nb in ((0, allb), (p // 2, allb), (p - 1, allb), (3, allb & ~1)):
        check_literal(pkg, orc, e, p, v, nb, 12)


@pytest.mark.parametrize("p,K", [(32, 4), (63, 3)])
def test_literal_acceptance_up_to_62_candidates(pkg, orc, layouts, p, K):
    """accept_literal_kernel over 31 and 62 candidates (rank layout, 1-word masks up to bit 62)"""
    e = layouts["rank"]
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=1500, seed=300 + p)
    e.set_continuous(x)
    allb = (1 << p) - 1
    for v, nb in ((0, allb), (p - 1, allb), (5, allb & ~1)):
        check_literal(pkg, orc, e, p, v, nb, K)


def test_literal_acceptance_refuses_63_candidates(pkg, eng):
    x, _ = pkg.datagen.linear_gaussian_sem(p=64, n=500, seed=64)
    eng.set_continuous(x)
    with pytest.raises(pkg.UrlGpuError, match="at most 62 candidates"):
        eng.score_variable(0, (1 << 64) - 1, 1, pkg.CBIC, lam=LAM, flags=pkg.CBIC_ACCEPT_LITERAL)
    m, _ = no_accept(eng, pkg, 0, (1 << 64) - 1, 1)
    assert len(m) == 64


# ------------------------------------------------------------------------------------------------ 5. standalone prune

def prune_case(nvars, seed, words=3):
    """a few thousand distinct masks spanning exactly `nvars` variables, bit 0 unused, some above bit 64 (and 128);
    scores with many exact ties -> (masks uint64 [m, words], scores, variables)"""
    rng = np.random.default_rng(seed)
    hi = [int(i) for i in rng.choice(np.arange(128, 64 * words), size=min(3, nvars // 3), replace=False)]
    mid = [int(i) for i in rng.choice(np.arange(64, 128), size=min(3, nvars // 3), replace=False)]
    low = [int(i) for i in rng.choice(np.arange(1, 64), size=nvars - len(hi) - len(mid), replace=False)]
    vars_ = sorted(hi + mid + low)
    sets = {0}
    for j in range(nvars):
        sets.add(1 << j)
    while len(sets) < 3000:
        l = int(rng.integers(2, min(nvars, 7) + 1))
        sets.add(sum(1 << int(j) for j in rng.choice(nvars, size=l, replace=False)))
    compact = np.array(sorted(sets), dtype=np.uint64)
    rng.shuffle(compact)
    full = np.zeros((len(compact), words), dtype=np.uint64)
    for i, cm in enumerate(compact):
        for j in range(nvars):
            if (int(cm) >> j) & 1:
                full[i, vars_[j] >> 6] |= np.uint64(1) << np.uint64(vars_[j] & 63)
    scores = (-rng.integers(1, 12, size=len(compact)) * 7.25).astype(np.float32)
    return full, compact, scores


@pytest.mark.parametrize("nvars", [12, 13, 20, 30])
def test_standalone_prune_many_variables(pkg, orc, eng, nvars):
    """urlgpu_prune: the union compacted to nvars bits, segment DP with 2^(nvars - 11) high parts (hb = 1, 2, 9, 19), the
    scatter and gather around it; against the oracle's prune on the order-preserving relabelling of the masks"""
    full, compact, scores = prune_case(nvars, seed=nvars)
    keep = eng.prune(full, scores)
    ref = orc.prune(compact, scores)
    assert 0 < ref.sum() < len(ref)
    assert np.array_equal(keep, ref)


def test_standalone_prune_refuses_31_variables(pkg, eng):
    full, _, scores = prune_case(31, seed=31)
    with pytest.raises(pkg.UrlGpuError, match="more than 30 distinct variables"):
        eng.prune(full, scores)
    full, compact, scores = prune_case(12, seed=3)
    assert eng.prune(full, scores).sum() > 0
