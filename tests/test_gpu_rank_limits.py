"""Rank-layout score caches past 2^31 parent sets, up to the 2^32 - 16 sets a family may have.

The rank layout (rank_kernels.cuh) numbers a family's sets by 32-bit colex index, and ``make_rank_space`` admits families of
up to 4 294 967 280 sets.  BIC with ``-p 5`` on a 200-column CSV without a skeleton already has 2.5e9 sets per variable.
Every stage is held here to an exact answer at such indices: direct counting (``bic_score_direct``), the per-set cBIC
sweeps, the store rule, the acceptance and prune DPs, the compaction, the index-to-mask expansion and the range checks.

The answers come from two helpers, tied to the oracle by ``test_colex_helpers_and_closed_form_match_the_oracle``:

- colex rank and unrank in exact Python integers: index(S) = layer_base[|S|] + sum_i C(e_i, i);
- a closed form for discrete scores when most candidates are CONSTANT (arity 1, every code 0).  Such a candidate leaves the
  contingency table, the penalty product and BDeu's a_ij unchanged, so score(S) == score(S & I) bit for bit, I the
  informative candidates.  With the m informative candidates at the top positions, the sets of layer l whose informative
  part is J = {e_1 < .. < e_j} form one block starting at layer_base[l] + sum_i C(e_i, l - j + i), of length
  C(c - m, l - j); the blocks tile the layer (Vandermonde).  A whole family of billions of raw scores is then at most
  2^m (K + 1) runs of values known from the oracle on the (m + 1)-variable sub-problem.

Large caches are fetched in slices at an offset into torch buffers and compared on the device.  Each GPU case first checks
free device (and host) memory against its peak and skips, naming the numbers, when the machine cannot hold it.

- index limit: family sizes at and above the limit, and BIC / fNML / BDeu ranges up to index 2^32 - 34 (c = 32, K = 30);
- a whole BIC family of 2 147 630 816 sets (c = 109, K = 6), unfiltered, by range and pruned; fNML and BDeu across 2^31;
- a whole cBIC family of 4 258 490 216 sets (c = 122, K = 6), 99.2 % of 2^32, without and with acceptance and prune;
- range and fetch refusals whose uint64 sums would wrap, after which the context still scores and fetches.
"""
from itertools import combinations
from math import comb

import numpy as np
import pytest

from conftest import engine_with_env
from test_gpu_record_limits import _need

LAM = 2.0
TOL = 1e-9
ERR_ARG, ERR_LIMIT = -1, -3
U64 = (1 << 64) - 1


# ------------------------------------------------------------------------------------------------ colex helpers
def layer_bases(c: int, K: int) -> list[int]:
    """first index of each layer l = 0..K, then the family size"""
    out, b = [], 0
    for l in range(K + 1):
        out.append(b)
        b += comb(c, l)
    return out + [b]


def colex_index(c: int, K: int, pos) -> int:
    """ascending candidate positions -> index in the family's canonical (|S|, colex) numbering"""
    pos = sorted(pos)
    return layer_bases(c, K)[len(pos)] + sum(comb(e, i + 1) for i, e in enumerate(pos))


def colex_unrank(c: int, K: int, idx: int) -> list[int]:
    """index -> ascending candidate positions"""
    base = layer_bases(c, K)
    l = max(j for j in range(K + 1) if base[j] <= idx)
    r, e, hi = idx - base[l], [0] * l, c - 1
    for i in range(l, 0, -1):
        b = hi
        while comb(b, i) > r:
            b -= 1
        e[i - 1] = b
        r -= comb(b, i)
        hi = b - 1
    return e


def closed_form_runs(c: int, K: int, m: int):
    """(start, length, J) in index order: the sets whose informative part (the top m positions) is J, J a tuple of positions"""
    base = layer_bases(c, K)
    runs = []
    for l in range(K + 1):
        for j in range(min(l, m) + 1):
            if l - j > c - m:
                continue
            for J in combinations(range(c - m, c), j):
                runs.append((base[l] + sum(comb(e, l - j + i + 1) for i, e in enumerate(J)), comb(c - m, l - j), J))
    return sorted(runs)


def _ulps(a, b):
    a = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a)
    b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def _padded(codes_inf, card_inf, child, p, inf_vars, v=0):
    """[p, n] codes: the child at v, the informative columns at inf_vars, every other variable constant (arity 1)"""
    n = codes_inf.shape[1]
    codes = np.zeros((p, n), dtype=np.uint8)
    card = np.ones(p, dtype=np.int32)
    codes[v], card[v] = codes_inf[child], card_inf[child]
    others = [i for i in range(len(card_inf)) if i != child]
    for q, i in zip(inf_vars, others):
        codes[q], card[q] = codes_inf[i], card_inf[i]
    return codes, card


def _sub_scores(orc, codes, card, v, inf_vars, score_type, pkg, ess=1.0):
    """oracle scores of (v, J) for every J within inf_vars, on the sub-problem [v] + inf_vars -> {frozenset of variables: float32}"""
    sub = sorted([v] + list(inf_vars))
    vs = sub.index(v)
    Js = [J for j in range(len(inf_vars) + 1) for J in combinations(inf_vars, j)]
    masks = np.array([sum(1 << sub.index(q) for q in J) for J in Js], dtype=np.uint64)
    if score_type == pkg.BIC:
        s = orc.bic_score_many(codes[sub], card[sub], vs, masks)
    elif score_type == pkg.FNML:
        s = orc.fnml_score_many(codes[sub], card[sub], vs, masks)
    else:
        s = orc.bdeu_score_many(codes[sub], card[sub], vs, masks, ess=ess)
    return {frozenset(J): np.float32(x) for J, x in zip(Js, s)}


# ------------------------------------------------------------------------------------------------ CPU: the helpers
@pytest.mark.parametrize("c,K,m", [(9, 4, 3), (10, 10, 4), (12, 5, 5), (7, 3, 0)])
def test_colex_helpers_and_closed_form_match_the_oracle(pkg, orc, c, K, m):
    """the oracle's enumeration in canonical order is index order for colex_index / colex_unrank; the closed form's runs
    tile the family and hold exactly the sets with their informative part; and the oracle's BIC, fNML and BDeu of every set
    equal those of its informative part bit for bit, with the constant columns present"""
    p, v = c + 1, 0
    om = orc.enumerate_sets(v, (1 << p) - 1, p, K)
    om = om[orc.canonical_order(om)]
    base = layer_bases(c, K)
    assert len(om) == base[-1]
    positions = [[q - 1 for q in range(1, p) if (int(mk) >> q) & 1] for mk in om]
    for i, pos in enumerate(positions):
        assert colex_index(c, K, pos) == i and colex_unrank(c, K, i) == pos
    runs = closed_form_runs(c, K, m)
    top = set(range(c - m, c))
    at = 0
    for start, length, J in runs:
        assert start == at and length > 0
        for i in range(start, start + length):
            assert tuple(sorted(set(positions[i]) & top)) == J
        at += length
    assert at == len(om)
    codes_inf, card_inf, _, _ = pkg.datagen.discrete_bn(p=m + 1, n=997, seed=c + m, arities=(2, 3, 4), window=3, max_indegree=2)
    inf_vars = [q + 1 for q in range(c - m, c)]
    codes, card = _padded(codes_inf, card_inf, m, p, inf_vars)
    for st, full in ((pkg.BIC, orc.bic_score_many), (pkg.FNML, orc.fnml_score_many), (pkg.BDEU, None)):
        got = full(codes, card, v, om) if full else orc.bdeu_score_many(codes, card, v, om, ess=1.0)
        want = _sub_scores(orc, codes, card, v, inf_vars, st, pkg)
        for i, mk in enumerate(om):
            assert _bits(got[i]) == _bits(want[frozenset(q for q in inf_vars if (int(mk) >> q) & 1)])


# ------------------------------------------------------------------------------------------------ GPU
def _rc_family_size(eng, v, nb, K, st):
    """(return code, size) of urlgpu_family_size"""
    import ctypes as C
    words = (eng.p + 63) // 64
    w = np.array([(nb >> (64 * i)) & U64 for i in range(words)], dtype=np.uint64)
    n = C.c_uint64()
    rc = eng.lib.urlgpu_family_size(eng._h, v, w.ctypes.data, words, K, st, C.byref(n))
    return rc, n.value


def _mask_of(pos, cand):
    return sum(1 << cand[e] for e in pos)


def _informative_data(pkg, m, n, seed, arities):
    """m informative columns and a child that depends on some of them (child = column m); every column takes all its values"""
    codes, card, _, _ = pkg.datagen.discrete_bn(p=m + 1, n=n, seed=seed, arities=arities, window=m, max_indegree=3)
    assert (card >= 2).all()
    return codes, card


@pytest.mark.gpu
def test_index_limit_family_sizes_and_ranges_to_2_32(pkg, orc):
    """family sizes on both sides of 2^32 - 16, then ranges of the c = 32, K = 30 BIC family (4 294 967 263 sets) near its end,
    across 2^31 and across every layer base from layer 14 up: BIC and fNML bit-equal to the oracle, BDeu bit-equal to
    score_sets of the same sets and within one ulp of the oracle.  12 informative candidates of arity 2 or 3 at mixed
    positions (tables up to 3 3^12 cells: shared-memory and global tiers), the other 20 constant."""
    _need(4)
    eng = pkg.Engine(0)
    try:
        # cBIC sizes on an installed Gram (256 variables)
        eng.set_gram(np.eye(256) * 1000.0, 1000)
        assert _rc_family_size(eng, 0, (1 << 123) - 1, 6, pkg.CBIC) == (0, 4258490216)
        assert _rc_family_size(eng, 0, (1 << 256) - 1, 5, pkg.CBIC)[0] == ERR_LIMIT
        p, v, K, n = 33, 0, 30, 3001
        cand = list(range(1, p))
        inf_pos = [0, 3, 5, 9, 12, 14, 17, 20, 24, 27, 30, 31]
        inf_vars = [cand[e] for e in inf_pos]
        codes_inf, card_inf = _informative_data(pkg, 12, n, 32, (2, 3))
        codes, card = _padded(codes_inf, card_inf, 12, p, inf_vars)
        eng.set_discrete(codes, card)
        nb = (1 << p) - 1
        T = layer_bases(32, K)[-1]
        assert T == 4294967263
        assert _rc_family_size(eng, v, nb, K, pkg.BIC) == (0, T)
        assert _rc_family_size(eng, v, nb, 31, pkg.BIC)[0] == ERR_LIMIT
        base = layer_bases(32, K)
        slices = [(T - 600, 600), ((1 << 31) - 97, 194)] + [(base[l] - 80, 160) for l in range(14, K + 1)]
        idx = np.concatenate([np.arange(f, f + k) for f, k in slices])
        pos = [colex_unrank(32, K, int(i)) for i in idx]
        inf_set = set(inf_vars)
        Jof = [frozenset(q for q in (cand[e] for e in ps) if q in inf_set) for ps in pos]
        assert min(len(ps) for ps in pos) == 13 and max(len(ps) for ps in pos) == K
        for st in (pkg.BIC, pkg.FNML, pkg.BDEU):
            raw = np.concatenate([eng.score_range(v, nb, K, st, f, k, lam=1.0) for f, k in slices])
            want = _sub_scores(orc, codes, card, v, inf_vars, st, pkg)
            ref = np.array([want[J] for J in Jof], dtype=np.float32)
            if st == pkg.BDEU:
                assert _ulps(raw, ref).max() <= 1
                one, _ = eng.score_sets([v] * len(pos), [_mask_of(ps, cand) for ps in pos], pkg.BDEU, lam=1.0)
                assert np.array_equal(_bits(raw), _bits(one))
            else:
                assert np.array_equal(_bits(raw), _bits(ref)), st
    finally:
        eng.close()


def _full_bic_case(pkg):
    """c = 109, K = 6: variable 0 the child, five informative candidates of arity 2-4 at the top positions 104..108
    (variables 105..109), 104 constant candidates; n = 4 099 (not a multiple of 16)"""
    p, v, K, n, m = 110, 0, 6, 4099, 5
    codes_inf, card_inf = _informative_data(pkg, m, n, 109, (2, 3, 4))
    inf_vars = list(range(105, 110))
    codes, card = _padded(codes_inf, card_inf, m, p, inf_vars)
    return p, v, K, m, codes, card, inf_vars


def _check_runs(torch, scores_dev, runs, cand, value_of):
    """every run [start, start + length) of the device array holds the bits of value_of(J)"""
    for start, length, J in runs:
        want = int(_bits(value_of(frozenset(cand[e] for e in J))).view(np.int32))
        seg = scores_dev[start:start + length].view(torch.int32)
        bad = int((seg != want).sum())
        assert bad == 0, (start, length, J, bad)


@pytest.mark.gpu
def test_whole_bic_family_past_2_31(pkg, orc):
    """T = 2 147 630 816 sets, 147 169 of them above 2^31 - 1.  score_variable (store rule): every set stored, every score on
    its closed-form run, masks = unrank(index) at layer edges, at 2^31 - 1 and 2^31, at T - 1 and at random entries;
    score_range(0, T) gives the same bits; those raw scores with PRUNE_DOMINATED leave exactly the oracle's pruned cache of
    the 32 informative subsets (a set with constant members ties with its informative part, and a tie drops the larger set):
    the prune DP and the compaction over 2.1e9 entries.  fNML and BDeu over [2^31 - 5 000, 2^31 + 5 000) by closed form."""
    import torch
    _need(55)
    p, v, K, m, codes, card, inf_vars = _full_bic_case(pkg)
    c = p - 1
    cand = list(range(1, p))
    T = layer_bases(c, K)[-1]
    assert T == 2147630816 and T - ((1 << 31) - 1) == 147169
    runs = closed_form_runs(c, K, m)
    bic = _sub_scores(orc, codes, card, v, inf_vars, pkg.BIC, pkg)
    eng = pkg.Engine(0)
    try:
        eng.set_discrete(codes, card)
        nb = (1 << p) - 1
        res = eng.score_variable(v, nb, K, pkg.BIC)
        assert res.scored() == T and res.count() == T
        got = torch.empty(T, dtype=torch.float32, device="cuda")
        assert res.fetch_device(0, got.data_ptr()) == T
        torch.cuda.synchronize()
        _check_runs(torch, got, runs, cand, bic.__getitem__)
        base = layer_bases(c, K)
        rng = np.random.default_rng(109)
        probe = {0, (1 << 31) - 1, 1 << 31, T - 1} | {b for b in base[1:K + 1]} | {b - 1 for b in base[1:K + 2]}
        probe |= {int(i) for i in rng.integers(0, T, size=200)}
        for i in sorted(probe):
            mk, sc = res.fetch(first=i, n=1)
            assert pkg.words_to_mask(mk[0]) == _mask_of(colex_unrank(c, K, i), cand), i
            assert _bits(sc[0]) == _bits(got[i].item())
        res.free()
        # the same family by range, into a device buffer
        raw = torch.empty(T, dtype=torch.float32, device="cuda")
        assert eng.score_range(v, nb, K, pkg.BIC, 0, T, out_device_ptr=raw.data_ptr()) is None
        torch.cuda.synchronize()
        assert torch.equal(raw.view(torch.int32), got.view(torch.int32))
        del got
        torch.cuda.empty_cache()
        # prune
        res = eng.result_from_scores(v, nb, K, pkg.BIC, raw.data_ptr(), T, flags=pkg.PRUNE_DOMINATED)
        masks, scores = res.fetch()
        res.free()
        sub = [v] + inf_vars
        om = np.array([sum(1 << sub.index(q) for q in J) for J in bic], dtype=np.uint64)
        osc = np.array(list(bic.values()), dtype=np.float32)
        assert (osc < 0).all()
        keep = orc.prune(om, osc, K)
        want = sorted(((len(J), sum(1 << q for q in J), s) for (J, s), k in zip(bic.items(), keep) if k), key=lambda t: t[:2])
        assert [pkg.words_to_mask(row) for row in masks] == [w[1] for w in want]
        assert np.array_equal(_bits(scores), _bits([w[2] for w in want]))
        del raw
        torch.cuda.empty_cache()
        # fNML and BDeu: the same launches; a 10 000-set range across 2^31
        first, count = (1 << 31) - 5000, 10000
        Jof = [frozenset(cand[e] for e in colex_unrank(c, K, first + i) if e >= c - m) for i in range(count)]
        fn = eng.score_range(v, nb, K, pkg.FNML, first, count)
        fw = _sub_scores(orc, codes, card, v, inf_vars, pkg.FNML, pkg)
        assert np.array_equal(_bits(fn), _bits([fw[J] for J in Jof]))
        bd = eng.score_range(v, nb, K, pkg.BDEU, first, count, lam=1.0)
        bw = _sub_scores(orc, codes, card, v, inf_vars, pkg.BDEU, pkg)
        assert _ulps(bd, [bw[J] for J in Jof]).max() <= 1
        Js = sorted(set(Jof), key=sorted)
        one, _ = eng.score_sets([v] * len(Js), [sum(1 << q for q in J) for J in Js], pkg.BDEU, lam=1.0)
        gpu_j = {J: s for J, s in zip(Js, one)}
        assert np.array_equal(_bits(bd), _bits([gpu_j[J] for J in Jof]))
    finally:
        eng.close()
        torch.cuda.empty_cache()


def _popcount64(torch, x):
    """per-element popcount of an int64 tensor (SWAR; the arithmetic shifts are masked)"""
    x = x - ((x >> 1) & 0x5555555555555555)
    x = (x & 0x3333333333333333) + ((x >> 2) & 0x3333333333333333)
    x = (x + (x >> 4)) & 0x0F0F0F0F0F0F0F0F
    return (x * 0x0101010101010101) >> 56


def _words_i64(mask, words):
    return np.array([(mask >> (64 * w)) & U64 for w in range(words)], dtype=np.uint64).view(np.int64)


def _scan_cache(torch, res, n, words, regions, chunk=1 << 27):
    """walk the whole stored cache on the device in slices: popcounts non-decreasing throughout, and the entries whose mask
    lies inside each of `regions` (masks) -> [(masks uint64 [k, words], scores float32 [k])]"""
    mb = torch.empty((chunk, words), dtype=torch.int64, device="cuda")
    sb = torch.empty(chunk, dtype=torch.float32, device="cuda")
    outside = [torch.from_numpy(~_words_i64(r, words)).cuda() for r in regions]
    found = [([], []) for _ in regions]
    last = -1
    for first in range(0, n, chunk):
        k = min(chunk, n - first)
        assert res.fetch_device(mb.data_ptr(), sb.data_ptr(), first=first, n=k) == k
        mm, ss = mb[:k], sb[:k]
        pc = _popcount64(torch, mm).sum(dim=1)
        assert int(pc[0]) >= last and bool((pc[1:] >= pc[:-1]).all()), first
        last = int(pc[-1])
        for (fm, fs), out in zip(found, outside):
            inside = ((mm & out) == 0).all(dim=1)
            fm.append(mm[inside].cpu().numpy().view(np.uint64))
            fs.append(ss[inside].cpu().numpy())
        torch.cuda.synchronize()
    return [(np.concatenate(fm), np.concatenate(fs)) for fm, fs in found]


@pytest.mark.gpu
def test_whole_cbic_family_near_2_32(pkg, orc):
    """c = 122, K = 6: T = 4 258 490 216 sets, 99.2 % of 2^32.  CBIC_NO_ACCEPT: every set stored; at layer edges, 2^31 +- 1,
    T - 1 and random entries the mask is unrank(index), the score within one ulp of the oracle on the relabelled sub-problem
    and bit-equal to score_one.  Without acceptance, with it and with PRUNE_DOMINATED: popcounts non-decreasing over the
    whole cache, and its restrictions to the first 24 candidates (the bottom of every layer) and to the last 24 equal the
    24-candidate families scored in the dense layout on the same Gram (acceptance and prune of S look only at subsets of S)."""
    import torch
    _need(80)
    p, v, K, n = 123, 0, 6, 2000
    c = p - 1
    cand = list(range(1, p))
    T = layer_bases(c, K)[-1]
    assert T == 4258490216
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=123, mean_indegree=2.0)
    eng = pkg.Engine(0)
    dense = engine_with_env(pkg, {"URLGPU_LAYOUT": "dense"})
    try:
        eng.set_continuous(x)
        dense.set_gram(eng.gram(), n)
        nb = (1 << p) - 1
        assert eng.family_size(v, nb, K, pkg.CBIC) == T
        first24 = sum(1 << q for q in cand[:24])
        last24 = sum(1 << q for q in cand[-24:])
        base = layer_bases(c, K)
        rng = np.random.default_rng(122)
        probe = {0, (1 << 31) - 1, 1 << 31, (1 << 31) + 1, T - 1} | set(base[1:K + 1]) | {b - 1 for b in base[1:K + 2]}
        probe |= {int(i) for i in rng.integers(0, T, size=300)}
        for flags in (pkg.CBIC_NO_ACCEPT, 0, pkg.PRUNE_DOMINATED):
            res = eng.score_variable(v, nb, K, pkg.CBIC, lam=LAM, flags=flags)
            assert res.scored() == T
            stored = res.count()
            if flags == pkg.CBIC_NO_ACCEPT:
                assert stored == T
                for i in sorted(probe):
                    mk, neg = res.fetch(first=i, n=1)
                    members = [cand[e] for e in colex_unrank(c, K, i)]
                    mask = sum(1 << q for q in members)
                    assert pkg.words_to_mask(mk[0]) == mask, i
                    sub = sorted(members + [v])
                    r = orc.cbic_residual(orc.standardise(x[sub]), sub.index(v), sum(1 << sub.index(q) for q in members), LAM)
                    assert _ulps(-neg[0], np.float32(r)) <= 1, (i, members)
                    s, ts64 = eng.score_one(v, mask, pkg.CBIC, LAM)
                    assert abs(ts64 - r) <= TOL * max(1.0, abs(r))
                    assert _bits(s) == _bits(neg[0])
            found = _scan_cache(torch, res, stored, 2, [first24, last24])
            res.free()
            torch.cuda.empty_cache()
            for region, (fm, fs) in zip((first24, last24), found):
                rd = dense.score_variable(v, region | (1 << v), K, pkg.CBIC, lam=LAM, flags=flags)
                md, sd = rd.fetch()
                rd.free()
                assert len(md) > 0 and np.array_equal(fm, md), (flags, region == first24)
                assert np.array_equal(_bits(fs), _bits(sd)), (flags, region == first24)
    finally:
        eng.close()
        dense.close()
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_range_and_fetch_refusals_that_would_wrap(pkg):
    """score_range past the family's end and with first + count wrapping past 2^64, and result_fetch / result_fetch_device with
    offset + n wrapping: each refused with URLGPU_ERR_ARG, and the context still scores and fetches the same bits"""
    import ctypes as C
    import torch
    _need(2)
    p, v, K = 33, 0, 30
    codes_inf, card_inf = _informative_data(pkg, 12, 3001, 32, (2, 3))
    codes, card = _padded(codes_inf, card_inf, 12, p, [1, 4, 6, 10, 13, 15, 18, 21, 25, 28, 31, 32])
    eng = pkg.Engine(0)
    try:
        eng.set_discrete(codes, card)
        nb = (1 << p) - 1
        T = eng.family_size(v, nb, K, pkg.BIC)
        before = eng.score_range(v, nb, K, pkg.BIC, T - 300, 300)
        words = np.array([nb], dtype=np.uint64)
        out = torch.empty(4, dtype=torch.float32, device="cuda")
        for first, count in ((T, 1), (U64, 2), (T - 1, U64)):
            rc = eng.lib.urlgpu_score_range(eng._h, v, words.ctypes.data, 1, K, pkg.BIC, 0.0, first, count, C.c_void_p(out.data_ptr()), 1)
            assert rc == ERR_ARG and "exceeds the family" in eng.lib.urlgpu_last_error(eng._h).decode()
        res = eng.score_variable(v, nb, 3, pkg.BIC, flags=pkg.PRUNE_DOMINATED)
        m0, s0 = res.fetch()
        assert len(m0) > 2
        mh = np.zeros((2, 1), dtype=np.uint64)
        sh = np.zeros(2, dtype=np.float32)
        md = torch.empty(2, dtype=torch.int64, device="cuda")
        for off, k in ((U64, 2), (len(m0), 1), (1, U64)):
            assert eng.lib.urlgpu_result_fetch(res._h, off, k, mh.ctypes.data, sh.ctypes.data) == ERR_ARG
            assert eng.lib.urlgpu_result_fetch_device(res._h, off, k, 1, 0, C.c_void_p(md.data_ptr()), C.c_void_p(out.data_ptr())) == ERR_ARG
        m1, s1 = res.fetch(first=len(m0) - 2, n=2)
        assert np.array_equal(m1, m0[-2:]) and np.array_equal(_bits(s1), _bits(s0[-2:]))
        assert res.fetch_device(md.data_ptr(), out.data_ptr(), first=len(m0) - 2, n=2) == 2
        assert np.array_equal(md.cpu().numpy().view(np.uint64), m0[-2:, 0]) and np.array_equal(_bits(out[:2].cpu().numpy()), _bits(s0[-2:]))
        res.free()
        assert np.array_equal(_bits(eng.score_range(v, nb, K, pkg.BIC, T - 300, 300)), _bits(before))
    finally:
        eng.close()
