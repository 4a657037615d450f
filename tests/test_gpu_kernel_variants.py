"""GPU parity of every shipped kernel variant, selected on purpose rather than by accident of shape.

Each test names the instantiation or route it reaches and checks it against the CPU oracle (tests/oracle_lib.py) or a
plain numpy reference, at the project's tolerances: BIC and fNML bit-exact, BDeu within one float32 ulp on under 2 % of
the scores with identical stored lists, cBIC within 1e-9 relative on the FP64 value and one float32 ulp on the float.

- root kernel ``bic_root_kernel<RV, NW>``: RV = 2, 3, 4 and 0 (generic child arity), NW = 8, 12 and 16 warps, fused and
  plain roots, both cache layouts, segment caps at both ends, and the slice route switched off;
- the root kernel's shared-memory sizing at the largest budget and segment cap the switches admit;
- the direct-counting tiers (``bic_classify_kernel`` / ``bic_count_smem_kernel`` / the global tier) with tables exactly on
  and just above each tier boundary, a call of several global batches, and the range and part entry points;
- one table above the global tier's batch size through ``score_one`` / ``contingency``, and the 2^30-cell refusals;
- ``cube_derive_kernel<0>`` with 16-bit tables;
- K3 level B: every ``cbic_dfs_kernel<0..4>`` and ``cbic_tree_kernel<7..11>``.
"""
from math import comb

import numpy as np
import pytest

from conftest import engine_with_env

pytestmark = pytest.mark.gpu

T0_CELLS = 12 * 1024              # tier 0 of the direct path: tables of at most this many cells (48 KB of shared memory)
BATCH_CELLS = 12 << 20            # the global tier's scratch: tables of one batch, int32 cells
TOL = 1e-9


def _tier1_cells():
    """tier 1 of the direct path: what one block may opt into, less 2 KB, in int32 cells (the library's own sizing)"""
    import torch
    return (torch.cuda.get_device_properties(0).shared_memory_per_block_optin - 2048) // 4


def _ulps(a, b):
    a = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a)
    b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)


def _bits(idx):
    return sum(1 << int(i) for i in idx)


def _random_codes(card, n, seed):
    """uniform codes, each later column leaning on two earlier ones, so that tables are neither uniform nor sparse alone"""
    rng = np.random.default_rng(seed)
    p = len(card)
    codes = np.zeros((p, n), dtype=np.uint8)
    for i, r in enumerate(card):
        col = rng.integers(0, r, size=n)
        if i >= 2:
            dep = (codes[i - 1].astype(np.int64) * 7 + codes[i - 2]) % r
            col = np.where(rng.random(n) < 0.4, dep, col)
        codes[i] = col
    return codes


class Oracle:
    """the whole family's oracle scores, once per (child, candidates, K, score)"""

    def __init__(self, orc, codes, card):
        self.orc, self.codes, self.card, self.p = orc, codes, np.asarray(card, dtype=np.int32), codes.shape[0]
        self.memo = {}

    def raw(self, pkg, v, nb, K, st):
        key = (v, nb, K, st)
        if key not in self.memo:
            om = self.orc.enumerate_sets(v, nb, self.p, K)
            om = om[self.orc.canonical_order(om)]
            if st == pkg.BIC:
                osc = self.orc.bic_score_many(self.codes, self.card, v, om)
            elif st == pkg.FNML:
                osc = self.orc.fnml_score_many(self.codes, self.card, v, om)
            else:
                osc = self.orc.bdeu_score_many(self.codes, self.card, v, om, ess=1.0)
            self.memo[key] = (om, osc)
        return self.memo[key]

    def cache(self, pkg, v, nb, K, st, prune):
        """the stored list in canonical order (score_calculator.cpp's store rule, then the subset-dominance prune)"""
        om, osc = self.raw(pkg, v, nb, K, st)
        stored = np.array([(s < 1) if m == 0 else (s < 0) for m, s in zip(om, osc)])
        om, osc = om[stored], osc[stored]
        if prune:
            keep = self.orc.prune(om, osc, K)
            om, osc = om[keep], osc[keep]
        return om, osc

    def cells(self, v, om):
        return np.array([int(self.card[v]) * int(np.prod([int(self.card[i]) for i in range(self.p) if (int(m) >> i) & 1])) for m in om],
                        dtype=np.int64)


def _fetch(eng, v, nb, K, st, flags=0, lam=0.0):
    res = eng.score_variable(v, nb, K, st, lam=lam, flags=flags)
    masks, scores = res.fetch()
    scored = res.scored()
    res.free()
    return masks, scores, scored


def _check_discrete(pkg, ora, eng, v, nb, K, st, flags=0, what=""):
    lam = 1.0 if st == pkg.BDEU else 0.0
    masks, scores, scored = _fetch(eng, v, nb, K, st, flags, lam)
    om, osc = ora.cache(pkg, v, nb, K, st, bool(flags & pkg.PRUNE_DOMINATED))
    assert scored == len(ora.raw(pkg, v, nb, K, st)[0]), what
    assert [int(m) for m in masks[:, 0]] == [int(m) for m in om], what
    if st == pkg.BDEU:
        d = _ulps(scores, osc)
        assert d.max() <= 1 and (d > 0).mean() < 0.02, (what, int(d.max()), float((d > 0).mean()))
    else:
        assert np.array_equal(scores.view(np.uint32), osc.view(np.uint32)), what
    return masks, scores


# ------------------------------------------------------------------------------------------------ 1. root kernel matrix
# Four children of arity 2, 3, 4 and 6 (bic_root_kernel<2|3|4|0, NW>), twelve candidates of arities 2..4 interleaved by
# index (the cube order sorts them).  n = 70 001 (ragged, >= 65 536: the packed rows exist), K = 9: the cost model roots
# the family at layer 11, ten roots of 0.2-1.5M cells, i.e. above tier 1 and cut into >= 128 slices.  Roots missing a low
# cube bit are fused (their children come out of the root kernel), the others are plain roots.
ROOT_N = 70_001
ROOT_CHILDREN = {2: 0, 3: 1, 4: 2, 6: 3}                       # child arity -> column
ROOT_CAND_AR = [4, 2, 3, 4, 3, 2, 4, 3, 4, 2, 3, 4]
ROOT_CARD = [2, 3, 4, 6] + ROOT_CAND_AR
ROOT_NB = _bits(range(4, 4 + len(ROOT_CAND_AR)))
ROOT_K = 9


@pytest.fixture(scope="module")
def root_data(orc):
    codes = _random_codes(ROOT_CARD, ROOT_N, seed=70001)
    return codes, Oracle(orc, codes, ROOT_CARD)


def _root_family_sweep(pkg, ora, eng, what, scores=None, flags_set=None):
    for rv, v in ROOT_CHILDREN.items():
        for st in scores or (pkg.BIC, pkg.FNML):
            for flags in flags_set or (0, pkg.PRUNE_DOMINATED):
                _check_discrete(pkg, ora, eng, v, ROOT_NB, ROOT_K, st, flags, what=f"{what} rv={rv} st={st} flags={flags}")


@pytest.mark.parametrize("warps", [8, 12, 16])
def test_root_kernel_warps_fusion_layouts(pkg, root_data, warps):
    """bic_root_kernel<RV, NW> for RV = 2, 3, 4, 0 and NW = `warps`: fused and plain roots (URLGPU_FUSE_ROOTS), dense and
    rank layouts, BIC and fNML, with and without the prune; bit-exact against the oracle.  Fused roots really occur: a fused
    root's table never reaches HBM, and its children are the ones the plain route derives and writes, so every child's
    family writes fewer K1 bytes (stats k1_bytes_written) with URLGPU_FUSE_ROOTS=1 than with 0"""
    codes, ora = root_data
    written = {}
    for fuse in ("1", "0"):
        for layout in ("dense", "rank"):
            eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_ROOT_WARPS": str(warps), "URLGPU_FUSE_ROOTS": fuse,
                                        "URLGPU_LAYOUT": layout})
            eng.set_discrete(codes, ROOT_CARD)
            _root_family_sweep(pkg, ora, eng, f"warps={warps} fuse={fuse} {layout}")
            if layout == "dense":
                for rv, v in ROOT_CHILDREN.items():
                    eng.reset_stats()
                    _fetch(eng, v, ROOT_NB, ROOT_K, pkg.BIC)
                    written[fuse, rv] = eng.stats()["k1_bytes_written"]
            eng.close()
    for rv in ROOT_CHILDREN:
        assert 0 < written["1", rv] < written["0", rv], (rv, written["1", rv], written["0", rv])


@pytest.mark.parametrize("warps,segs", [(16, 32), (8, 32), (12, 8192), (16, 8192)])
def test_root_kernel_segment_caps(pkg, root_data, warps, segs):
    """URLGPU_ROOT_SEGS at its lower clamp (32: most slices take the fragmented-segment branch of the root kernel) and at
    8192 (every slice's segment table in shared memory; with the default 24K-cell budget that still fits the opt-in)"""
    codes, ora = root_data
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_ROOT_WARPS": str(warps), "URLGPU_ROOT_SEGS": str(segs)})
    eng.set_discrete(codes, ROOT_CARD)
    _root_family_sweep(pkg, ora, eng, f"warps={warps} segs={segs}", flags_set=(0,))
    eng.close()


def test_root_slice_route_witness_and_red_route(pkg, root_data):
    """URLGPU_SLICE_COUNT=0 sends the same roots through the global-atomic (RED) batches instead: bit-exact too.  And the
    slice route really ran above: it adds the packed-row launches (key, scan, scatter, map, root kernel) to the count
    family, which the RED route's one or two batches do not reach"""
    codes, ora = root_data
    sliced = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_SLICE_COUNT": "1"})
    red = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_SLICE_COUNT": "0"})
    for e in (sliced, red):
        e.set_discrete(codes, ROOT_CARD)
    _root_family_sweep(pkg, ora, red, "slice=0")
    for rv, v in ROOT_CHILDREN.items():
        launches = []
        for e in (sliced, red):
            e.reset_stats()
            _fetch(e, v, ROOT_NB, ROOT_K, pkg.BIC)
            launches.append(e.stats()["launches_count"])
        assert launches[0] > launches[1], (rv, launches)
    sliced.close()
    red.close()


# ------------------------------------------------------------------------------------------------ 2. root shared memory
@pytest.mark.parametrize("budget,segs", [(1_000_000, 1_000_000), (48 * 1024, 4096)])
def test_root_shared_memory_at_the_largest_switches(pkg, root_data, budget, segs):
    """URLGPU_ROOT_BUDGET and URLGPU_ROOT_SEGS at the top of their clamps (48K cells, 8192 segments), and a 48K budget with
    4096 segments, ask bic_root_kernel for more shared memory, with its static shared memory, than a block may opt into.
    urlgpu_create lowers the segment cap until they fit (every sm_100 device opts into 227 KB, so it always can), and the
    context then counts its roots in 48K-cell slices, bit-exact: the slice route runs (more count launches than the same
    budget with URLGPU_SLICE_COUNT=0) for the children whose roots make enough slices.  No later call meets a stale error"""
    codes, ora = root_data
    env = {"URLGPU_BIC_MODE": "cube", "URLGPU_ROOT_BUDGET": str(budget), "URLGPU_ROOT_SEGS": str(segs)}
    eng = engine_with_env(pkg, env)
    red = engine_with_env(pkg, {**env, "URLGPU_SLICE_COUNT": "0"})
    for e in (eng, red):
        e.set_discrete(codes, ROOT_CARD)
    _root_family_sweep(pkg, ora, eng, f"budget={budget} segs={segs}", flags_set=(0,))
    for rv in (4, 6):   # 0.4M-1.5M-cell roots: >= 128 slices of 48K cells
        launches = []
        for e in (eng, red):
            e.reset_stats()
            _fetch(e, ROOT_CHILDREN[rv], ROOT_NB, ROOT_K, pkg.BIC)
            launches.append(e.stats()["launches_count"])
        assert launches[0] > launches[1], (rv, launches)
    s, _ = eng.score_one(2, _bits([4, 5, 6]), pkg.BIC)
    assert s.view(np.uint32) == ora.orc.bic_score(codes, ROOT_CARD, 2, _bits([4, 5, 6]))[0].view(np.uint32)
    eng.close()
    red.close()
    after = pkg.Engine(0)   # a context created after it is unaffected
    after.set_discrete(codes, ROOT_CARD)
    _check_discrete(pkg, ora, after, 2, ROOT_NB, ROOT_K, pkg.BIC, what="default engine afterwards")
    after.close()


# ------------------------------------------------------------------------------------------------ 3. direct-counting tiers
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
    assert all(b <= 256 for b in bins)
    return sorted(bins, reverse=True)


def _tier_layout():
    """columns and families whose largest tables sit exactly on, and just above, the two shared-memory tier bounds, and one
    family whose global-tier tables add up to more than one batch"""
    t1 = _tier1_cells()
    t1_par = _split(t1 // 4)
    assert 4 * int(np.prod(t1_par)) == t1
    card = [3, 4] + [4] * 10 + t1_par + [t1_par[0] + 1]
    a4 = list(range(2, 12))
    tp = list(range(12, 12 + len(t1_par)))
    above = [len(card) - 1] + tp[1:]
    fams = {
        "tier0 exact (3*4^6)": (0, _bits(a4[:6]), 6, T0_CELLS),
        "tier0 + 1 digit (4^7)": (1, _bits(a4[:6]), 6, 4 * 4 ** 6),
        "tier1 exact": (1, _bits(tp), len(tp), t1),
        "just above tier1": (1, _bits(above), len(above), 4 * (t1_par[0] + 1) * int(np.prod(t1_par[1:]))),
        "several global batches": (1, _bits(a4), 10, 4 ** 11),
    }
    return t1, card, fams


def _expected_count_launches(cells, t0, t1):
    """launches of the count family for one direct-path call over sets of these table sizes (index order): one per
    shared-memory tier in use, three per global batch (zero the scratch, count, score), batches cut as the library does.
    This restates direct_global_tier's batching (first fit in index order, 4-cell alignment, <= 65 535 sets per batch), so
    a change there has to change this too.  The scratch is taken as max(12M cells, largest table): a context keeps the
    largest scratch it ever grew, so this holds only on a context that has seen no larger table (a fresh one per test)"""
    glob = [int(c) for c in cells if c > t1]
    batches, i = 0, 0
    cap = max(BATCH_CELLS, max(glob, default=0))
    while i < len(glob):
        used, j = 0, i
        while j < len(glob) and (j == i or used + glob[j] <= cap) and j - i < 65535:
            used += (glob[j] + 3) // 4 * 4
            j += 1
        batches += 1
        i = j
    return int(np.any(cells <= t0)) + int(np.any((cells > t0) & (cells <= t1))) + 3 * batches, batches


@pytest.fixture(scope="module")
def tier_data(orc):
    t1, card, fams = _tier_layout()
    codes = _random_codes(card, 30_011, seed=30011)
    return t1, card, fams, codes, Oracle(orc, codes, card)


@pytest.mark.parametrize("layout", ["dense", "rank"])
def test_direct_tier_edges_through_score_variable(pkg, tier_data, layout):
    """URLGPU_BIC_MODE=direct: bic_classify_kernel sends every set to tier 0 (<= 12 288 cells), tier 1 (<= the opt-in less
    2 KB) or the global tier.  Tables exactly on each bound and the next product above it; BIC, fNML and BDeu against the
    oracle; the tiers and the number of global batches each call ran are read back from the count-launch statistics and
    must match a host-side classification of the same tables"""
    t1, card, fams, codes, ora = tier_data
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "direct", "URLGPU_LAYOUT": layout})
    eng.set_discrete(codes, card)
    for name, (v, nb, K, top) in fams.items():
        om, _ = ora.raw(pkg, v, nb, K, pkg.BIC)
        cells = ora.cells(v, om)
        assert cells.max() == top, name
        want, batches = _expected_count_launches(cells, T0_CELLS, t1)
        if name == "several global batches":
            assert int(cells[cells > t1].sum()) > BATCH_CELLS and batches >= 2
        for st in (pkg.BIC, pkg.FNML, pkg.BDEU):
            for flags in ((0, pkg.PRUNE_DOMINATED) if st != pkg.BDEU else (0,)):
                eng.reset_stats()
                _check_discrete(pkg, ora, eng, v, nb, K, st, flags, what=f"{name} st={st} flags={flags}")
                assert eng.stats()["launches_count"] == want, (name, st, eng.stats()["launches_count"], want)
    eng.close()


def test_direct_tier_edges_through_ranges_and_parts(pkg, tier_data):
    """the same families through urlgpu_score_range (a cut inside a layer, a one-set range, a range ending at the last set,
    which is the family's largest table) and through urlgpu_score_part's range fallback (parts 2, 3, 8 merged by int32 MIN,
    filtered by urlgpu_result_from_scores): equal to the oracle, and to score_variable bit for bit"""
    t1, card, fams, codes, ora = tier_data
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "direct"})
    eng.set_discrete(codes, card)
    NOT_SCORED = np.uint32(0x7FC0BEEF)
    for name, (v, nb, K, _) in fams.items():
        total = eng.family_size(v, nb, K, pkg.BIC)
        c = bin(nb).count("1")
        bases = np.cumsum([0] + [comb(c, l) for l in range(K + 1)])
        widest = int(np.argmax(np.diff(bases)))
        cut = int(bases[widest] + (bases[widest + 1] - bases[widest]) // 2)   # inside the widest layer
        ranges = [(0, cut), (cut, 1), (cut + 1, total - cut - 1), (total - 1, 1)]
        for st in (pkg.BIC, pkg.FNML, pkg.BDEU):
            lam = 1.0 if st == pkg.BDEU else 0.0
            om, osc = ora.raw(pkg, v, nb, K, st)
            assert total == len(om)
            for first, count in ranges:
                if count == 0:
                    continue
                got = eng.score_range(v, nb, K, st, first, count, lam=lam)
                want = osc[first:first + count]
                if st == pkg.BDEU:
                    assert _ulps(got, want).max() <= 1, (name, first, count)
                else:
                    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (name, st, first, count)
            for parts in (2, 3, 8):
                arrs = [eng.score_part(v, nb, K, st, part, parts, lam=lam) for part in range(parts)]
                scored = np.stack([a.view(np.uint32) for a in arrs]) != NOT_SCORED
                assert np.all(scored.sum(axis=0) == 1), (name, parts)
                merged = np.min(np.stack([a.view(np.int32) for a in arrs]), axis=0).view(np.float32)
                for flags in (0, pkg.PRUNE_DOMINATED):
                    mw, sw, _ = _fetch(eng, v, nb, K, st, flags, lam)
                    got = eng.result_from_scores(v, nb, K, st, merged, flags=flags)
                    mg, sg = got.fetch()
                    got.free()
                    assert np.array_equal(mw, mg) and np.array_equal(sw.view(np.uint32), sg.view(np.uint32)), (name, st, parts, flags)
    eng.close()


# ------------------------------------------------------------------------------------------------ 4. one big table
def test_one_table_above_the_batch_size_and_the_cell_limit(pkg, orc):
    """score_one and contingency on a set of 4 * 4^11 = 16.8M cells, above the global tier's 12M-cell batch: the scratch
    grows for it.  Counts against numpy.bincount of the mixed-radix index (child digit first, stride 1, then the parents
    in ascending order), the score bit-exact against the oracle.  Then a set of 4^16 cells and a family containing one:
    refused by the host before anything is launched"""
    p, n = 16, 100_003
    card = [4] * p
    codes = _random_codes(card, n, seed=16)
    for mode in ("cube", "direct"):
        eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": mode})
        eng.set_discrete(codes, card)
        for v, parents in ((0, list(range(1, 12))), (15, list(range(3, 14)))):
            cells = 4 * 4 ** len(parents)
            assert cells > BATCH_CELLS
            idx = codes[v].astype(np.int64)
            stride = 4
            for q in sorted(parents):
                idx += codes[q].astype(np.int64) * stride
                stride *= 4
            want = np.bincount(idx, minlength=cells)
            got = eng.contingency(v, _bits(parents), cells)
            assert got.sum() == n and np.array_equal(got, want)
            s, ll = eng.score_one(v, _bits(parents), pkg.BIC)
            rs, rll = orc.bic_score(codes, card, v, _bits(parents))
            assert s.view(np.uint32) == rs.view(np.uint32) and ll == rll
        huge = _bits(range(1, 16))          # 4^16 = 2^32 cells
        with pytest.raises(pkg.UrlGpuError, match="exceeds 2\\^30 cells"):
            eng.score_one(0, huge, pkg.BIC)
        with pytest.raises(pkg.UrlGpuError, match="exceeds 2\\^30 cells"):
            eng.contingency(0, huge, 16)
        with pytest.raises(pkg.UrlGpuError, match="more than 2\\^30 cells"):
            eng.score_variable(0, huge, 15, pkg.BIC)
        s, _ = eng.score_one(3, _bits([1, 2]), pkg.BIC)     # the context is still usable
        assert s.view(np.uint32) == orc.bic_score(codes, card, 3, _bits([1, 2]))[0].view(np.uint32)
        eng.close()


# ------------------------------------------------------------------------------------------------ 5. generic-arity derive, 16-bit
def test_generic_arity_derive_with_16bit_tables(pkg, orc):
    """cube_derive_kernel<0> (child arity >= 5) reading and writing uint16 tables: URLGPU_TABLE16_MINLAYER=1 puts every
    derived layer in 16 bits.  Children of arity 5, 6 and 7, candidates of arity 5..7; BIC and fNML bit-exact.  The 16-bit
    tables are really written: the same families write fewer K1 bytes (stats k1_bytes_written counts 2 bytes per uint16
    cell) than with URLGPU_TABLE16=0, and no variable fell back to 32 bits"""
    card = [5, 6, 7, 5, 6, 7, 5, 6]
    codes = _random_codes(card, 40_009, seed=5)
    ora = Oracle(orc, codes, card)
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_TABLE16_MINLAYER": "1"})
    wide = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_TABLE16": "0"})
    nb = (1 << len(card)) - 1
    for e in (eng, wide):
        e.set_discrete(codes, card)
    for v in (0, 1, 2):
        for st in (pkg.BIC, pkg.FNML):
            for flags in (0, pkg.PRUNE_DOMINATED):
                _check_discrete(pkg, ora, eng, v, nb, 6, st, flags, what=f"v={v} st={st} flags={flags}")
        written = []
        for e in (eng, wide):
            e.reset_stats()
            _check_discrete(pkg, ora, e, v, nb, 6, pkg.BIC, what=f"v={v} written")
            stats = e.stats()
            assert stats["launches_cube"] > 0 and stats["table16_fallbacks"] == 0
            written.append(stats["k1_bytes_written"])
        assert 0 < written[0] < written[1], (v, written)
    eng.close()
    wide.close()


# ------------------------------------------------------------------------------------------------ 6. K3 level B widths
# Level B walks the J lowest candidate bits: J = min(c, 3) up to c = 13, 4 for c = 14..16, min(11, c - 10) above.
# cbic_dfs_kernel<J> for J <= 4 (c <= 16), cbic_tree_kernel<J> for J = 7..11 (c = 17..21 and above).  Level A sweeps the
# c - J high bits in 1, 2 or 3 stages.
CBIC_P, CBIC_N, LAM = 27, 3000, 2.0
CBIC_CS = list(range(0, 23)) + [26]


def _cbic_K(c):
    return c if c <= 14 else (6 if c <= 22 else 4)


@pytest.fixture(scope="module")
def cbic_data(pkg, orc):
    x, _ = pkg.datagen.linear_gaussian_sem(p=CBIC_P, n=CBIC_N, seed=27)
    return x, orc.standardise(x)


def test_cbic_every_level_b_width(pkg, orc, cbic_data):
    """c = 0..22 and 26 candidates of variable 0 (K = c up to 14, then 6, then 4): every cbic_dfs_kernel<0..4>, every
    cbic_tree_kernel<7..11>, level A in 1, 2 and 3 stages, segment DPs with and without high bits.  The dense cache equals
    the rank-layout cache bit for bit (no acceptance, acceptance, prune); >= 100 sampled sets per family against the
    oracle's residual form (1e-9) and score_one (bit-equal); acceptance and prune decisions against the oracle given the
    engine's own float32 scores"""
    x, z = cbic_data
    dense = engine_with_env(pkg, {"URLGPU_LAYOUT": "dense"})
    rank = engine_with_env(pkg, {"URLGPU_LAYOUT": "rank"})
    for e in (dense, rank):
        e.set_continuous(x)
    rng = np.random.default_rng(0)
    v = 0
    for c in CBIC_CS:
        K = _cbic_K(c)
        nb = _bits(range(1, c + 1))
        om = orc.enumerate_sets(v, nb, CBIC_P, K)
        om = om[orc.canonical_order(om)]
        caches = {}
        for flags in (pkg.CBIC_NO_ACCEPT, 0, pkg.PRUNE_DOMINATED):
            md, sd, nd = _fetch(dense, v, nb, K, pkg.CBIC, flags, LAM)
            mr, sr, nr = _fetch(rank, v, nb, K, pkg.CBIC, flags, LAM)
            assert nd == nr == len(om), (c, flags)
            assert np.array_equal(md, mr) and np.array_equal(sd.view(np.uint32), sr.view(np.uint32)), (c, flags)
            caches[flags] = (md[:, 0], sd)
        m0, neg_ts = caches[pkg.CBIC_NO_ACCEPT]
        assert np.array_equal(m0, om), c
        ts = -neg_ts
        for i in (range(len(om)) if len(om) <= 100 else rng.choice(len(om), size=100, replace=False)):
            r = orc.cbic_residual(z, v, int(om[i]), LAM)
            s, ts64 = dense.score_one(v, int(om[i]), pkg.CBIC, LAM)
            assert abs(ts64 - r) <= TOL * max(1.0, abs(r)), (c, int(om[i]))
            assert _ulps(ts[i], np.float32(r)) <= 1 and _ulps(-s, ts[i]) == 0, (c, int(om[i]))
        stored, val = orc.cbic_accept(v, CBIC_P, om, ts)
        ma, sa = caches[0]
        assert np.array_equal(ma, om[stored]) and np.array_equal(sa.view(np.uint32), val[stored].view(np.uint32)), c
        keep = orc.prune(om[stored], val[stored], K)
        mp, sp = caches[pkg.PRUNE_DOMINATED]
        assert np.array_equal(mp, om[stored][keep]) and np.array_equal(sp.view(np.uint32), val[stored][keep].view(np.uint32)), c
    dense.close()
    rank.close()
