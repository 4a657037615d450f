"""GPU parity of the cube path's two-digit groups.

A set T that holds cube bits 0 and 1 is derived by ``cube_derive_kernel`` in groups of card[0] * card[1] configurations,
and the pass scores T, T \\ {0}, T \\ {1} and T \\ {0,1} from the same registers.  Only tables that a pass reads are written.
Pairs whose parent's pass built no such groups keep groups of card[0] x 1 and 1 x 1: the children of plain roots, and the
children T \\ {1} of a fused root's children T.  (2, 2) runs a compile-time group; any other shape runs the group
configuration by configuration.  Here the two lowest cube digits have arities (2, 2), (2, 3), (3, 3) and (2, 4); children
have arity 2, 3, 4 and 6; roots are fused and plain; the candidates number K + 1 (the root layer is K or K + 1) or K + 3
(up to K + 2, where the layers above K hold only sets with their lowest bits forced); families of 1, 2 and 3 candidates;
the family split into parts; 16-bit tables forced down to layer 1, and skewed data whose 16-bit tables overflow and fall
back to 32 bits.  BIC and fNML, dense and rank layouts, bit-exact against the oracle.
"""
import numpy as np
import pytest

from conftest import engine_with_env
from test_gpu_kernel_variants import Oracle, _bits, _check_discrete, _fetch, _random_codes

pytestmark = pytest.mark.gpu

N = 70_001
CHILDREN = {2: 0, 3: 1, 4: 2, 6: 3}     # child arity -> column
# arities of the two lowest cube digits -> candidate arities (cube order sorts by arity, ties by index: the first two listed
# are the lowest digits).  Twelve candidates at n = 70 001: the roots hold 0.2-50M cells, above the shared-memory tiers, and
# are cut into enough slices for the root kernel, which fuses them where URLGPU_FUSE_ROOTS allows it
CASES = {
    (2, 2): [2, 2, 3, 4, 3, 4, 3, 4, 3, 4, 2, 3],
    (2, 3): [2, 3, 3, 4, 3, 4, 3, 4, 3, 3, 4, 3],
    (3, 3): [3, 3, 3, 4, 3, 4, 3, 3, 4, 3, 3, 3],
    (2, 4): [2, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4],
}
KS = (11, 9)                              # the root layer is K or K + 1 (12 = K + 1 candidates), or up to K + 2


def _data(low):
    cand = CASES[low]
    card = [2, 3, 4, 6] + cand
    codes = _random_codes(card, N, seed=9000 + 10 * low[0] + low[1])
    return codes, card, _bits(range(4, 4 + len(cand)))


@pytest.mark.parametrize("low", sorted(CASES))
def test_two_digit_groups_fused_and_plain(pkg, orc, low):
    """every child arity, both root routes, K + 1 and K + 3 candidates; the fused route really occurs (its families write
    fewer K1 bytes than the plain route's)"""
    codes, card, nb = _data(low)
    ora = Oracle(orc, codes, card)
    written = {}
    for fuse, layouts in (("1", ("dense", "rank")), ("0", ("dense",))):
        for layout in layouts:
            eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_FUSE_ROOTS": fuse, "URLGPU_LAYOUT": layout})
            eng.set_discrete(codes, card)
            for rv, v in CHILDREN.items():
                for K in KS:
                    for st in (pkg.BIC, pkg.FNML):
                        _check_discrete(pkg, ora, eng, v, nb, K, st, pkg.PRUNE_DOMINATED, what=f"low={low} fuse={fuse} {layout} rv={rv} K={K} st={st}")
                if layout == "dense":
                    eng.reset_stats()
                    for K in KS:
                        _fetch(eng, v, nb, K, pkg.BIC)
                    written[fuse, rv] = eng.stats()["k1_bytes_written"]
            eng.close()
    for rv in CHILDREN:
        assert 0 < written["1", rv] < written["0", rv], (low, rv, written["1", rv], written["0", rv])


@pytest.mark.parametrize("low", [(2, 2), (2, 3)])
def test_two_digit_groups_in_parts(pkg, orc, low):
    """urlgpu_score_part: each part derives the sub-forest of its roots (T \\ {1} is scored with T); the parts are disjoint, cover the
    family, and their int32-MIN merge is the oracle's cache"""
    NOT_SCORED = np.uint32(0x7FC0BEEF)
    codes, card, nb = _data(low)
    ora = Oracle(orc, codes, card)
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_LAYOUT": "dense"})
    eng.set_discrete(codes, card)
    for v in (0, 3):
        for K in KS:
            for st in (pkg.BIC, pkg.FNML):
                for parts in (2, 3):
                    arrs = [eng.score_part(v, nb, K, st, part, parts) for part in range(parts)]
                    scored = np.stack([a.view(np.uint32) for a in arrs]) != NOT_SCORED
                    assert np.all(scored.sum(axis=0) == 1), (low, v, K, st, parts)
                    merged = np.min(np.stack([a.view(np.int32) for a in arrs]), axis=0).view(np.float32)
                    got = eng.result_from_scores(v, nb, K, st, merged, flags=pkg.PRUNE_DOMINATED)
                    masks, scores = got.fetch()
                    got.free()
                    om, osc = ora.cache(pkg, v, nb, K, st, True)
                    assert [int(m) for m in masks[:, 0]] == [int(m) for m in om], (low, v, K, st, parts)
                    assert np.array_equal(scores.view(np.uint32), osc.view(np.uint32)), (low, v, K, st, parts)
    eng.close()


def test_two_digit_groups_small_families(pkg, orc):
    """families of 1, 2 and 3 candidates (bit 1 or bit 2 missing), every K, through the cube path"""
    codes, card, _ = _data((2, 3))
    ora = Oracle(orc, codes, card)
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube"})
    eng.set_discrete(codes, card)
    for cols in ([4], [5], [4, 5], [5, 7], [4, 5, 6], [5, 6, 7], [4, 5, 7]):
        nb = _bits(cols)
        for K in range(1, len(cols) + 1):
            for rv, v in CHILDREN.items():
                for st in (pkg.BIC, pkg.FNML):
                    _check_discrete(pkg, ora, eng, v, nb, K, st, what=f"cols={cols} K={K} rv={rv} st={st}")
    eng.close()


def test_two_digit_groups_16bit_tables(pkg, orc):
    """(a) 16-bit cells forced down to layer 1 (URLGPU_TABLE16_MINLAYER=1): exact and no fallback; (b) skewed data whose
    modal configuration holds > 65535 records in every table: the written 16-bit tables overflow, the variable falls back
    to 32-bit tables and stays exact"""
    codes, card, nb = _data((2, 3))
    ora = Oracle(orc, codes, card)
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_TABLE16_MINLAYER": "1"})
    eng.set_discrete(codes, card)
    eng.reset_stats()
    for rv, v in CHILDREN.items():
        for K in KS:
            _check_discrete(pkg, ora, eng, v, nb, K, pkg.BIC, what=f"forced16 rv={rv} K={K}")
    assert eng.stats()["table16_fallbacks"] == 0
    eng.close()

    rng = np.random.default_rng(11)
    n = 200_003
    scard = [2, 2, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3]
    skew = np.stack([(rng.random(n) < 0.04).astype(np.uint8) * rng.integers(1, r, size=n).astype(np.uint8) for r in scard])
    for i, r in enumerate(scard):
        skew[i, :3] = np.minimum([0, 1, 2], r - 1)   # every value appears, in order
    sora = Oracle(orc, skew, scard)
    eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_TABLE16_MINLAYER": "3"})
    eng.set_discrete(skew, scard)
    eng.reset_stats()
    snb = _bits(range(1, len(scard)))
    for K in (9, 8):
        _check_discrete(pkg, sora, eng, 0, snb, K, pkg.BIC, pkg.PRUNE_DOMINATED, what=f"skew K={K}")
    assert eng.stats()["table16_fallbacks"] == 1   # once for the variable: its later scorings go straight to 32-bit tables
    eng.close()
