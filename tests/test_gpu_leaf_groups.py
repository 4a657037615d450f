"""GPU parity of the cube path's leaf scoring when the lowest candidate arity r0 is not 2.

A leaf (a set without cube bit 0) is scored from the groups of r0 configurations of the pass that derives its parent:
``cube_derive_kernel`` and the fused-root passes of ``bic_root_kernel``.  r0 = 2 runs a compile-time group; any other r0
goes configuration by configuration and adds each one into the leaf's counts.  Here every candidate has arity >= 3, so
cube bit 0 has r0 = 3, 4 or 5, the children have arity 2, 3, 4 and 6, n >= 65 536 (the packed rows of the root kernel
exist), and roots are fused and plain.  BIC and fNML, dense and rank layouts, bit-exact against the oracle.
"""
import pytest

from conftest import engine_with_env
from test_gpu_kernel_variants import Oracle, _bits, _check_discrete, _fetch, _random_codes

pytestmark = pytest.mark.gpu

N = 70_001
CHILDREN = {2: 0, 3: 1, 4: 2, 6: 3}     # child arity -> column
# r0 -> (candidate arities, K).  The plan's cost model roots these families above K (layer K + 2 for r0 = 3; K + 1 or K + 2
# by child arity for r0 = 4 and 5) in tables of 0.6-4.9M cells, above the shared-memory tiers: the roots go through the root
# kernel and are fused when URLGPU_FUSE_ROOTS allows it
CASES = {
    3: ([3, 3, 3, 4, 3, 3, 4, 3, 3, 3, 4, 3], 9),
    4: ([4, 4, 5, 4, 4, 5, 4, 4, 4, 4, 4], 8),
    5: ([5, 5, 5, 5, 5, 5, 5, 5, 5, 5], 7),
}


@pytest.mark.parametrize("r0", sorted(CASES))
def test_leaf_groups_wider_than_two(pkg, orc, r0):
    """every child arity and score through the fused and the plain root route; the fused route really occurs (its families
    write fewer K1 bytes than the plain route's)"""
    cand, K = CASES[r0]
    card = [2, 3, 4, 6] + cand
    nb = _bits(range(4, 4 + len(cand)))
    codes = _random_codes(card, N, seed=7000 + r0)
    ora = Oracle(orc, codes, card)
    written = {}
    for fuse, layouts in (("1", ("dense", "rank")), ("0", ("dense",))):
        for layout in layouts:
            eng = engine_with_env(pkg, {"URLGPU_BIC_MODE": "cube", "URLGPU_FUSE_ROOTS": fuse, "URLGPU_LAYOUT": layout})
            eng.set_discrete(codes, card)
            for rv, v in CHILDREN.items():
                for st in (pkg.BIC, pkg.FNML):
                    _check_discrete(pkg, ora, eng, v, nb, K, st, pkg.PRUNE_DOMINATED, what=f"r0={r0} fuse={fuse} {layout} rv={rv} st={st}")
                if layout == "dense":
                    eng.reset_stats()
                    _fetch(eng, v, nb, K, pkg.BIC)
                    written[fuse, rv] = eng.stats()["k1_bytes_written"]
            eng.close()
    for rv in CHILDREN:
        assert 0 < written["1", rv] < written["0", rv], (r0, rv, written["1", rv], written["0", rv])
