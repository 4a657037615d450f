"""Pins the oracle's continuous-BIC restatement against the REFERENCE'S OWN CODE: scoring_function/BIC_OLS.cpp and
score_calculator.cpp compiled from an urlearning-cpp checkout (oracle/_ref/libref_cbic.so, oracle/ref.mk) over shim Boost headers and a
minimal Armadillo / mlpack (oracle/shim_arma: matrices, mean, var, a no-intercept linear regression written from their
published algorithms in the oracle's arithmetic order).  Pinned here: the standardisation, the score formula, the acceptance
test with its recursion exactly AS WRITTEN (SURVEY.md Q5: arma::uvec zero-filled) and the enumeration / store loop — the
reference's control flow and formulas.  NOT pinned: the floating-point arithmetic inside Armadillo / mlpack, which both
sides restate."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "oracle", "_ref", "libref_cbic.so")
pytestmark = pytest.mark.skipif(not os.path.exists(SO), reason="oracle/_ref/libref_cbic.so not built (reference sources were absent)")


@pytest.fixture(scope="module")
def refc():
    L = C.CDLL(SO)
    L.refc_open.restype = C.c_void_p
    L.refc_open.argtypes = [C.c_char_p, C.c_double]
    L.refc_p.argtypes = [C.c_void_p]
    L.refc_calculate_score.restype = C.c_float
    L.refc_calculate_score.argtypes = [C.c_void_p, C.c_int, C.c_uint64]
    L.refc_score_variable.restype = C.c_int64
    L.refc_score_variable.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
    return L


def _reference_cache(L, h, v, nb, K, prune=False):
    n = L.refc_score_variable(h, v, nb, K, int(prune), None, None, 0)
    masks, scores = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.float32)
    L.refc_score_variable(h, v, nb, K, int(prune), masks.ctypes.data, scores.ctypes.data, n)
    return {int(m): s for m, s in zip(masks, scores)}


def _compare(orc, L, csv, lam, expect_clean_differs):
    t = orc.Table(csv)
    x, p = t.values(), t.p
    z = orc.standardise(x)
    h = L.refc_open(csv.encode(), lam)
    assert h and L.refc_p(h) == p
    differs_from_clean = 0
    for v in range(p):
        nb = (1 << p) - 1
        om = orc.enumerate_sets(v, nb, p, p - 1)
        ts = np.array([orc.cbic_residual(z, v, int(m), lam) for m in om], dtype=np.float64).astype(np.float32)
        for m, t_ in list(zip(om, ts))[::7]:      # single sets on an empty cache: -the_score, bit for bit
            r = np.float32(L.refc_calculate_score(h, v, int(m)))
            assert r == np.float32(-t_) and (r != 0 or True)
        ref = _reference_cache(L, h, v, nb, p - 1)
        stored, val = orc.cbic_accept(v, p, om, ts, mode=1)          # the recursion as written
        mine = {int(m): s for m, k, s in zip(om, stored, val) if k}
        assert set(ref) == set(mine), (v, len(set(ref) ^ set(mine)))
        assert all(np.float32(ref[m]).view(np.uint32) == np.float32(mine[m]).view(np.uint32) for m in ref), v
        clean, _ = orc.cbic_accept(v, p, om, ts, mode=0)
        differs_from_clean += len(set(ref) ^ {int(m) for m, k in zip(om, clean) if k})
        # the commented-out prune, applied by the reference's own ScoreCalculator::prune to its own cache
        pruned = _reference_cache(L, h, v, nb, p - 1, prune=True)
        km = np.array(sorted(mine), dtype=np.uint64)
        ks = np.array([mine[int(m)] for m in km], dtype=np.float32)
        keep = orc.prune(km, ks, p - 1)
        assert set(pruned) == {int(m) for m in km[keep]}, v
    assert (differs_from_clean > 0) == expect_clean_differs
    return differs_from_clean


def test_figure_1_against_the_compiled_reference(orc, refc):
    _compare(orc, refc, os.path.join(ROOT, "tests", "data", "Figure_1", "raw_data_8000.csv"), 2.0, expect_clean_differs=False)


@pytest.mark.parametrize("p,n,seed", [(9, 500, 3), (10, 400, 4)])
def test_literal_acceptance_where_it_differs_from_clean(orc, pkg, refc, tmp_path, p, n, seed):
    """p >= 9: the recursion as written stores a different key set than the clean one (SURVEY Q5 measured 5-9 % of the keys);
    the oracle's literal mode reproduces the reference's compiled code key for key and bit for bit"""
    x, _ = pkg.datagen.linear_gaussian_sem(p=p, n=n, seed=seed)
    csv = str(tmp_path / "x.csv")
    np.savetxt(csv, x.T, delimiter=",", fmt="%.17g")
    assert _compare(orc, refc, csv, 2.0, expect_clean_differs=True) > 50
