"""fNML (SURVEY.md §8f rank 4): the regret tables and the oracle's fNML restatement, pinned against the reference's own
code (oracle/_ref: fnml_scoring_function.cpp + getRegretCache compiled from the checkout URLEARNING_CPP_SRC names) and,
for the K = 2 table, against the literals in the reference's header when that checkout is present."""
import os
import re
import struct
import zlib

import numpy as np
import pytest

import ref_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEP = os.path.join(ROOT, "tests", "data", "hepatitis.clean.csv")
REF_SRC = os.environ.get("URLEARNING_CPP_SRC")
REF_HEADER = os.path.join(REF_SRC, "urlearning", "scoring_function", "fnml_scoring_function.h") if REF_SRC else None
R2_CRC = 0x85246587   # crc32 of the 1001 float32 bit patterns (tools/gen_regret_table.py)


def read_inc(path):
    bits = [int(x, 16) for x in re.findall(r"0x([0-9a-f]{8})u", open(path).read())]
    assert len(bits) == 1001
    return bits


def test_generated_r2_tables_are_identical_and_match_their_crc():
    a = read_inc(os.path.join(ROOT, "oracle", "regret_r2.inc"))
    b = read_inc(os.path.join(ROOT, "urlearning-cpp_b200", "csrc", "regret_r2.inc"))
    assert a == b
    assert zlib.crc32(struct.pack("<1001I", *a)) == R2_CRC
    f = np.array(a, dtype=np.uint32).view(np.float32)
    assert f[0] == 1 and f[1] == 2 and f[2] == 2.5 and f[3] == np.float32(26 / 9)   # C(N,2) by hand
    assert np.all(np.diff(f) > 0)


@pytest.mark.skipif(not (REF_HEADER and os.path.exists(REF_HEADER)), reason="reference sources not present")
def test_r2_table_equals_the_reference_literals_as_float32():
    src = open(REF_HEADER).read()
    body = src[src.index("r2_1000[] = {") + len("r2_1000[] = {"):]
    body = body[:body.index("};")]
    ref = np.array([float(x) for x in re.findall(r"[-+0-9.eE]+", body)], dtype=np.float64).astype(np.float32)
    mine = np.array(read_inc(os.path.join(ROOT, "oracle", "regret_r2.inc")), dtype=np.uint32).view(np.float32)
    assert len(ref) == 1001 and np.array_equal(ref.view(np.uint32), mine.view(np.uint32))


def test_log_regret_rows(orc):
    r1 = orc.log_regret(50, 1)
    assert np.all(r1 == 0)                                        # C(N, 1) = 1
    r2 = orc.log_regret(2000, 2)
    assert r2[0] == 0 and r2[1] == np.float32(np.log(2.0)) and r2[2] == np.float32(np.log(2.5))
    assert abs(float(r2[1001]) - float(r2[1000])) < 1e-3          # Szpankowski's approximation joins the table smoothly
    r3 = orc.log_regret(10, 3)
    # C(N,3) = C(N,2) + N * C(N,1): N = 1 -> 3, N = 2 -> 4.5
    assert r3[1] == np.float32(np.log(3.0)) and r3[2] == np.float32(np.log(np.float32(4.5)))


@pytest.mark.skipif(not ref_lib.available(), reason="oracle/_ref not built (reference sources were absent)")
def test_regret_and_fnml_scores_against_the_reference(orc):
    ref = ref_lib.Reference(HEP, has_header=True)
    codes = ref.codes()
    for r in sorted(set(int(c) for c in ref.card)):
        mine = orc.log_regret(ref.n, r)
        theirs = np.array([ref.regret(r, N) for N in range(ref.n + 1)], dtype=np.float32)
        assert np.array_equal(mine.view(np.uint32), theirs.view(np.uint32)), r
    rng = np.random.default_rng(5)
    cases = [(0, 0), (0, 2), (19, 0)]
    for _ in range(200):
        k = int(rng.integers(0, 5))
        cases.append((int(rng.integers(20)), sum(1 << int(i) for i in rng.choice(20, size=k, replace=False))))
    worst, exact, n = 0.0, 0, 0
    for v, m in cases:
        m &= ~(1 << v)
        r = ref.fnml_score(v, m)
        q = orc.fnml_score_many(codes, ref.card, v, [m], mode=0, threads=1)[0]
        lit = orc.fnml_score_many(codes, ref.card, v, [m], mode=1, threads=1)[0]
        worst = max(worst, abs(float(r) - float(q)) / abs(float(r)), abs(float(r) - float(lit)) / abs(float(r)))
        exact += int(r.view(np.uint32) == lit.view(np.uint32))
        n += 1
    assert worst < 3e-6            # float32 accumulation order (boost::unordered_map iteration) vs the exact contract
    assert exact >= 0.4 * n


def test_fnml_large_n_rows_use_the_approximation(orc):
    r = orc.log_regret(5000, 4)
    assert np.all(np.isfinite(r)) and np.all(np.diff(r[1:]) > 0)


@pytest.mark.skipif(not ref_lib.available(), reason="oracle/_ref not built (reference sources were absent)")
@pytest.mark.parametrize("ess", [1.0, 10.0, 0.25])
def test_bdeu_scores_against_the_reference(orc, ess):
    """the oracle's BDeu (both modes) vs the reference's own BDeuScoringFunction::calculateScore: float32 running-sum noise"""
    ref = ref_lib.Reference(HEP, has_header=True)
    codes = ref.codes()
    rng = np.random.default_rng(7)
    cases = [(0, 0), (0, 2), (19, 0)]
    for _ in range(150):
        k = int(rng.integers(0, 5))
        cases.append((int(rng.integers(20)), sum(1 << int(i) for i in rng.choice(20, size=k, replace=False))))
    worst, exact, n = 0.0, 0, 0
    for v, m in cases:
        m &= ~(1 << v)
        r = ref.bdeu_score(v, m, ess)
        q = orc.bdeu_score_many(codes, ref.card, v, [m], ess=ess, mode=0, threads=1)[0]
        lit = orc.bdeu_score_many(codes, ref.card, v, [m], ess=ess, mode=1, threads=1)[0]
        worst = max(worst, abs(float(r) - float(q)) / abs(float(r)), abs(float(r) - float(lit)) / abs(float(r)))
        exact += int(r.view(np.uint32) == lit.view(np.uint32))
        n += 1
    assert worst < 5e-6
    assert exact >= 0.1 * n       # the configuration terms are added in boost::unordered_map order there, ascending here


def test_bdeu_known_answer_by_hand(orc):
    """two binary variables, 4 records (0,0),(0,1),(1,0),(1,1), ess = 1, X0 with parent X1: r = 2, a_ij = 1/2, a_ijk = 1/4,
    every cell 1, every configuration 2:  4*(lgamma(1.25) - lgamma(0.25)) + 2*(lgamma(0.5) - lgamma(2.5))"""
    from math import lgamma
    codes = np.array([[0, 0, 1, 1], [0, 1, 0, 1]], dtype=np.uint8)
    want = 4 * (lgamma(1.25) - lgamma(0.25)) + 2 * (lgamma(0.5) - lgamma(2.5))
    got = orc.bdeu_score_many(codes, [2, 2], 0, [0b10], ess=1.0, mode=0, threads=1)[0]
    assert abs(float(got) - want) < 1e-6 * abs(want)


def test_product_regret_builder_equals_the_oracle(orc, tmp_path):
    """the engine's host-side table builder (csrc/regret.hpp, compiled here with g++ as plain C++) against the oracle's
    restatement, bit for bit: arities 1..9, N up to 3000 (the exact K=2 row, Szpankowski's approximation above 1000, the
    float32 recurrence), and an arity whose regret overflows float32"""
    import ctypes as C
    import subprocess
    so = str(tmp_path / "regret_probe.so")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, os.path.join(ROOT, "tests", "regret_probe.cpp")])
    lib = C.CDLL(so)
    lib.probe_log_regret.argtypes = [C.c_int64, C.c_int, C.c_void_p]
    for r in range(1, 10):
        mine = np.zeros(3001, dtype=np.float32)
        lib.probe_log_regret(3000, r, mine.ctypes.data)
        assert np.array_equal(mine.view(np.uint32), orc.log_regret(3000, r).view(np.uint32)), r
    wide = np.zeros(200001, dtype=np.float32)
    lib.probe_log_regret(200000, 60, wide.ctypes.data)
    ref = orc.log_regret(200000, 60)
    assert np.array_equal(wide.view(np.uint32), ref.view(np.uint32)) and not np.all(np.isfinite(wide))


@pytest.mark.skipif(not ref_lib.available(), reason="oracle/_ref not built (reference sources were absent)")
def test_regret_fnml_bdeu_against_the_reference_at_n_3000(orc, pkg, tmp_path):
    """a synthetic network with 3000 records: the regret rows beyond N = 1000 (Szpankowski's approximation + the float32
    recurrence) are bit-equal to the reference's compiled getRegretCache, and fNML / BDeu scores agree to accumulation noise"""
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=8, n=3000, seed=23, arities=(2, 3, 4), window=3, max_indegree=2)
    path = str(tmp_path / "syn.csv")
    pkg.datagen.write_csv(path, codes)
    ref = ref_lib.Reference(path)
    assert ref.n == 3000 and np.array_equal(ref.codes(), codes)       # first-appearance coding of the generator's columns
    for r in sorted(set(int(c) for c in ref.card)):
        mine = orc.log_regret(ref.n, r)
        theirs = np.array([ref.regret(r, N) for N in range(ref.n + 1)], dtype=np.float32)
        assert np.array_equal(mine.view(np.uint32), theirs.view(np.uint32)), r
    rng = np.random.default_rng(11)
    worst_f = worst_b = 0.0
    for _ in range(120):
        v = int(rng.integers(8))
        k = int(rng.integers(0, 4))
        m = sum(1 << int(i) for i in rng.choice(8, size=k, replace=False)) & ~(1 << v)
        rf, rb = float(ref.fnml_score(v, m)), float(ref.bdeu_score(v, m, 1.0))
        of = float(orc.fnml_score_many(codes, ref.card, v, [m], mode=0, threads=1)[0])
        ob = float(orc.bdeu_score_many(codes, ref.card, v, [m], ess=1.0, mode=0, threads=1)[0])
        worst_f = max(worst_f, abs(rf - of) / abs(rf))
        worst_b = max(worst_b, abs(rb - ob) / abs(rb))
    assert worst_f < 2e-5 and worst_b < 5e-5      # float32 running sums (and, for BDeu, lgammaf) over up to 256 cells at N = 3000 (SURVEY Q4: ~1e-5)
