"""Host-side consumers of the `.pss` (SURVEY.md 8(f) rows 1-2): the product's boost-free restatement (liburlsearch.so,
urlearning-cpp_b200/host/search_host.hpp) pinned against the REFERENCE'S OWN classes compiled from their sources
(oracle/_ref/libref_search.so: ScoreCache::read, SparseParentList / Bitwise / Tree, StaticPatternDatabase, PriorityQueue,
Node, Skeleton; only the A* loop of astar_main.cpp is restated in the driver) and against the reference's published golden
DAGs.  CPU only.  The `.pss` inputs here come from the oracle; tests/test_gpu_search.py feeds the GPU-written ones."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref_search.so")
DATA = os.path.join(ROOT, "tests", "data")


@pytest.fixture(scope="module")
def S():
    return importlib.import_module("urlearning-cpp_b200.search")


@pytest.fixture(scope="module")
def ref():
    if not os.path.exists(REF_SO):
        src = os.environ.get("URLEARNING_CPP_SRC")
        if not src or not os.path.isdir(os.path.join(src, "urlearning")):
            pytest.skip("oracle/_ref/libref_search.so was not built and URLEARNING_CPP_SRC names no reference checkout")
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "-f", "ref.mk", "REF=" + os.path.abspath(src)])
    L = C.CDLL(REF_SO)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.refs_open.restype = vp
    L.refs_open.argtypes = [C.c_char_p]
    L.refs_variable_count.argtypes = [vp]
    L.refs_name.restype = C.c_char_p
    L.refs_name.argtypes = [vp, i32]
    L.refs_arity.argtypes = [vp, i32]
    L.refs_entries.restype = i64
    L.refs_entries.argtypes = [vp, i32, vp, vp, i64]
    L.refs_best_scores.argtypes = [vp, C.c_char_p, i32, vp, i64, vp, vp]
    L.refs_astar.argtypes = [vp, C.c_char_p, i32, C.c_char_p, C.POINTER(C.c_float), vp, C.POINTER(C.c_int)]
    L.refs_last_error.restype = C.c_char_p
    L.refs_last_error.argtypes = [vp]
    return L


@pytest.fixture(scope="module")
def pss_files(orc, tmp_path_factory):
    d = tmp_path_factory.mktemp("pss")
    skel = os.path.join(DATA, "skeleton4_ones.csv")
    out = {"hep": str(d / "hep.pss"), "hep_pruned": str(d / "hep_pruned.pss"), "f1": str(d / "f1.pss"), "f2": str(d / "f2.pss")}
    orc.score_file(os.path.join(DATA, "hepatitis.clean.csv"), out["hep"], "BIC", has_header=True)
    orc.score_file(os.path.join(DATA, "hepatitis.clean.csv"), out["hep_pruned"], "BIC", has_header=True, prune=True)
    orc.score_file(os.path.join(DATA, "Figure_1", "raw_data_8000.csv"), out["f1"], "cBIC", skeleton=skel, lam=2.0)
    orc.score_file(os.path.join(DATA, "Figure_2", "raw_data_5000.csv"), out["f2"], "cBIC", skeleton=skel, lam=2.0)
    return out


def _ref_entries(ref, h, v):
    n = ref.refs_entries(h, v, None, None, 0)
    m, s = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.float32)
    ref.refs_entries(h, v, m.ctypes.data, s.ctypes.data, n)
    return m, s


@pytest.mark.parametrize("key", ["hep", "hep_pruned", "f1"])
def test_reader_equals_reference_reader(S, ref, pss_files, key):
    """every (variable, parent set, score) the reference's ScoreCache::read extracts from the file, and nothing else"""
    mine = S.ScoreCache(pss_files[key])
    h = ref.refs_open(pss_files[key].encode())
    assert h and ref.refs_variable_count(h) == mine.p
    assert [ref.refs_name(h, v).decode() for v in range(mine.p)] == mine.names
    assert [ref.refs_arity(h, v) for v in range(mine.p)] == mine.arity
    total = 0
    for v in range(mine.p):
        rm, rs = _ref_entries(ref, h, v)
        mm, ms = mine.entries(v)
        a = dict(zip((int(x) for x in rm), (float(np.float32(x)) for x in rs)))
        b = dict(zip((int(x) for x in mm), (float(np.float32(x)) for x in ms)))
        assert a == b
        assert np.all(np.diff(ms) >= 0)  # sorted by score (the search side minimises)
        total += len(a)
    assert total > 0
    assert mine.meta("pss_version") == "0.1" and mine.meta("score_type") in ("bic", "cbic")


def test_reader_quirks_match_reference(S, ref, tmp_path):
    """case-insensitive VAR/META, comments and blank lines, entry order, an unknown parent name (-> variable 0,
    bayesian_network.cpp:55-57).  (A variable NAME containing "meta" makes the reference's reader index past the end of
    its token vector, score_cache.cpp:115-126 — undefined behaviour there, so nothing to pin.)"""
    text = ("# comment\nMETA pss_version = 0.1\nmeta  num_records=80\n\nvar A\nMETA arity=2\n-1.500000 \n-3.250000 B \n\n"
            "VAR B\nMeta arity=3\n-2.000000 A C \n-9.000000 \n-4.000000 nobody \n\nVar C\nMETA arity=2\n-7.125000 A \n-8.000000 \n")
    path = str(tmp_path / "quirks.pss")
    open(path, "w").write(text)
    mine = S.ScoreCache(path)
    h = ref.refs_open(path.encode())
    assert ref.refs_variable_count(h) == mine.p == 3
    for v in range(3):
        rm, rs = _ref_entries(ref, h, v)
        mm, ms = mine.entries(v)
        assert dict(zip(map(int, rm), map(float, rs))) == dict(zip(map(int, mm), map(float, ms)))
    assert dict(zip(map(int, mine.entries(1)[0]), map(float, mine.entries(1)[1]))) == {0b101: 2.0, 0: 9.0, 0b001: 4.0}


@pytest.mark.parametrize("kind", ["list", "bitwise"])
def test_best_score_queries_equal_reference_structures(S, ref, pss_files, kind):
    """getScore(pars) = best cached subset (sparse_parent_list.cpp:44-55, sparse_parent_bitwise.cpp:90-110)"""
    mine = S.ScoreCache(pss_files["hep"])
    h = ref.refs_open(pss_files["hep"].encode())
    rng = np.random.default_rng(5)
    for v in (0, 9, 19):
        q = rng.integers(0, 1 << 20, size=600, dtype=np.uint64) & ~np.uint64(1 << v)
        q[:3] = [0, (1 << 20) - 1 - (1 << v), 1 << ((v + 1) % 20)]
        best, parents = mine.best_scores(v, q, kind)
        rb, rp = np.zeros(len(q), dtype=np.float32), np.zeros(len(q), dtype=np.uint64)
        for rkind in ("list", "bitwise", "tree") if v == 0 else (kind,):
            assert ref.refs_best_scores(h, rkind.encode(), v, q.ctypes.data, len(q), rb.ctypes.data, rp.ctypes.data) == 0
            assert np.array_equal(best.view(np.uint32), rb.view(np.uint32))
        # the parent SET may differ only between entries of exactly equal score
        mm, ms = mine.entries(v)
        score_of = dict(zip(map(int, mm), ms))
        for a, b, s in zip(parents, rp, best):
            assert int(a) == int(b) or score_of[int(a)] == score_of[int(b)] == s


@pytest.mark.parametrize("key,skel", [("hep", None), ("hep_pruned", None), ("f1", "skeleton4_ones.csv"), ("f2", "skeleton4_ones.csv")])
def test_astar_equals_reference_structures(S, ref, pss_files, key, skel):
    """same optimal cost; the same DAG whenever no two cached sets of a variable tie; node counts equal (same heap, same
    heuristic, same expansion order)"""
    mine = S.ScoreCache(pss_files[key])
    h = ref.refs_open(pss_files[key].encode())
    skel_path = os.path.join(DATA, skel) if skel else None
    for kind in ("list", "bitwise"):
        cost, parents, nodes, comps = mine.astar(kind, 2, skel_path)
        rc, rn = C.c_float(), C.c_int()
        rp = np.zeros(mine.p, dtype=np.uint64)
        n = ref.refs_astar(h, kind.encode(), 2, (skel_path or "").encode(), C.byref(rc), rp.ctypes.data, C.byref(rn))
        assert n == comps, ref.refs_last_error(h)
        assert np.float32(cost) == np.float32(rc.value)
        assert nodes == rn.value
        ties = any(len(set(map(float, mine.entries(v)[1]))) != len(mine.entries(v)[1]) for v in range(mine.p))
        if not ties:
            assert np.array_equal(parents, rp)
        # either way both are DAGs of that cost
        for par in (parents, rp):
            tot = np.float32(0)
            scores = [dict(zip(map(int, mine.entries(v)[0]), mine.entries(v)[1])) for v in range(mine.p)]
            assert abs(sum(float(scores[v][int(par[v])]) for v in range(mine.p)) - cost) <= 1e-3 * max(1.0, abs(cost))


@pytest.mark.parametrize("fig,fn,dag", [("Figure_1", "raw_data_8000.csv", "astar_dag_8000.csv"), ("Figure_2", "raw_data_5000.csv", "astar_dag_5000.csv")])
def test_astar_binary_reproduces_published_dag(orc, pss_files, tmp_path, fig, fn, dag):
    """BASELINE configs[1]: `astar` on the cBIC lambda=2 `.pss` of Figure_1/2 writes the reference's published
    astar_dag_*.csv — the same DAG, edge for edge ((i,j) = 1: j -> i), not merely the same equivalence class"""
    exe = os.path.join(ROOT, "urlearning-cpp_b200", "astar")
    net = str(tmp_path / "net")
    subprocess.check_call([exe, pss_files["f1" if fig == "Figure_1" else "f2"], "-k", os.path.join(DATA, "skeleton4_ones.csv"), "-n", net, "--quiet"],
                          stdout=subprocess.DEVNULL)
    got = np.loadtxt(net + ".csv", delimiter=",")
    want = np.loadtxt(os.path.join(DATA, fig, dag), delimiter=",")
    assert np.array_equal(got, want)


def test_library_exports_every_declared_symbol(S):
    lib = S.load_library()
    assert all(hasattr(lib, s) for s in S.ABI_SYMBOLS)
    hdr = open(os.path.join(ROOT, "include", "urlsearch.h")).read()
    assert all(s in hdr for s in S.ABI_SYMBOLS)
