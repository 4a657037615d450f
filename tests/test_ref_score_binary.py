"""The reference's OWN `score` program (score/score_main.cpp with its own main(), compiled from an urlearning-cpp checkout by oracle/ref.mk
over shim Boost headers — program_options that parses, threads that run — and, for cBIC, the minimal Armadillo / mlpack of
oracle/shim_arma) against the oracle's restatement of the whole run (orc_score_file): the header block byte for byte, the
same variables, arities and parent sets, and the scores — bit-identical text for cBIC (same arithmetic on both sides),
to the reference's float32 accumulation noise for BIC / fNML / BDeu.  This pins the option handling (parent limit rule),
the 2-hop neighbour rule of scoringThread, the store rules and the `.pss` writer to the compiled reference."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "ref_score")
DATA = os.path.join(ROOT, "tests", "data")
pytestmark = pytest.mark.skipif(not os.path.exists(REF), reason="oracle/_ref/ref_score not built (reference sources were absent)")


def _blocks(path):
    """header text, {variable name: (arity line, {frozenset(parents): score text})}"""
    text = open(path).read()
    head, _, body = text.partition("\n\n")
    out = {}
    for block in body.split("\n\n"):
        lines = [l for l in block.split("\n") if l != ""]
        if not lines:
            continue
        assert lines[0].startswith("VAR ") and lines[1].startswith("META arity=")
        entries = {}
        for l in lines[2:]:
            assert l.endswith(" ")                      # every line ends with the trailing blank of "%s "
            tok = l.split(" ")[:-1]
            entries[frozenset(tok[1:])] = tok[0]
        assert len(entries) == len(lines) - 2
        out[lines[0][4:]] = (lines[1], entries)
    return head, out


def _run_both(orc, tmp_path, inp, ref_args, **orc_kwargs):
    ref_out, mine = str(tmp_path / "ref.pss"), str(tmp_path / "orc.pss")
    subprocess.check_call([REF, inp, ref_out] + ref_args, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    orc.score_file(inp, mine, **orc_kwargs)
    (hr, br), (hm, bm) = _blocks(ref_out), _blocks(mine)
    assert hr == hm                                      # META pss_version .. ess, byte for byte
    assert list(br) == list(bm)                          # variables in file order
    for name in br:
        assert br[name][0] == bm[name][0]
        assert set(br[name][1]) == set(bm[name][1]), name
    return br, bm


@pytest.mark.parametrize("function,extra,kw,tol", [
    ("BIC", [], {}, 2e-6),
    ("fNML", ["-p", "3"], {"max_parents": 3}, 3e-6),
    ("BDeu", ["-p", "3", "-e", "2"], {"max_parents": 3, "ess": 2.0}, 5e-6)])
def test_hepatitis_whole_run(orc, tmp_path, function, extra, kw, tol):
    inp = os.path.join(DATA, "hepatitis.clean.csv")
    br, bm = _run_both(orc, tmp_path, inp, ["-s", "-f", function] + extra, function=function, has_header=True, **kw)
    n = same_text = 0
    for name in br:
        for ps, s in br[name][1].items():
            a, b = float(s), float(bm[name][1][ps])
            assert abs(a - b) <= tol * abs(a) + 2e-6
            n += 1
            same_text += int(s == bm[name][1][ps])
    assert n == 23200 and same_text > 0      # the reference accumulates in float32 (BDeu: with lgammaf): 8-22 % of its six-decimal texts equal the exact contract's


def test_two_threads_and_a_skeleton(orc, pkg, tmp_path):
    """-t 2 (variable % threadCount striping) and -k: the 2-hop neighbour rule of scoringThread decides the families"""
    import numpy as np
    codes, card, edges, _ = pkg.datagen.discrete_bn(p=9, n=2000, seed=17, window=3, max_indegree=2)
    inp, skel = str(tmp_path / "d.csv"), str(tmp_path / "skel.csv")
    pkg.datagen.write_csv(inp, codes)
    pkg.datagen.write_skeleton_matrix(skel, edges, 9)
    br, bm = _run_both(orc, tmp_path, inp, ["-f", "BIC", "-k", skel, "-t", "2"], function="BIC", skeleton=skel)
    assert sum(len(v[1]) for v in br.values()) > 50


@pytest.mark.parametrize("fig,n", [("Figure_1", 8000), ("Figure_2", 5000)])
def test_cbic_whole_run_is_identical_text(orc, tmp_path, fig, n):
    """cBIC lambda=2 with a skeleton: the reference's BIC_OLS code and the oracle (acceptance as written) print the same lines"""
    inp = os.path.join(DATA, fig, f"raw_data_{n}.csv")
    skel = os.path.join(DATA, "skeleton4_ones.csv")
    br, bm = _run_both(orc, tmp_path, inp, ["-f", "cBIC", "--lambda=2", "-k", skel], function="cBIC", skeleton=skel, lam=2.0, accept_mode=1)
    for name in br:
        assert br[name][1] == bm[name][1], name
