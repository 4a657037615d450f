"""Every discrete score and cBIC at the record counts the API admits, far beyond what the CPU oracle can count.

The data sets are TILED: a seeded base block of L rows (L = 1 000 003, not a multiple of 16) repeated m times, then its
first R rows, n = m L + R, built on the device with torch and uploaded with the ``*_device`` entry points.  Every
contingency table is then known exactly, m counts(base) + counts(base[:, :R]), with the base counts from the oracle
(``orc.bic_counts``), and the reference scores follow from those counts in Python integers:

- BIC: acc = sum q[n_ijk] - sum q[n_ij] with q[c] = 2^23 (float)(c ln c), acc 2^-23 rounded ONCE to float32 (integer
  arithmetic, no detour through a double), minus the float32 penalty;
- fNML: the per-configuration term q[N] + round(2^23 log_regret[N]) with the oracle's regret row;
- BDeu: the 2^-30 fixed-point brackets of bic_kernels.cuh with math.lgamma, within one float32 ulp (device lgamma);
- cBIC: the Gram from the tiled sums in exact integer arithmetic, the_score from the oracle's Gram form.

``test_reference_matches_the_oracle`` ties this count-based reference to the oracle bit for bit on small tiled data.  Each
GPU case first checks free device (and host) memory against its stated peak and skips, naming the numbers, when the
machine cannot hold it: nothing is allocated in the hope that it fits.

- fused cube roots whose child accumulators pass 2^32 nats (bic_root_kernel's warp sums), n = 2^30;
- BIC at n = 2e9, the largest data set ``set_discrete`` takes, and the refusal of 2e9 + 1;
- fNML at n = 2e8 for child arities 2, 3, 4, at the largest n the reference's regret admits (238 609 293), its refusal
  one record above, and the float32-overflow refusal of a wide arity at its exact boundary;
- BDeu at its 1e8 limit with one cell holding nearly every record, and the refusal of 1e8 + 1;
- cBIC at n = 5.5e8, past 65 535 row slices of 8192 records in the Gram kernel's grid.
"""
import math
import os
import time
from fractions import Fraction

import numpy as np
import pytest

from conftest import engine_with_env

BASE_L = 1_000_003
GB = 1e9


# ------------------------------------------------------------------------------------------------ the reference
def _q(c: int) -> int:
    """qlog[c] = (int64) 2^23 (float)(c ln c): the table set_discrete builds (libm's log, as math.log)"""
    return int(math.ldexp(float(np.float32(c * math.log(c))), 23)) if c > 1 else 0


def _f32_once(acc: int, e: int) -> np.float32:
    """acc 2^-e rounded once, to nearest even, to float32 (exact integer arithmetic)"""
    if acc == 0:
        return np.float32(0.0)
    a = abs(acc)
    shift = max(0, a.bit_length() - 24)
    if shift:
        q, rem, half = a >> shift, a & ((1 << shift) - 1), 1 << (shift - 1)
        if rem > half or (rem == half and q & 1):
            q += 1
        a = q
    return np.float32(math.copysign(math.ldexp(a, shift - e), acc))


def _sum_terms(values: np.ndarray, term) -> int:
    """sum of term(x) over an integer array, evaluated once per distinct value"""
    u, k = np.unique(np.asarray(values, dtype=np.int64), return_counts=True)
    return sum(int(c) * term(int(x)) for x, c in zip(u, k))


def _tval(card, v, parents) -> np.float32:
    t = np.float32(card[v] - 1)
    for i in range(len(card)):
        if (parents >> i) & 1:
            t = np.float32(t * np.float32(card[i]))
    return t


def ref_bic(counts: np.ndarray, card, v: int, parents: int, n: int) -> np.float32:
    t = counts.reshape(-1, card[v])
    cells, nij = t.ravel(), t.sum(axis=1)
    acc = _sum_terms(cells[cells > 1], _q) - _sum_terms(nij[nij > 1], _q)
    base = np.float32(math.log(float(n)) / 2)
    return np.float32(_f32_once(acc, 23) - np.float32(_tval(card, v, parents) * base))


def ref_fnml(counts: np.ndarray, rv: int, log_regret: np.ndarray) -> np.float32:
    """log_regret: the oracle's row for arity rv, covering every N_ij of the table"""
    t = counts.reshape(-1, rv)
    cells, nij = t.ravel(), t.sum(axis=1)
    acc = _sum_terms(cells[cells > 1], _q) - _sum_terms(nij[nij > 0], lambda N: _q(N) + round(math.ldexp(float(log_regret[N]), 23)))
    return _f32_once(acc, 23)


def ref_bdeu(counts: np.ndarray, card, v: int, parents: int, ess: float) -> np.float32:
    """bic_kernels.cuh score_configs_bdeu: float32 a_ij, a_ijk and (float) counts, FP64 brackets on the 2^-30 grid"""
    f = np.float32
    rv = card[v]
    nconf = int(np.prod([card[i] for i in range(len(card)) if (parents >> i) & 1], dtype=np.int64))
    a_ij, a_ijk = f(f(ess) / f(nconf)), f(f(ess) / f(nconf * rv))
    lg_ij, lg_ijk = float(f(math.lgamma(float(a_ij)))), float(f(math.lgamma(float(a_ijk))))
    t = counts.reshape(-1, rv)
    cells, nij = t.ravel(), t.sum(axis=1)
    acc = _sum_terms(cells[cells > 0], lambda c: round((float(f(math.lgamma(float(f(a_ijk + f(c)))))) - lg_ijk) * 1073741824.0))
    acc += _sum_terms(nij[nij > 0], lambda N: round((lg_ij - math.lgamma(float(f(a_ij + f(N))))) * 1073741824.0))
    return _f32_once(acc, 30)


def _ulps(a, b):
    a = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a)
    b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)


def _bits(idx):
    return sum(1 << int(i) for i in idx)


def _family(orc, v, nb, p, K):
    om = orc.enumerate_sets(v, nb, p, K)
    return om[orc.canonical_order(om)]


def _tiled_counts(orc, base, card, n, v, parents):
    """the exact table of (v, parents) over the tiling of `base` to n rows, int64"""
    m, R = divmod(n, base.shape[1])
    c = orc.bic_counts(base, card, v, parents).astype(np.int64) * m
    if R:
        c += orc.bic_counts(np.ascontiguousarray(base[:, :R]), card, v, parents)
    return c


def _stored(om, scores):
    """score_calculator.cpp's store rule (the empty set below 1, every other set below 0), canonical order kept"""
    keep = np.array([(s < 1) if m == 0 else (s < 0) for m, s in zip(om, scores)])
    return om[keep], np.asarray(scores, dtype=np.float32)[keep]


# ------------------------------------------------------------------------------------------------ device data
def _need(device_gb: float, host_gb: float = 0.0):
    """skip, naming the numbers, when the device (or the host) cannot hold the case's stated peak"""
    import torch
    free, total = torch.cuda.mem_get_info()
    if free < device_gb * GB:
        pytest.skip(f"needs {device_gb:.0f} GB of free device memory; {free / GB:.1f} GB of {total / GB:.1f} GB are free")
    if host_gb:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
        if avail < host_gb * GB:
            pytest.skip(f"needs {host_gb:.0f} GB of free host memory; {avail / GB:.1f} GB are free")


def _device_tiles(base: np.ndarray, n: int):
    """[p, n] device tensor: `base` ([p, L]) repeated m times, then base[:, :R]; n = m L + R"""
    import torch
    p, L = base.shape
    m, R = divmod(n, L)
    b = torch.from_numpy(np.ascontiguousarray(base)).cuda()
    t = torch.empty((p, n), dtype=b.dtype, device="cuda")
    if m:
        t[:, :m * L].view(p, m, L).copy_(b.unsqueeze(1).expand(p, m, L))
    if R:
        t[:, m * L:].copy_(b[:, :R])
    del b
    torch.cuda.synchronize()
    return t


def _upload_discrete(eng, base, n, card):
    """tile `base` to n rows on the device ([p, n]: the row pitch is n), upload, free the tensor (the engine keeps a copy)"""
    import torch
    t = _device_tiles(base, n)
    eng.set_discrete_device(t.data_ptr(), n, base.shape[0], card)
    del t
    torch.cuda.empty_cache()


def _peak_gb():
    import torch
    return torch.cuda.max_memory_allocated() / GB


class _Clock:
    def __init__(self, name):
        self.name, self.t0 = name, time.perf_counter()

    def lap(self, what):
        print(f"[{self.name}] {what}: {time.perf_counter() - self.t0:.1f} s", flush=True)


def _fetch(eng, v, nb, K, st, lam=0.0):
    res = eng.score_variable(v, nb, K, st, lam=lam)
    masks, scores = res.fetch()
    scored = res.scored()
    res.free()
    return masks[:, 0], scores, scored


def _check_bits(what, om, want, masks, scores, scored):
    """the stored list (masks, scores) equals the reference's, bit for bit; a mismatch names the sets a wrong score dropped"""
    sm, ss = _stored(om, want)
    assert scored == len(om), what
    got = dict(zip((int(m) for m in masks), scores))
    missing = [int(m) for m in sm if int(m) not in got]
    assert [int(m) for m in masks] == [int(m) for m in sm], f"{what}: {len(missing)} of {len(sm)} stored sets missing, first {missing[:4]}"
    bad = np.flatnonzero(scores.view(np.uint32) != ss.view(np.uint32))
    assert len(bad) == 0, (f"{what}: {len(bad)} of {len(ss)} scores differ; first: set {int(sm[bad[0]]):#x} "
                           f"got {float(scores[bad[0]])!r} want {float(ss[bad[0]])!r} "
                           f"(difference {float(scores[bad[0]]) - float(ss[bad[0]]):.6g} nats = {(float(scores[bad[0]]) - float(ss[bad[0]])) / 2 ** 33:.4f} x 2^33)")


# ------------------------------------------------------------------------------------------------ 0. the reference itself
def test_reference_matches_the_oracle(pkg, orc):
    """the count-based reference on small tiled data (m = 3 copies of a 4 999-row block and a 1 234-row tail): the tiled
    counts equal the oracle's counts of the whole data set, and BIC and fNML equal the oracle bit for bit, BDeu within one
    float32 ulp (math.lgamma against glibc's), for every set of the families of a 256-ary child over skewed parents, of
    a constant column and of two small children"""
    rng = np.random.default_rng(12)
    L, m, R = 4999, 3, 1234
    card = [256, 8, 8, 3, 4, 1, 2]
    base = np.zeros((len(card), L), dtype=np.uint8)
    base[0] = rng.integers(0, 256, L)
    for i in (1, 2):
        base[i] = np.where(rng.random(L) < 0.05, rng.integers(1, 8, L), 0)
    base[3] = rng.integers(0, 3, L)
    base[4] = (base[3] + (rng.random(L) < 0.3) * rng.integers(0, 4, L)) % 4
    base[6] = np.where(rng.random(L) < 0.8, base[3] % 2, rng.integers(0, 2, L))
    n = m * L + R
    full = np.concatenate([np.tile(base, (1, m)), base[:, :R]], axis=1)
    p = len(card)
    for v in (0, 4, 5, 6):
        nb = ((1 << p) - 1) & ~(1 << v)
        om = _family(orc, v, nb, p, 3)
        lr = orc.log_regret(n + 1, card[v])
        bic = orc.bic_score_many(full, card, v, om)
        fnml = orc.fnml_score_many(full, card, v, om)
        bdeu = orc.bdeu_score_many(full, card, v, om, ess=1.0)
        for i, s in enumerate(om):
            counts = _tiled_counts(orc, base, card, n, v, int(s))
            assert np.array_equal(counts, orc.bic_counts(full, card, v, int(s))), (v, int(s))
            assert ref_bic(counts, card, v, int(s), n).view(np.uint32) == bic[i].view(np.uint32), (v, int(s))
            if np.all(np.isfinite(lr)):   # C(N, 256) overflows float32 from N = 16 231 on: the engine refuses that child
                assert ref_fnml(counts, card[v], lr).view(np.uint32) == fnml[i].view(np.uint32), (v, int(s))
            assert _ulps(ref_bdeu(counts, card, v, int(s), 1.0), bdeu[i]) <= 1, (v, int(s))


def test_single_rounding_helper():
    """_f32_once rounds the exact value once: acc = 2^53 + 2^29 + 1 lies just above the midpoint between two float32 values
    (2^53 and 2^53 + 2^30), so it rounds up; through a double it first becomes the midpoint and then ties to even (down)"""
    acc = (1 << 53) + (1 << 29) + 1
    assert float(_f32_once(acc, 0)) == float((1 << 53) + (1 << 30))
    assert float(np.float32(float(acc))) == float(1 << 53)
    assert float(_f32_once(-acc, 23)) == -float((1 << 53) + (1 << 30)) / 2 ** 23
    for a in (1, 3, (1 << 24) - 1, (1 << 24) + 1, (1 << 25) + 3, 123456789123, -987654321987):
        assert _f32_once(a, 7) == np.float32(a / 128.0), a     # below 2^53 the double is exact: one rounding either way


# ------------------------------------------------------------------------------------------------ 1. fused roots past 2^32 nats
# Child: arity 256, uniform.  Seven candidates of arity 8, each 0 on all but ~0.1 % of the rows: ~99.3 % of the records sit
# in the all-zero parent configuration.  Packed rows take 8-bit fields ((7 + 1) * 8 = 64 bits).  With K = 3 the cube path
# roots the family at layer 4 = K + 1 (fused roots score their children, layer 3), 20 roots of 256 * 8^4 cells in 64 slices
# each; the fused ones have runs of 1 or 2 low digits.  Thread 0 (warp 0) of the slice holding the all-zero configuration
# owns configuration 0 of every child, n_ij ~ 1.07e9 rows with H(child | config) ~ ln 256: its exact partial is
# ~2^23 * 5.9e9 > 2^55, i.e. above 2^32 nats.
C1_N = 1 << 30
C1_CARD = [256] + [8] * 7
C1_K = 3
C1_NB = _bits(range(1, 8))


def _case1_base():
    rng = np.random.default_rng(2 ** 30)
    base = np.zeros((len(C1_CARD), BASE_L), dtype=np.uint8)
    base[0] = rng.integers(0, 256, BASE_L)
    for i in range(1, 8):
        base[i] = np.where(rng.random(BASE_L) < 0.001, rng.integers(1, 8, BASE_L), 0)
    return base


@pytest.mark.gpu
def test_fused_roots_past_2_32_nats(pkg, orc):
    """BIC of a family whose fused cube roots sum child accumulators above 2^55 (2^32 nats) in one warp: the default
    engine, URLGPU_FUSE_ROOTS=0, URLGPU_SLICE_COUNT=0 and URLGPU_BIC_MODE=direct give the reference's bits and stored list.
    The routes are witnessed: fused roots write fewer K1 bytes than plain ones, the slice route launches more count kernels
    than the global-atomic route.  Contingency of the widest set against the exact counts.  Peak: ~50 GB of device memory
    (codes and qlog 8.6 GB each, packed rows and keys 13 GB, cached per engine), 9 GB of host memory"""
    import torch
    _need(64, 12)
    clk = _Clock("fused roots")
    base = _case1_base()
    om = _family(orc, 0, C1_NB, len(C1_CARD), C1_K)
    counts = {int(s): _tiled_counts(orc, base, C1_CARD, C1_N, 0, int(s)) for s in om}
    want = np.array([ref_bic(counts[int(s)], C1_CARD, 0, int(s), C1_N) for s in om], dtype=np.float32)
    zero = counts[_bits([1, 2, 3])].reshape(-1, 256)[0].sum()
    assert zero > 1.06e9   # the all-zero configuration: 2^32 / ln 256 = 7.75e8 records are enough to pass 2^55
    clk.lap("reference")
    torch.cuda.reset_peak_memory_stats()
    owner = pkg.Engine(0)
    _upload_discrete(owner, base, C1_N, C1_CARD)
    clk.lap("upload")
    widest = _bits([1, 2, 3])
    got = owner.contingency(0, widest, 256 * 8 ** 3)
    assert np.array_equal(got, counts[widest])
    clk.lap("contingency")
    stats = {}
    engines = [("default", owner)] + [(name, engine_with_env(pkg, env)) for name, env in (
        ("fuse=0", {"URLGPU_FUSE_ROOTS": "0"}), ("slice=0", {"URLGPU_SLICE_COUNT": "0"}), ("direct", {"URLGPU_BIC_MODE": "direct"}))]
    try:
        for name, eng in engines:
            if eng is not owner:
                eng.share_discrete(owner)
            eng.reset_stats()
            masks, scores, scored = _fetch(eng, 0, C1_NB, C1_K, pkg.BIC)
            stats[name] = eng.stats()
            clk.lap(f"score_variable {name}")
            _check_bits(name, om, want, masks, scores, scored)
            if eng is not owner:
                eng.close()
    finally:
        for name, eng in engines:
            eng.close()
    print(f"[fused roots] device peak of the torch allocator {_peak_gb():.1f} GB; free now {torch.cuda.mem_get_info()[0] / GB:.1f} GB")
    assert 0 < stats["default"]["k1_bytes_written"] < stats["fuse=0"]["k1_bytes_written"], stats
    assert stats["default"]["launches_count"] > stats["slice=0"]["launches_count"], stats


# ------------------------------------------------------------------------------------------------ 2. BIC at 2e9 records
C2_N = 2_000_000_000
C2_CARD = [64, 16, 16, 16]


@pytest.mark.gpu
def test_bic_at_2e9_records_and_the_refusal_above(pkg, orc):
    """n = 2e9 (qlog reaches 2e9 + 1 entries; the empty set looks up q[2e9]): a family of 8 sets through score_variable,
    the contingency table of its widest set (262 144 cells, the global tier) and one score_one of that set, against the
    tiled reference.  Then a real device buffer of 2e9 + 1 bytes: refused before anything is read.  Peak: ~33 GB of device
    memory (codes 8 GB, qlog 16 GB, the tiling tensor 8 GB), 17 GB of host memory (set_discrete's qlog)"""
    import torch
    _need(40, 20)
    clk = _Clock("2e9")
    rng = np.random.default_rng(2_000_000_000)
    base = np.zeros((4, BASE_L), dtype=np.uint8)
    base[1:] = rng.integers(0, 16, (3, BASE_L))
    base[0] = (base[1].astype(np.int64) * 5 + base[2] + np.where(rng.random(BASE_L) < 0.5, rng.integers(0, 64, BASE_L), 0)) % 64
    nb = _bits([1, 2, 3])
    om = _family(orc, 0, nb, 4, 3)
    counts = {int(s): _tiled_counts(orc, base, C2_CARD, C2_N, 0, int(s)) for s in om}
    want = np.array([ref_bic(counts[int(s)], C2_CARD, 0, int(s), C2_N) for s in om], dtype=np.float32)
    clk.lap("reference")
    torch.cuda.reset_peak_memory_stats()
    eng = pkg.Engine(0)
    try:
        _upload_discrete(eng, base, C2_N, C2_CARD)
        clk.lap("upload")
        _check_bits("2e9 score_variable", om, want, *_fetch(eng, 0, nb, 3, pkg.BIC))
        clk.lap("score_variable")
        got = eng.contingency(0, nb, 64 * 16 ** 3)
        assert np.array_equal(got, counts[nb]) and int(got.sum()) == C2_N
        clk.lap("contingency")
        s, _ = eng.score_one(0, nb, pkg.BIC)
        assert s.view(np.uint32) == want[-1].view(np.uint32), (float(s), float(want[-1]))
        clk.lap("score_one")
    finally:
        eng.close()
    print(f"[2e9] device peak of the torch allocator {_peak_gb():.1f} GB")
    torch.cuda.empty_cache()
    buf = torch.zeros(C2_N + 1, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    eng = pkg.Engine(0)
    try:
        with pytest.raises(pkg.UrlGpuError, match="more than 2e9 records"):
            eng.set_discrete_device(buf.data_ptr(), C2_N + 1, 1, [2])
    finally:
        eng.close()
        del buf
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ 3. fNML
FNML_MAX_N = 238_609_293      # 9 (n + 1) <= INT_MAX: the regret table covers N = 0..n+1 and r2 computes 9 * N in int


def _fnml_base(card, seed):
    rng = np.random.default_rng(seed)
    base = np.zeros((len(card), BASE_L), dtype=np.uint8)
    for i, r in enumerate(card):
        if i >= 3 and r > 1:
            base[i] = rng.integers(0, r, BASE_L)
    for i in range(3):   # the children lean on the two 256-ary parents
        if card[i] > 1:
            dep = (base[3].astype(np.int64) + 3 * base[4]) % card[i]
            base[i] = np.where(rng.random(BASE_L) < 0.6, dep, rng.integers(0, card[i], BASE_L))
    return base


def _check_fnml(pkg, orc, eng, base, card, n, v, nb, K, what):
    om = _family(orc, v, nb, len(card), K)
    lr = orc.log_regret(n, card[v])
    want = np.array([ref_fnml(_tiled_counts(orc, base, card, n, v, int(s)), card[v], lr) for s in om], dtype=np.float32)
    del lr
    _check_bits(what, om, want, *_fetch(eng, v, nb, K, pkg.FNML))
    return want


@pytest.mark.gpu
def test_fnml_at_2e8_records_and_the_regret_limit(pkg, orc):
    """n = 2e8: children of arity 2, 3 and 4 under two 256-ary parents (N up to 2e8: the Szpankowski rows five orders of
    magnitude past the tabulated N <= 1000), bit-exact.  n = 238 609 293, the largest n the reference's regret admits:
    bit-exact for an arity-2 child.  One record more: refused with the integer-overflow limit, while a constant child
    (C(N, 1) = 1) still scores.  Peak: ~5 GB of device memory, ~4 GB of host memory"""
    import torch
    _need(8, 8)
    clk = _Clock("fNML")
    card = [2, 3, 4, 256, 256, 1]
    base = _fnml_base(card, 200)
    nb = _bits([3, 4])
    eng = pkg.Engine(0)
    try:
        _upload_discrete(eng, base, 200_000_000, card)
        for v in (0, 1, 2):
            _check_fnml(pkg, orc, eng, base, card, 200_000_000, v, nb, 2, f"n=2e8 arity {card[v]}")
            clk.lap(f"n = 2e8, arity {card[v]}")
        _upload_discrete(eng, base, FNML_MAX_N, card)
        _check_fnml(pkg, orc, eng, base, card, FNML_MAX_N, 0, nb, 2, f"n={FNML_MAX_N} arity 2")
        clk.lap(f"n = {FNML_MAX_N}")
        _upload_discrete(eng, base, FNML_MAX_N + 1, card)
        with pytest.raises(pkg.UrlGpuError, match=f"fNML: more than {FNML_MAX_N} records .*9 \\* N in int, which overflows at N = 238609295"):
            eng.score_variable(0, nb, 2, pkg.FNML)
        with pytest.raises(pkg.UrlGpuError, match=f"more than {FNML_MAX_N} records"):
            eng.score_one(1, _bits([3]), pkg.FNML)
        want = _check_fnml(pkg, orc, eng, base, card, FNML_MAX_N + 1, 5, nb, 2, "constant child")
        assert np.all(want == 0)
        clk.lap(f"n = {FNML_MAX_N + 1}")
    finally:
        eng.close()
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_fnml_float_overflow_refusal_at_its_boundary(pkg, orc):
    """a child of arity 16: C(N, 16) overflows float32 from N* on, N* found in the oracle's regret row (790 314 with the
    reference's float recurrence).  n = N* - 2 (the table's last entry is N* - 1) is accepted and bit-exact; n = N* - 1
    is refused, naming N*"""
    lr = orc.log_regret(1_000_000, 16)
    bad = np.flatnonzero(~np.isfinite(lr))
    assert len(bad), "C(N, 16) stays finite up to 1e6"
    nstar = int(bad[0])
    assert np.all(np.isfinite(lr[:nstar]))
    card = [16, 4, 4]
    rng = np.random.default_rng(16)
    base = np.zeros((3, BASE_L), dtype=np.uint8)
    base[1:] = rng.integers(0, 4, (2, BASE_L))
    base[0] = np.where(rng.random(BASE_L) < 0.5, (base[1] * 4 + base[2]).astype(np.int64), rng.integers(0, 16, BASE_L))
    nb = _bits([1, 2])
    eng = pkg.Engine(0)
    try:
        _upload_discrete(eng, base, nstar - 2, card)
        _check_fnml(pkg, orc, eng, base, card, nstar - 2, 0, nb, 2, f"n = N* - 2 = {nstar - 2}")
        _upload_discrete(eng, base, nstar - 1, card)
        with pytest.raises(pkg.UrlGpuError, match=f"arity 16 overflows float32 at N = {nstar} "):
            eng.score_variable(0, nb, 2, pkg.FNML)
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------ 4. BDeu
BDEU_MAX_N = 100_000_000


@pytest.mark.gpu
def test_bdeu_at_1e8_records_and_the_refusal_above(pkg, orc):
    """n = 1e8 exactly, BDeu's limit: one cell (all zero) holds ~99.9 % of the records, so its lgamma brackets are the
    largest the fixed-point accumulator meets (|acc| > 2^53: the single final rounding matters), and counts above 2^24
    that float32 cannot hold go through the kernel's (float) conversion.  Within one float32 ulp of the reference,
    identical stored lists, ess 1 and 10.  1e8 + 1 records are refused.  Peak: ~1 GB of device memory"""
    import torch
    _need(4)
    clk = _Clock("BDeu")
    card = [2, 3, 2, 5]
    rng = np.random.default_rng(100_000_000)
    base = np.zeros((4, BASE_L), dtype=np.uint8)
    for i, r in enumerate(card):
        base[i] = np.where(rng.random(BASE_L) < 0.0003, rng.integers(1, r, BASE_L), 0)
    nb = _bits([1, 2, 3])
    om = _family(orc, 0, nb, 4, 3)
    counts = {int(s): _tiled_counts(orc, base, card, BDEU_MAX_N, 0, int(s)) for s in om}
    full = counts[nb]
    assert full[0] > 0.998 * BDEU_MAX_N
    assert any(float(np.float32(c)) != c for t in counts.values() for c in t.tolist()), "no count that float32 rounds"
    eng = pkg.Engine(0)
    try:
        _upload_discrete(eng, base, BDEU_MAX_N, card)
        got = eng.contingency(0, nb, int(np.prod(card)))
        assert np.array_equal(got, full)
        for ess in (1.0, 10.0):
            want = np.array([ref_bdeu(counts[int(s)], card, 0, int(s), ess) for s in om], dtype=np.float32)
            masks, scores, scored = _fetch(eng, 0, nb, 3, pkg.BDEU, lam=ess)
            sm, ss = _stored(om, want)
            assert scored == len(om)
            assert [int(m) for m in masks] == [int(m) for m in sm], ess
            assert _ulps(scores, ss).max() <= 1, (ess, scores, ss)
            clk.lap(f"ess {ess}")
        _upload_discrete(eng, base, BDEU_MAX_N + 1, card)
        with pytest.raises(pkg.UrlGpuError, match="more than 1e8 records"):
            eng.score_variable(0, nb, 3, pkg.BDEU, lam=1.0)
        with pytest.raises(pkg.UrlGpuError, match="more than 1e8 records"):
            eng.score_one(0, _bits([1]), pkg.BDEU, lam=1.0)
    finally:
        eng.close()
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ 5. cBIC Gram slices
C5_N = 550_000_000            # > 65 535 * 8192 = 536 862 720: more slices of 8192 records than gridDim.y holds
C5_LAM = 2.0


def _cbic_base():
    """integer-valued doubles (every sum below is exact in int64), correlated, one column far from zero"""
    rng = np.random.default_rng(550)
    x = np.zeros((3, BASE_L), dtype=np.int64)
    x[0] = rng.integers(-50, 51, BASE_L)
    x[1] = 2 * x[0] + rng.integers(-30, 31, BASE_L)
    x[2] = x[0] - x[1] + rng.integers(-20, 21, BASE_L) + 1000
    return x


def _gram_from_tiles(x: np.ndarray, n: int) -> np.ndarray:
    """the standardised Gram (mean, sample std with n - 1) of the tiling of integer data x, in exact rationals"""
    m, R = divmod(n, x.shape[1])
    p = x.shape[0]
    tail = x[:, :R]
    s = [m * int(x[a].sum()) + int(tail[a].sum()) for a in range(p)]
    ss = [[m * int(x[a] @ x[b]) + int(tail[a] @ tail[b]) for b in range(p)] for a in range(p)]
    c = [[Fraction(ss[a][b]) - Fraction(s[a] * s[b], n) for b in range(p)] for a in range(p)]
    g = np.zeros((p, p))
    for a in range(p):
        for b in range(p):
            g[a, b] = float(c[a][b] * (n - 1)) / math.sqrt(float(c[a][a]) * float(c[b][b]))
    return g


@pytest.mark.gpu
def test_cbic_gram_past_65535_slices(pkg, orc):
    """n = 5.5e8, p = 3, tiled doubles through set_continuous_device: the Gram within 1e-12 n of the exact Gram of the
    tiles, and every set's the_score within 1e-9 relative of the oracle's Gram form on it; the cache (no acceptance)
    equal to score_one bit for bit.  Peak: ~27 GB of device memory (the tensor and the engine's padded copy, 13.2 GB each)"""
    import torch
    _need(32)
    clk = _Clock("cBIC")
    x = _cbic_base()
    ref = _gram_from_tiles(x, C5_N)
    torch.cuda.reset_peak_memory_stats()
    t = _device_tiles(x.astype(np.float64), C5_N)
    eng = pkg.Engine(0)
    try:
        eng.set_continuous_device(t.data_ptr(), C5_N, 3)
        del t
        torch.cuda.empty_cache()
        clk.lap("upload + Gram")
        g = eng.gram()
        assert np.array_equal(g, g.T)
        assert np.max(np.abs(g - ref)) <= 1e-12 * C5_N, np.max(np.abs(g - ref))
        for v in range(3):
            nb = 7 & ~(1 << v)
            om = _family(orc, v, nb, 3, 2)
            res = eng.score_variable(v, nb, 2, pkg.CBIC, lam=C5_LAM, flags=pkg.CBIC_NO_ACCEPT)
            cm, cs = res.fetch()
            res.free()
            assert [int(m) for m in cm[:, 0]] == [int(m) for m in om], v
            for i, s in enumerate(om):
                want = orc.cbic_gram(ref, C5_N, v, int(s), C5_LAM)
                f, ts = eng.score_one(v, int(s), pkg.CBIC, C5_LAM)
                assert abs(ts - want) <= 1e-9 * max(1.0, abs(want)), (v, int(s), ts, want)
                assert f.view(np.uint32) == cs[i].view(np.uint32), (v, int(s))
        clk.lap("scores")
    finally:
        eng.close()
    print(f"[cBIC] device peak of the torch allocator {_peak_gb():.1f} GB")
