"""urlearning-cpp_b200 — B200-native local-score engine for URLearning (Python binding of liburlgpu.so).

This module is a thin ctypes binding of the C ABI declared in ``include/urlgpu.h``; all computation happens in
the hand-written sm_100a kernels under ``csrc/``.  There is no CPU fallback: importing works anywhere (so the
symbol table can be checked without a GPU) but creating an :class:`Engine` raises :class:`UrlGpuError` when no
Blackwell device is usable or the shared library has not been built.

Host-side helpers mirror the reference's driver logic (paths relative to /root/reference/urlearning/):

* :func:`two_hop_neighbors`      score/score_main.cpp:145-155
* :func:`effective_max_parents`  score/score_main.cpp:296-304
"""
from __future__ import annotations

import ctypes as C
import math
import os
import weakref
from typing import Iterable, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liburlgpu.so")

BIC, CBIC, FNML, BDEU = 0, 1, 2, 3   # BDEU: the `lam` argument of the scoring calls is the equivalent sample size
KEEP_ALL, PRUNE_DOMINATED, CBIC_NO_ACCEPT, CBIC_ACCEPT_LITERAL = 0, 2, 4, 8

# every symbol include/urlgpu.h declares (tests check the built library exports all of them)
ABI_SYMBOLS = [
    "urlgpu_create", "urlgpu_destroy", "urlgpu_last_error", "urlgpu_device_count", "urlgpu_set_stream",
    "urlgpu_synchronize", "urlgpu_set_discrete", "urlgpu_set_discrete_device", "urlgpu_share_discrete", "urlgpu_set_continuous",
    "urlgpu_set_continuous_device", "urlgpu_shard_begin", "urlgpu_shard_moments", "urlgpu_shard_finish", "urlgpu_get_gram", "urlgpu_set_gram", "urlgpu_score_variable",
    "urlgpu_result_prefetch", "urlgpu_result_count", "urlgpu_result_scored", "urlgpu_result_fetch", "urlgpu_result_free",
    "urlgpu_host_alloc", "urlgpu_host_free",
    "urlgpu_score_one", "urlgpu_score_sets", "urlgpu_contingency", "urlgpu_prune", "urlgpu_stats_reset", "urlgpu_stats_get",
    "urlgpu_stats_enable_timing", "urlgpu_probe_fp64", "urlgpu_family_size", "urlgpu_score_range", "urlgpu_result_from_scores", "urlgpu_score_part",
    "urlgpu_spg_build", "urlgpu_spg_query", "urlgpu_spg_free",
    "urlgpu_peer_alloc", "urlgpu_peer_open", "urlgpu_peer_close", "urlgpu_peer_free",
    "urlgpu_result_fetch_device", "urlgpu_copy_to_host", "urlgpu_order_search",
    "urlgpu_order_search_layered", "urlgpu_order_local_search", "urlgpu_order_local_search_sparse",
]


class UrlGpuError(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [
        ("launches_total", C.c_uint64), ("launches_count", C.c_uint64), ("launches_cube", C.c_uint64),
        ("launches_cbic", C.c_uint64), ("launches_accept", C.c_uint64), ("launches_prune", C.c_uint64),
        ("launches_other", C.c_uint64),
        ("ms_count", C.c_double), ("ms_cube", C.c_double), ("ms_cbic", C.c_double), ("ms_accept", C.c_double),
        ("ms_prune", C.c_double), ("ms_gram", C.c_double),
        ("sets_scored", C.c_uint64), ("algorithmic_bytes", C.c_double), ("algorithmic_flops", C.c_double), ("gram_flops", C.c_double),
        ("launches_tree", C.c_uint64), ("ms_tree", C.c_double), ("k1_bytes_read", C.c_double), ("k1_bytes_written", C.c_double),
        ("ms_standardise", C.c_double), ("table16_fallbacks", C.c_uint64), ("ms_order_tables", C.c_double),
        ("ms_order_layers", C.c_double),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def load_library():
    """Load liburlgpu.so (built in-tree by ``__graft_entry__.build()`` / ``make``).  Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise UrlGpuError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64
    P = C.POINTER
    lib.urlgpu_create.argtypes = [P(vp), i32]
    lib.urlgpu_destroy.argtypes = [vp]
    lib.urlgpu_last_error.argtypes = [vp]
    lib.urlgpu_last_error.restype = C.c_char_p
    lib.urlgpu_device_count.argtypes = []
    lib.urlgpu_set_stream.argtypes = [vp, vp]
    lib.urlgpu_synchronize.argtypes = [vp]
    lib.urlgpu_set_discrete.argtypes = [vp, vp, i64, i32, vp]
    lib.urlgpu_set_discrete_device.argtypes = [vp, vp, i64, i32, vp]
    lib.urlgpu_share_discrete.argtypes = [vp, vp]
    lib.urlgpu_set_continuous.argtypes = [vp, vp, i64, i32]
    lib.urlgpu_set_continuous_device.argtypes = [vp, vp, i64, i32]
    lib.urlgpu_shard_begin.argtypes = [vp, vp, i64, i32, i32]
    lib.urlgpu_shard_moments.argtypes = [vp, vp, vp, vp]
    lib.urlgpu_shard_finish.argtypes = [vp, vp, vp, i64]
    lib.urlgpu_get_gram.argtypes = [vp, vp]
    lib.urlgpu_set_gram.argtypes = [vp, vp, i64, i32]
    lib.urlgpu_score_variable.argtypes = [vp, i32, vp, i32, i32, i32, C.c_double, C.c_uint, P(vp)]
    lib.urlgpu_result_prefetch.argtypes = [vp]
    lib.urlgpu_result_count.argtypes = [vp, P(u64)]
    lib.urlgpu_result_scored.argtypes = [vp, P(u64)]
    lib.urlgpu_result_fetch.argtypes = [vp, u64, u64, vp, vp]
    lib.urlgpu_result_free.argtypes = [vp]
    lib.urlgpu_host_alloc.argtypes = [u64]
    lib.urlgpu_host_free.argtypes = [vp]
    lib.urlgpu_score_one.argtypes = [vp, i32, vp, i32, i32, C.c_double, P(C.c_float), P(C.c_double)]
    lib.urlgpu_score_sets.argtypes = [vp, u64, vp, vp, i32, i32, C.c_double, vp, vp]
    lib.urlgpu_contingency.argtypes = [vp, i32, vp, i32, vp, i64]
    lib.urlgpu_prune.argtypes = [vp, vp, vp, u64, i32, vp]
    lib.urlgpu_stats_reset.argtypes = [vp]
    lib.urlgpu_stats_get.argtypes = [vp, P(Stats)]
    lib.urlgpu_stats_enable_timing.argtypes = [vp, i32]
    lib.urlgpu_probe_fp64.argtypes = [vp, P(C.c_double), P(C.c_double)]
    lib.urlgpu_spg_build.argtypes = [vp, vp, vp, u64, i32, i32, P(vp)]
    lib.urlgpu_spg_query.argtypes = [vp, vp, u64, vp, vp, vp]
    lib.urlgpu_spg_free.argtypes = [vp]
    lib.urlgpu_result_fetch_device.argtypes = [vp, u64, u64, i32, i32, vp, vp]
    lib.urlgpu_copy_to_host.argtypes = [vp, vp, vp, u64]
    lib.urlgpu_peer_alloc.argtypes = [vp, u64, P(vp), vp]
    lib.urlgpu_peer_open.argtypes = [vp, vp, P(vp)]
    lib.urlgpu_peer_close.argtypes = [vp, vp]
    lib.urlgpu_peer_free.argtypes = [vp, vp]
    lib.urlgpu_family_size.argtypes = [vp, i32, vp, i32, i32, i32, P(u64)]
    lib.urlgpu_score_range.argtypes = [vp, i32, vp, i32, i32, i32, C.c_double, u64, u64, vp, i32]
    lib.urlgpu_score_part.argtypes = [vp, i32, vp, i32, i32, i32, C.c_double, i32, i32, vp, i32]
    lib.urlgpu_result_from_scores.argtypes = [vp, i32, vp, i32, i32, i32, vp, u64, i32, C.c_uint, P(vp)]
    lib.urlgpu_order_search.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, P(C.c_float), vp, vp]
    lib.urlgpu_order_search_layered.argtypes = lib.urlgpu_order_search.argtypes
    lib.urlgpu_order_local_search.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, C.c_uint32, u64, P(C.c_float), vp, vp, vp, vp]
    lib.urlgpu_order_local_search_sparse.argtypes = lib.urlgpu_order_local_search.argtypes
    for name in ABI_SYMBOLS:
        if name not in ("urlgpu_last_error", "urlgpu_host_alloc", "urlgpu_host_free"):
            getattr(lib, name).restype = C.c_int
    lib.urlgpu_host_alloc.restype = vp
    lib.urlgpu_host_free.restype = None
    _lib = lib
    return lib


# ------------------------------------------------------------------------------------------ host-side mirrors

def mask_words_for(p: int) -> int:
    return max(1, (p + 63) // 64)


def mask_to_words(mask: int, words: int) -> np.ndarray:
    return np.array([(mask >> (64 * w)) & 0xFFFFFFFFFFFFFFFF for w in range(words)], dtype=np.uint64)


def words_to_mask(row: Sequence[int]) -> int:
    m = 0
    for w, x in enumerate(row):
        m |= int(x) << (64 * w)
    return m


def two_hop_neighbors(edges: Sequence[int] | None, p: int, v: int) -> int:
    """score_main.cpp:145-155: N(v) | U_{j in N(v), j != v} N(j); ``edges=None`` = no skeleton (all ones)."""
    allbits = (1 << p) - 1
    nb = (lambda i: allbits) if edges is None else (lambda i: int(edges[i]))
    orig = nb(v)
    out = orig
    for j in range(p):
        if (orig >> j) & 1 and j != v:
            out |= nb(j)
    return out


def table_bytes(offsets: np.ndarray, masks: np.ndarray, comp: np.ndarray) -> int:
    """the bytes of urlgpu_order_local_search's best-parent tables, the sum of 4 2^c_v over the component's variables, where c_v
    is the popcount of the union of v's qualifying parent sets (those inside the component).  offsets [p + 1], masks [n, words]
    and comp [words] as order_local_search passes them to the C ABI"""
    inside = ~np.any(masks & ~comp, axis=1)
    total = 0
    for v in range(len(offsets) - 1):
        if not (int(comp[v >> 6]) >> (v & 63)) & 1:
            continue
        rows = masks[int(offsets[v]):int(offsets[v + 1])][inside[int(offsets[v]):int(offsets[v + 1])]]
        total += 4 << (int(np.bitwise_count(np.bitwise_or.reduce(rows, axis=0)).sum()) if len(rows) else 0)
    return total


# order_local_search takes the table form while its tables take at most this many bytes, the sparse form above (DESIGN §5).
# A variable with c_v > 32, which the table form refuses, alone needs 32 GiB.
TABLE_MAX_BYTES = 4 << 30


def components(p: int, edges: Sequence[int] | None) -> list[int]:
    """urlsearch::components (host/search_host.hpp:435-456, skeleton.cpp:187-230): the connected components of the skeleton
    as variable masks, in the order of their smallest variable; ``edges=None`` = one component of all p variables."""
    if edges is None:
        return [(1 << p) - 1]
    out, visited = [], 0
    for v in range(p):
        if (visited >> v) & 1:
            continue
        comp, stack = 0, [v]
        while stack:
            u = stack.pop()
            if (visited >> u) & 1:
                continue
            visited |= 1 << u
            comp |= 1 << u
            stack.extend(i for i in range(p - 1, -1, -1) if (int(edges[u]) >> i) & 1 and not (visited >> i) & 1)
        out.append(comp)
    return out


def effective_max_parents(max_parents: int, p: int, n_records: int, is_bic: bool) -> int:
    """score_main.cpp:296-304 (the BIC cap uses integer 2*N and natural logs, truncated)."""
    if max_parents > p or max_parents < 1:
        max_parents = p - 1
    if is_bic:
        cap = int(math.log((2 * n_records) / math.log(n_records)))
        max_parents = min(max_parents, cap)
    return max_parents


# ------------------------------------------------------------------------------------------ engine

class Result:
    """One variable's score cache on the device (the reference's per-variable FloatMap)."""

    def __init__(self, eng: "Engine", handle, words: int):
        self._eng, self._h, self.words = eng, handle, words
        eng._live[id(self)] = weakref.ref(self)   # Engine.close() frees what is still alive: a result must not outlive its context

    def prefetch(self) -> "Result":
        """enqueue the on-device compaction behind the scoring kernels (no host sync); fetch() then only waits for it"""
        self._eng._check(self._eng.lib.urlgpu_result_prefetch(self._h))
        return self

    def count(self) -> int:
        n = C.c_uint64()
        self._eng._check(self._eng.lib.urlgpu_result_count(self._h, C.byref(n)))
        return n.value

    def scored(self) -> int:
        n = C.c_uint64()
        self._eng._check(self._eng.lib.urlgpu_result_scored(self._h, C.byref(n)))
        return n.value

    def fetch(self, pinned: bool = False, first: int = 0, n: int | None = None):
        """-> (masks uint64[n, words], scores float32[n]) in canonical (|S|, mask) order: the stored entries [first, first + n),
        by default all of them.
        pinned=True: the arrays are views of the engine's page-locked result buffer (PCIe-speed copy, no page faults on
        fresh memory); they stay valid until the next pinned fetch on the same engine."""
        if n is None:
            n = self.count() - first
        if pinned:
            masks, scores = self._eng._pinned_views(n, self.words)
        else:
            masks = np.zeros((n, self.words), dtype=np.uint64)
            scores = np.zeros(n, dtype=np.float32)
        if n:
            self._eng._check(self._eng.lib.urlgpu_result_fetch(self._h, first, n, masks.ctypes.data, scores.ctypes.data))
        return masks, scores

    def fetch_device(self, masks_ptr: int, scores_ptr: int, words_out: int | None = None, shift: int = 0, first: int = 0,
                     n: int | None = None) -> int:
        """write the stored entries [first, first + n) (canonical order; by default all of them) to device addresses — local or
        peer-mapped (Engine.peer_open): masks as ``words_out`` words with every variable index shifted by ``shift``, scores as
        float32.  A null (0) address skips that part.  -> number of entries"""
        if n is None:
            n = self.count() - first
        if n:
            self._eng._check(self._eng.lib.urlgpu_result_fetch_device(self._h, first, n, int(words_out or self.words), int(shift),
                                                                      C.c_void_p(masks_ptr), C.c_void_p(scores_ptr)))
        return n

    def free(self):
        if self._h is not None:
            self._eng._live.pop(id(self), None)
            if self._eng._h is not None:          # after Engine.close() the context (and everything it owned) is gone already
                self._eng.lib.urlgpu_result_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    """One urlgpu context = one B200 + one stream (ScoringFunction + ScoreCalculator of the reference)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.urlgpu_create(C.byref(h), device)
        if rc != 0:
            raise UrlGpuError(self.lib.urlgpu_last_error(None).decode())
        self._h = h
        self.p = 0
        self._keep = []
        self._live = {}
        self._pin_ptr, self._pin_cap = None, 0

    def _pinned_views(self, n: int, words: int):
        """views of a page-locked buffer for n result entries, grown geometrically"""
        need = n * (8 * words + 4) + 64
        if need > self._pin_cap:
            if self._pin_ptr:
                self.lib.urlgpu_host_free(self._pin_ptr)
            cap = max(need + need // 2, 1 << 20)
            ptr = self.lib.urlgpu_host_alloc(cap)
            if not ptr:
                self._pin_ptr, self._pin_cap = None, 0
                raise UrlGpuError(f"cannot page-lock {cap} bytes of host memory")
            self._pin_ptr, self._pin_cap = ptr, cap
        mbytes = n * 8 * words
        buf = (C.c_char * self._pin_cap).from_address(self._pin_ptr)
        masks = np.frombuffer(buf, dtype=np.uint64, count=n * words, offset=0).reshape(n, words)
        scores = np.frombuffer(buf, dtype=np.float32, count=n, offset=(mbytes + 63) // 64 * 64)
        return masks, scores

    def close(self):
        for ref in list(getattr(self, "_live", {}).values()):   # results still alive are freed with their context
            r = ref()
            if r is not None:
                r.free()
        if getattr(self, "_pin_ptr", None):
            self.lib.urlgpu_host_free(self._pin_ptr)
            self._pin_ptr, self._pin_cap = None, 0
        if getattr(self, "_h", None):
            self.lib.urlgpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise UrlGpuError(self.lib.urlgpu_last_error(self._h).decode())

    # data --------------------------------------------------------------------------------
    def set_discrete(self, codes: np.ndarray, card: Iterable[int]):
        """codes: uint8 [p, n] (row i = all records of variable i, i.e. column-major records)."""
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        card = np.ascontiguousarray(list(card), dtype=np.int32)
        p, n = codes.shape
        self._check(self.lib.urlgpu_set_discrete(self._h, codes.ctypes.data, n, p, card.ctypes.data))
        self.p = p

    def set_discrete_device(self, dev_ptr: int, n: int, p: int, card: Iterable[int]):
        card = np.ascontiguousarray(list(card), dtype=np.int32)
        self._check(self.lib.urlgpu_set_discrete_device(self._h, C.c_void_p(dev_ptr), n, p, card.ctypes.data))
        self.p = p

    def share_discrete(self, owner: "Engine"):
        """score from `owner`'s device copy of the data set (same device, no copy)"""
        self._check(self.lib.urlgpu_share_discrete(self._h, owner._h))
        self.p = owner.p

    def set_continuous(self, x: np.ndarray):
        """x: float64 [p, n]."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        p, n = x.shape
        self._check(self.lib.urlgpu_set_continuous(self._h, x.ctypes.data, n, p))
        self.p = p

    def set_continuous_device(self, dev_ptr: int, n: int, p: int):
        self._check(self.lib.urlgpu_set_continuous_device(self._h, C.c_void_p(dev_ptr), n, p))
        self.p = p

    # row-sharded protocol (include/urlgpu.h): moments and the partial Gram of this rank's rows
    def shard_begin(self, x, n_local: int | None = None, p: int | None = None):
        """x: float64 [p, n_local] numpy array (copied) or a device pointer (int) used in place."""
        if isinstance(x, int):
            self._check(self.lib.urlgpu_shard_begin(self._h, C.c_void_p(x), n_local, p, 1))
            self.p = p
        else:
            x = np.ascontiguousarray(x, dtype=np.float64)
            self._keep = [x]
            self._check(self.lib.urlgpu_shard_begin(self._h, x.ctypes.data, x.shape[1], x.shape[0], 0))
            self.p = x.shape[0]

    def shard_moments(self, shift=None):
        s1 = np.zeros(self.p)
        s2 = np.zeros(self.p)
        sh = None if shift is None else np.ascontiguousarray(shift, dtype=np.float64)
        self._check(self.lib.urlgpu_shard_moments(self._h, None if sh is None else sh.ctypes.data, s1.ctypes.data, s2.ctypes.data))
        return s1, s2

    def shard_finish(self, mean, dev, n_total: int):
        mean = np.ascontiguousarray(mean, dtype=np.float64)
        dev = np.ascontiguousarray(dev, dtype=np.float64)
        self._check(self.lib.urlgpu_shard_finish(self._h, mean.ctypes.data, dev.ctypes.data, n_total))
        self._keep = []

    def gram(self) -> np.ndarray:
        g = np.zeros((self.p, self.p), dtype=np.float64)
        self._check(self.lib.urlgpu_get_gram(self._h, g.ctypes.data))
        return g

    def set_gram(self, g: np.ndarray, n_total: int):
        g = np.ascontiguousarray(g, dtype=np.float64)
        self._check(self.lib.urlgpu_set_gram(self._h, g.ctypes.data, n_total, g.shape[0]))
        self.p = g.shape[0]

    def set_stream(self, stream_ptr: int | None):
        self._check(self.lib.urlgpu_set_stream(self._h, C.c_void_p(stream_ptr or 0)))

    def synchronize(self):
        self._check(self.lib.urlgpu_synchronize(self._h))

    # scoring -----------------------------------------------------------------------------
    def score_variable(self, variable: int, neighbors: int, max_parents: int, score_type: int = BIC,
                       lam: float = 0.0, flags: int = KEEP_ALL) -> Result:
        words = mask_words_for(self.p)
        nb = mask_to_words(neighbors, words)
        h = C.c_void_p()
        self._check(self.lib.urlgpu_score_variable(self._h, variable, nb.ctypes.data, words, max_parents, score_type,
                                                   float(lam), flags, C.byref(h)))
        return Result(self, h, words)

    # (variable, parent-set range) shards ------------------------------------------------
    def family_size(self, variable: int, neighbors: int, max_parents: int, score_type: int = BIC) -> int:
        words = mask_words_for(self.p)
        nb = mask_to_words(neighbors, words)
        n = C.c_uint64()
        self._check(self.lib.urlgpu_family_size(self._h, variable, nb.ctypes.data, words, max_parents, score_type, C.byref(n)))
        return n.value

    def score_range(self, variable: int, neighbors: int, max_parents: int, score_type: int, first: int, count: int,
                    lam: float = 0.0, out_device_ptr: int | None = None):
        """raw scores of the family's sets [first, first+count) in canonical order -> float32 array, or written to a
        device buffer (out_device_ptr, e.g. a torch CUDA tensor's data_ptr()) when given"""
        words = mask_words_for(self.p)
        nb = mask_to_words(neighbors, words)
        if out_device_ptr is not None:
            self._check(self.lib.urlgpu_score_range(self._h, variable, nb.ctypes.data, words, max_parents, score_type, float(lam),
                                                    first, count, C.c_void_p(out_device_ptr), 1))
            return None
        out = np.zeros(count, dtype=np.float32)
        self._check(self.lib.urlgpu_score_range(self._h, variable, nb.ctypes.data, words, max_parents, score_type, float(lam),
                                                first, count, out.ctypes.data, 0))
        return out

    def score_part(self, variable: int, neighbors: int, max_parents: int, score_type: int, part: int, parts: int,
                   lam: float = 0.0, out_device_ptr: int | None = None):
        """one of `parts` disjoint parts of the family (engine-chosen: a sub-forest of root tables for BIC, a range otherwise):
        all family_size raw scores, NOT_SCORED (0x7fc0beef) outside the part; merge the parts with an int32 MIN"""
        words = mask_words_for(self.p)
        nb = mask_to_words(neighbors, words)
        if out_device_ptr is not None:
            self._check(self.lib.urlgpu_score_part(self._h, variable, nb.ctypes.data, words, max_parents, score_type, float(lam),
                                                   part, parts, C.c_void_p(out_device_ptr), 1))
            return None
        out = np.zeros(self.family_size(variable, neighbors, max_parents, score_type), dtype=np.float32)
        self._check(self.lib.urlgpu_score_part(self._h, variable, nb.ctypes.data, words, max_parents, score_type, float(lam),
                                               part, parts, out.ctypes.data, 0))
        return out

    def result_from_scores(self, variable: int, neighbors: int, max_parents: int, score_type: int, scores, n: int | None = None,
                           flags: int = KEEP_ALL) -> "Result":
        """scores: float32 numpy array of the whole family's raw scores, or a device pointer (int) with n entries"""
        words = mask_words_for(self.p)
        nb = mask_to_words(neighbors, words)
        h = C.c_void_p()
        if isinstance(scores, int):
            self._check(self.lib.urlgpu_result_from_scores(self._h, variable, nb.ctypes.data, words, max_parents, score_type,
                                                           C.c_void_p(scores), n, 1, flags, C.byref(h)))
        else:
            scores = np.ascontiguousarray(scores, dtype=np.float32)
            self._check(self.lib.urlgpu_result_from_scores(self._h, variable, nb.ctypes.data, words, max_parents, score_type,
                                                           scores.ctypes.data, len(scores), 0, flags, C.byref(h)))
        return Result(self, h, words)

    def sparse_parent_graph(self, masks: np.ndarray, scores: np.ndarray, variable_count: int) -> "SparseParentGraph":
        """device query structure over one variable's cache; scores with the search side's sign (lower is better)"""
        return SparseParentGraph(self, masks, scores, variable_count)

    def score_one(self, variable: int, parents: int, score_type: int = BIC, lam: float = 0.0):
        """ScoringFunction::calculateScore -> (float32 score, float64 pre-rounding value)."""
        words = mask_words_for(self.p)
        pm = mask_to_words(parents, words)
        s, v = C.c_float(), C.c_double()
        self._check(self.lib.urlgpu_score_one(self._h, variable, pm.ctypes.data, words, score_type, float(lam),
                                              C.byref(s), C.byref(v)))
        return np.float32(s.value), v.value

    def score_sets(self, variables, parents, score_type: int = BIC, lam: float = 0.0):
        """score a list of (variable, parent set) pairs in one call -> (float32 [n] scores, float64 [n] values), entry i bit-equal to
        score_one(variables[i], parents[i], score_type, lam).  parents: a sequence of Python ints, or an (n, words) uint64 array"""
        var = np.ascontiguousarray(variables, dtype=np.int32).reshape(-1)
        if isinstance(parents, np.ndarray) and parents.dtype == np.uint64:
            pm = np.ascontiguousarray(parents.reshape(-1, 1) if parents.ndim == 1 else parents)
        else:
            words = mask_words_for(self.p)
            ints = [int(m) for m in parents]
            pm = np.zeros((len(ints), words), dtype=np.uint64)
            for w in range(words):
                pm[:, w] = [(m >> (64 * w)) & 0xFFFFFFFFFFFFFFFF for m in ints]
        if len(pm) != len(var):
            raise ValueError(f"{len(var)} variables but {len(pm)} parent sets")
        n = len(var)
        scores = np.zeros(n, dtype=np.float32)
        values = np.zeros(n, dtype=np.float64)
        self._check(self.lib.urlgpu_score_sets(self._h, n, var.ctypes.data, pm.ctypes.data, max(pm.shape[1], 1), score_type, float(lam),
                                               scores.ctypes.data, values.ctypes.data))
        return scores, values

    def order_search(self, entries, p: int, component: int, edges: Sequence[int] | None = None):
        """urlgpu_order_search: the optimal DAG of one skeleton component over the order graph, layer by layer on the device.
        Components of more than 32 variables go to urlgpu_order_search_layered, the same search with a limit of 36.
        entries: p pairs (masks, scores) per variable in the search side's sign (lower is better), masks uint64 [n] or
        [n, words] or ints; component: a variable mask; edges: p skeleton masks or None.
        -> (float32 cost, order list (first = a root), parents uint64 [p] ([p, words] above 64 variables; 0 outside C))"""
        k = bin(int(component)).count("1")
        return self._order_search("urlgpu_order_search" if k <= 32 else "urlgpu_order_search_layered", entries, p, component, edges)

    def _order_search(self, symbol: str, entries, p: int, component: int, edges: Sequence[int] | None):
        """order_search through the named entry point, urlgpu_order_search or urlgpu_order_search_layered"""
        words, offsets, masks, scores, comp, ed = self._order_args(entries, p, component, edges)
        cost = C.c_float()
        order = np.zeros(max(1, bin(int(component)).count("1")), dtype=np.int32)
        parents = np.zeros((p, words), dtype=np.uint64)
        self._check(getattr(self.lib, symbol)(self._h, p, words, offsets.ctypes.data, masks.ctypes.data if len(masks) else None,
                                              scores.ctypes.data if len(scores) else None, None if ed is None else ed.ctypes.data,
                                              comp.ctypes.data, C.byref(cost), order.ctypes.data, parents.ctypes.data))
        return np.float32(cost.value), [int(x) for x in order], parents[:, 0].copy() if words == 1 else parents

    @staticmethod
    def _order_args(entries, p: int, component: int, edges: Sequence[int] | None):
        """the C arrays of the order searches -> (words, offsets, masks, scores, component words, skeleton rows or None)"""
        if len(entries) != p:
            raise ValueError(f"{len(entries)} entry lists for {p} variables")
        words = mask_words_for(p)
        rows, sc, offsets = [], [], np.zeros(p + 1, dtype=np.uint64)
        for v, (m, s_) in enumerate(entries):
            if isinstance(m, np.ndarray) and m.dtype == np.uint64:
                m = m.reshape(-1, 1) if m.ndim == 1 else m
                mm = np.zeros((len(m), words), dtype=np.uint64)
                mm[:, :min(words, m.shape[1])] = m[:, :words]
            else:
                mm = np.array([mask_to_words(int(x), words) for x in m], dtype=np.uint64).reshape(-1, words)
            rows.append(mm)
            sc.append(np.asarray(s_, dtype=np.float32).reshape(-1))
            if len(sc[-1]) != len(mm):
                raise ValueError(f"variable {v}: {len(mm)} masks but {len(sc[-1])} scores")
            offsets[v + 1] = offsets[v] + len(mm)
        masks = np.ascontiguousarray(np.concatenate(rows) if rows else np.zeros((0, words), dtype=np.uint64))
        scores = np.ascontiguousarray(np.concatenate(sc) if sc else np.zeros(0, dtype=np.float32))
        comp = mask_to_words(int(component), words)
        ed = None if edges is None else np.ascontiguousarray(np.stack([mask_to_words(int(e), words) for e in edges]))
        if ed is not None and len(ed) != p:
            raise ValueError(f"{len(ed)} skeleton rows for {p} variables")
        return words, offsets, masks, scores, comp, ed

    def order_local_search(self, entries, p: int, component: int, edges: Sequence[int] | None = None, restarts: int = 256, seed: int = 0):
        """urlgpu_order_local_search: insertion hill climbing over the admissible orders of one skeleton component of up to 256
        variables, from `restarts` random orders, with the objective of order_search (so its cost is never below order_search's).
        Same input conventions as order_search.  When the best-parent tables, 4 2^c_v bytes per variable (c_v: the candidate
        parents inside the component, the union of its qualifying parent sets), would take more than TABLE_MAX_BYTES, the call
        goes to urlgpu_order_local_search_sparse, which scans sorted lists instead (same contract, same bits where both run).
        -> (float32 cost, order list, parents as order_search returns them, float32 [restarts] final cost per restart,
            uint32 [restarts] moves per restart)"""
        args = self._order_args(entries, p, component, edges)
        symbol = "urlgpu_order_local_search" if table_bytes(args[1], args[2], args[4]) <= TABLE_MAX_BYTES else "urlgpu_order_local_search_sparse"
        return self._order_local_search(symbol, entries, p, component, edges, restarts, seed, args)

    def _order_local_search(self, symbol: str, entries, p: int, component: int, edges: Sequence[int] | None = None, restarts: int = 256,
                            seed: int = 0, args=None):
        """order_local_search through the named entry point (tests and measurements compare the table and sparse forms)"""
        words, offsets, masks, scores, comp, ed = args if args is not None else self._order_args(entries, p, component, edges)
        cost = C.c_float()
        order = np.zeros(max(1, bin(int(component)).count("1")), dtype=np.int32)
        parents = np.zeros((p, words), dtype=np.uint64)
        r_cost = np.zeros(max(1, int(restarts)), dtype=np.float32)
        r_moves = np.zeros(max(1, int(restarts)), dtype=np.uint32)
        self._check(getattr(self.lib, symbol)(self._h, p, words, offsets.ctypes.data, masks.ctypes.data if len(masks) else None,
                                              scores.ctypes.data if len(scores) else None, None if ed is None else ed.ctypes.data,
                                              comp.ctypes.data, int(restarts), int(seed) & 0xFFFFFFFFFFFFFFFF, C.byref(cost),
                                              order.ctypes.data, parents.ctypes.data, r_cost.ctypes.data, r_moves.ctypes.data))
        return (np.float32(cost.value), [int(x) for x in order], parents[:, 0].copy() if words == 1 else parents,
                r_cost[:restarts], r_moves[:restarts])

    @staticmethod
    def _cache_entries(cache):
        """a search.ScoreCache or a list of p (masks, scores) pairs -> (entries, p)"""
        if hasattr(cache, "entries") and hasattr(cache, "p"):
            return [cache.entries(v) for v in range(cache.p)], cache.p
        entries = list(cache)
        return entries, len(entries)

    def optimal_dag(self, cache, edges: Sequence[int] | None = None):
        """urlsearch_astar (host/search_capi.cpp:64-94) with urlgpu_order_search in place of A*: the skeleton's components
        (the rule of urlsearch::components), one search each, their costs summed in float32 in component order.
        cache: a search.ScoreCache or a list of p (masks, scores) pairs in search sign; edges: p skeleton masks or None.
        -> (total cost, parents uint64 [p]), the meaning and types of ScoreCache.astar's first two results"""
        return self._per_component(cache, edges, lambda entries, p, comp: self.order_search(entries, p, comp, edges))

    def local_search_dag(self, cache, edges: Sequence[int] | None = None, restarts: int = 256, seed: int = 0):
        """optimal_dag with order_local_search in place of order_search: one call per component, each with the same seed, the
        costs summed in float32 in component order.  Components of any size up to 256 variables, with any number of candidate
        parents per variable. -> (total cost, parents)"""
        return self._per_component(cache, edges, lambda entries, p, comp: self.order_local_search(entries, p, comp, edges, restarts, seed)[:3])

    def _per_component(self, cache, edges, search):
        entries, p = self._cache_entries(cache)
        total = np.float32(0)
        parents = None
        for comp in components(p, edges):
            cost, _, par = search(entries, p, comp)
            total = np.float32(total + cost)
            if parents is None:
                parents = np.zeros_like(par)
            for v in range(p):
                if (comp >> v) & 1:
                    parents[v] = par[v]
        return float(total), parents

    def contingency(self, variable: int, parents: int, n_cells: int) -> np.ndarray:
        words = mask_words_for(self.p)
        pm = mask_to_words(parents, words)
        out = np.zeros(n_cells, dtype=np.int32)
        self._check(self.lib.urlgpu_contingency(self._h, variable, pm.ctypes.data, words, out.ctypes.data, n_cells))
        return out

    def prune(self, masks: np.ndarray, scores: np.ndarray) -> np.ndarray:
        masks = np.ascontiguousarray(masks, dtype=np.uint64)
        if masks.ndim == 1:
            masks = masks.reshape(-1, 1)
        scores = np.ascontiguousarray(scores, dtype=np.float32)
        keep = np.zeros(len(scores), dtype=np.uint8)
        self._check(self.lib.urlgpu_prune(self._h, masks.ctypes.data, scores.ctypes.data, len(scores), masks.shape[1],
                                          keep.ctypes.data))
        return keep.astype(bool)

    # measurement -------------------------------------------------------------------------
    def stats(self) -> dict:
        st = Stats()
        self._check(self.lib.urlgpu_stats_get(self._h, C.byref(st)))
        return st.as_dict()

    def reset_stats(self):
        self._check(self.lib.urlgpu_stats_reset(self._h))

    def enable_timing(self, on: bool = True):
        self._check(self.lib.urlgpu_stats_enable_timing(self._h, int(on)))

    def copy_to_host(self, host: np.ndarray, dev_ptr: int, nbytes: int):
        """bytes at a device address -> a (preferably page-locked) host array"""
        self._check(self.lib.urlgpu_copy_to_host(self._h, host.ctypes.data, C.c_void_p(dev_ptr), int(nbytes)))

    def peer_alloc(self, nbytes: int):
        """a device buffer other ranks can map (urlgpu_peer_alloc) -> (device pointer, 64-byte handle)"""
        p = C.c_void_p()
        h = (C.c_ubyte * 64)()
        self._check(self.lib.urlgpu_peer_alloc(self._h, int(nbytes), C.byref(p), h))
        return p.value, bytes(h)

    def peer_open(self, handle: bytes) -> int:
        """map another rank's buffer into this process (CUDA IPC, peer access over NVLink) -> device pointer"""
        p = C.c_void_p()
        h = (C.c_ubyte * 64).from_buffer_copy(handle)
        self._check(self.lib.urlgpu_peer_open(self._h, h, C.byref(p)))
        return p.value

    def peer_close(self, ptr: int):
        self._check(self.lib.urlgpu_peer_close(self._h, C.c_void_p(ptr)))

    def peer_free(self, ptr: int):
        self._check(self.lib.urlgpu_peer_free(self._h, C.c_void_p(ptr)))

    def probe_fp64(self) -> dict:
        """measured FP64 issue rates of this device in TFLOP/s: {'dfma': ..., 'dmma': ...}"""
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.urlgpu_probe_fp64(self._h, C.byref(a), C.byref(b)))
        return {"dfma": a.value, "dmma": b.value}


class SparseParentGraph:
    """urlgpu_spg_*: SparseParentBitwise (score_cache/sparse_parent_bitwise.cpp) on the device, batched getScore."""

    def __init__(self, eng: Engine, masks, scores, variable_count: int):
        masks = np.ascontiguousarray(masks, dtype=np.uint64)
        if masks.ndim == 1:
            masks = masks.reshape(-1, 1)
        scores = np.ascontiguousarray(scores, dtype=np.float32)
        self._eng, self.words = eng, masks.shape[1]
        h = C.c_void_p()
        eng._check(eng.lib.urlgpu_spg_build(eng._h, masks.ctypes.data, scores.ctypes.data, len(scores), self.words, variable_count, C.byref(h)))
        self._h = h

    def query(self, allowed):
        """allowed: uint64 [nq] or [nq, words] sets of variables allowed as parents -> (best float32 [nq], parents uint64 [nq, words], index int64 [nq])"""
        q = np.ascontiguousarray(allowed, dtype=np.uint64)
        if q.ndim == 1:
            q = q.reshape(-1, 1)
        nq = q.shape[0]
        best = np.zeros(nq, dtype=np.float32)
        parents = np.zeros((nq, self.words), dtype=np.uint64)
        index = np.zeros(nq, dtype=np.int64)
        self._eng._check(self._eng.lib.urlgpu_spg_query(self._h, q.ctypes.data, nq, best.ctypes.data, parents.ctypes.data, index.ctypes.data))
        return best, parents, index

    def free(self):
        if self._h is not None:
            self._eng.lib.urlgpu_spg_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


from . import datagen, pss  # noqa: E402


def device_count() -> int:
    return load_library().urlgpu_device_count()


class EnginePool:
    """T urlgpu contexts (one stream each) on ONE device, driven by one host thread each — the `-t T` worker threads of
    the reference's `score` (score_main.cpp:132-139, 372-380) pointed at a single GPU.  Planning, enqueueing and
    reading back one variable overlap with the kernels of another, which closes the gaps a single in-order stream
    leaves between the many small kernels of small families (config 4: 451 -> 380 ms per pass with T = 3).
    The contexts share one device copy of the data set; results are bit-identical to a single Engine's."""

    def __init__(self, device: int = 0, threads: int = 2):
        self.engines = [Engine(device) for _ in range(max(1, threads))]

    def __len__(self):
        return len(self.engines)

    def _each(self, fn):
        import threading
        errs = []

        def run(e):
            try:
                fn(e)
            except Exception as ex:  # re-raised in the caller's thread
                errs.append(ex)
        th = [threading.Thread(target=run, args=(e,)) for e in self.engines]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]

    def set_discrete(self, codes, card):
        """one upload; the other contexts borrow the first one's device copy"""
        self.engines[0].set_discrete(codes, list(card))
        for e in self.engines[1:]:
            e.share_discrete(self.engines[0])

    def set_discrete_device(self, dev_ptr, n, p, card):
        self.engines[0].set_discrete_device(dev_ptr, n, p, list(card))
        for e in self.engines[1:]:
            e.share_discrete(self.engines[0])

    def set_continuous(self, x):
        self.engines[0].set_continuous(x)
        g = self.engines[0].gram()
        for e in self.engines[1:]:
            e.set_gram(g, x.shape[1])

    def set_gram(self, g, n_total):
        for e in self.engines:
            e.set_gram(g, n_total)

    def gram(self):
        return self.engines[0].gram()

    def run(self, items, max_parents, score_type=BIC, lam=0.0, flags=KEEP_ALL, fetch=False, costs=None, contexts=None):
        """items: [(variable, neighbors mask)].  Scores every item on one of the pool's contexts (dealt out by `costs`,
        longest first, else round robin).  fetch=True -> {variable: (masks, scores)}, read back one variable behind the
        one being scored (urlgpu_result_prefetch); fetch="pinned" -> {variable: stored entries}, every cache is read back
        into the context's page-locked result buffer (overwritten by the next one: for drivers that consume each cache as
        it arrives); fetch="keep" -> {variable: Result} with the compaction enqueued (for device-side consumers such as
        distributed.gather_results_p2p; the caller frees them); fetch=False -> {variable: sets scored}, results dropped on the device.
        contexts: use only the first `contexts` contexts (1 = strictly serial kernels, for per-kernel timing)."""
        T = len(self.engines) if contexts is None else max(1, min(contexts, len(self.engines)))
        order = sorted(range(len(items)), key=lambda i: (-(costs[i] if costs is not None else 0.0), i))
        load = [0.0] * T
        lists = [[] for _ in range(T)]
        for k, i in enumerate(order):
            t = min(range(T), key=lambda j: (load[j], j)) if costs is not None else k % T
            lists[t].append(i)
            load[t] += costs[i] if costs is not None else 1.0
        out = {}
        import threading
        errs = []

        def take(res):
            if fetch == "pinned":
                return len(res.fetch(pinned=True)[1])
            return res.fetch()

        keep = fetch == "keep"   # -> {variable: Result}, compaction enqueued, results alive: the caller reads and frees them

        def work(t):
            eng = self.engines[t]
            try:
                prev = None
                for i in lists[t]:
                    v, nb = items[i]
                    res = eng.score_variable(v, nb, max_parents, score_type, lam=lam, flags=flags)
                    if keep:
                        out[v] = res.prefetch()
                    elif fetch:
                        res.prefetch()
                        if prev is not None:
                            out[prev[0]] = take(prev[1])
                            prev[1].free()
                        prev = (v, res)
                    else:
                        # nothing is read back, but every result is still completed on the device: the compaction runs and the
                        # count is awaited one variable behind, which is also where a speculative 16-bit table that
                        # overflowed is noticed and the variable recomputed (result_wait_counts)
                        out[v] = res.scored()
                        res.prefetch()
                        if prev is not None:
                            prev[1].count()
                            prev[1].free()
                        prev = (v, res)
                if prev is not None:
                    if fetch:
                        out[prev[0]] = take(prev[1])
                    else:
                        prev[1].count()
                    prev[1].free()
                eng.synchronize()
            except Exception as ex:
                errs.append(ex)
        th = [threading.Thread(target=work, args=(t,)) for t in range(T)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        return out

    def stats(self):
        """sum of the contexts' statistics"""
        tot = None
        for e in self.engines:
            st = e.stats()
            tot = st if tot is None else {k: tot[k] + st[k] for k in st}
        return tot

    def reset_stats(self):
        for e in self.engines:
            e.reset_stats()

    def enable_timing(self, on):
        for e in self.engines:
            e.enable_timing(on)

    def close(self):
        for e in reversed(self.engines):  # borrowers first
            e.close()
