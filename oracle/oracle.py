"""ctypes loader for the CPU oracle (oracle/hnsw_oracle.c).

TEST INFRASTRUCTURE ONLY -- importable from tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  The product package never imports this.
Parity is UNPINNED: the reference mount has no source (/root/reference/README.md:1), so the
oracle restates upstream pgvector HNSW semantics from memory (see hnsw_oracle.h).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libhnsw_oracle.so")

L2, IP, COSINE, L1 = 0, 1, 2, 3
F32, F16 = 0, 1
CANON, NATURAL = 0, 1
HEAPTIDS = 10


class Counters(C.Structure):
    _fields_ = [("n_dist", C.c_int64), ("n_hop0", C.c_int64), ("n_hopu", C.c_int64), ("n_pair", C.c_int64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


def build_lib(force=False):
    """make -C oracle (gcc only)."""
    srcs = [os.path.join(_HERE, f) for f in ("hnsw_oracle.c", "hnsw_oracle.h", "dist_natural.c", "Makefile")]
    stale = force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if stale:
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build_lib()
    L = C.CDLL(_SO)
    vp, i32p, f32p, u8p, i64p = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
    L.orc_create.restype = C.c_void_p
    L.orc_create.argtypes = [C.c_int] * 6 + [C.c_uint64]
    L.orc_free.argtypes = [C.c_void_p]
    L.orc_set_dist_mode.argtypes = [C.c_void_p, C.c_int]
    L.orc_level_for.restype = C.c_int
    L.orc_level_for.argtypes = [C.c_uint64, C.c_int64, C.c_int]
    L.orc_max_level.restype = C.c_int
    L.orc_max_level.argtypes = [C.c_int]
    L.orc_splitmix64.restype = C.c_uint64
    L.orc_splitmix64.argtypes = [C.c_uint64]
    L.orc_insert.restype = C.c_int64
    L.orc_insert.argtypes = [C.c_void_p, vp, C.c_int64]
    L.orc_build.restype = C.c_int64
    L.orc_build.argtypes = [C.c_void_p, vp, C.c_int64, i64p]
    L.orc_bulk_delete.restype = C.c_int64
    L.orc_bulk_delete.argtypes = [C.c_void_p, i64p, C.c_int64]
    L.orc_vacuum_repair.restype = C.c_int64
    L.orc_vacuum_repair.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    L.orc_search_elements.restype = C.c_int
    L.orc_search_elements.argtypes = [C.c_void_p, vp, C.c_int, i32p, f32p, C.POINTER(Counters)]
    L.orc_search_tids.restype = C.c_int
    L.orc_search_tids.argtypes = [C.c_void_p, vp, C.c_int, C.c_int, i64p, f32p, C.POINTER(Counters)]
    L.orc_search_batch.argtypes = [C.c_void_p, vp, C.c_int64, C.c_int, i32p, f32p, i32p, C.POINTER(Counters), C.c_int]
    L.orc_search_layer.restype = C.c_int
    L.orc_search_layer.argtypes = [C.c_void_p, vp, i32p, C.c_int, C.c_int, C.c_int, i32p, f32p, C.POINTER(Counters)]
    L.orc_bruteforce.argtypes = [C.c_void_p, vp, C.c_int64, C.c_int, i32p, vp, C.c_int]
    L.orc_exact_topk.argtypes = [C.c_void_p, vp, C.c_int64, C.c_int, i32p, f32p, C.c_int]
    L.orc_iter_begin.restype = C.c_void_p
    L.orc_iter_begin.argtypes = [C.c_void_p, vp, C.c_int, C.c_int64]
    L.orc_iter_next.restype = C.c_int
    L.orc_iter_next.argtypes = [C.c_void_p, i32p, f32p]
    L.orc_iter_tuples.restype = C.c_int64
    L.orc_iter_tuples.argtypes = [C.c_void_p]
    L.orc_iter_discarded.restype = C.c_int64
    L.orc_iter_discarded.argtypes = [C.c_void_p]
    L.orc_iter_counters.argtypes = [C.c_void_p, C.POINTER(Counters)]
    L.orc_iter_end.argtypes = [C.c_void_p]
    L.orc_distance.restype = C.c_float
    L.orc_distance.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    L.orc_normalize.restype = C.c_int
    L.orc_normalize.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp]
    L.orc_n.restype = C.c_int64
    L.orc_n.argtypes = [C.c_void_p]
    L.orc_upper_rows.restype = C.c_int64
    L.orc_upper_rows.argtypes = [C.c_void_p]
    L.orc_entry.restype = C.c_int32
    L.orc_entry.argtypes = [C.c_void_p]
    L.orc_entry_level.restype = C.c_int
    L.orc_entry_level.argtypes = [C.c_void_p]
    L.orc_counters.argtypes = [C.c_void_p, C.POINTER(Counters)]
    L.orc_export.argtypes = [C.c_void_p, vp, u8p, i32p, i32p, i32p, u8p, i64p]
    L.orc_import.restype = C.c_void_p
    L.orc_import.argtypes = [C.c_int] * 6 + [C.c_int64, C.c_int64, C.c_int32, vp, u8p, i32p, i32p, i32p, u8p, i64p]
    _lib = L
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _np_dtype(dtype):
    return np.float32 if dtype == F32 else np.float16


def distance(a, b, metric=L2, dtype=F32, mode=CANON):
    a = np.ascontiguousarray(a, _np_dtype(dtype))
    b = np.ascontiguousarray(b, _np_dtype(dtype))
    code = L1 if metric == L1 else int(metric != L2)
    return float(lib().orc_distance(code, dtype, mode, a.shape[-1], _p(a), _p(b)))


def normalize(a, dtype=F32, mode=CANON):
    a = np.ascontiguousarray(a, _np_dtype(dtype))
    out = np.empty_like(a)
    ok = lib().orc_normalize(dtype, mode, a.shape[-1], _p(a), _p(out))
    return out, bool(ok)


def level_for(seed, seq, m):
    return lib().orc_level_for(seed, seq, m)


def splitmix64(x):
    return int(lib().orc_splitmix64(C.c_uint64(x & 0xFFFFFFFFFFFFFFFF)))


class Graph:
    """The flat graph image both the oracle and the CUDA library understand."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


class Index:
    def __init__(self, dim, m=16, ef_construction=64, metric=L2, dtype=F32, mode=CANON, seed=0, _h=None):
        self.dim, self.m, self.efc, self.metric, self.dtype, self.mode = dim, m, ef_construction, metric, dtype, mode
        self.seed = seed
        self._h = _h if _h is not None else lib().orc_create(dim, m, ef_construction, metric, dtype, mode, seed)
        if not self._h:
            raise ValueError("orc_create rejected the parameters")

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_free(self._h)
            self._h = None

    def _q(self, q):
        q = np.ascontiguousarray(q, _np_dtype(self.dtype))
        assert q.shape[-1] == self.dim
        return q

    def set_mode(self, mode):
        self.mode = mode
        lib().orc_set_dist_mode(self._h, mode)

    @property
    def n(self):
        return int(lib().orc_n(self._h))

    @property
    def entry(self):
        return int(lib().orc_entry(self._h)), int(lib().orc_entry_level(self._h))

    def insert(self, vec, tid):
        return int(lib().orc_insert(self._h, _p(self._q(vec)), tid))

    def build(self, vecs, tids=None):
        vecs = self._q(vecs)
        t = None if tids is None else np.ascontiguousarray(tids, np.int64)
        return int(lib().orc_build(self._h, _p(vecs), vecs.shape[0], _p(t)))

    def bulk_delete(self, dead_tids):
        """hnswvacuum.c RemoveHeapTids -> number of heap TIDs removed"""
        t = np.ascontiguousarray(dead_tids, np.int64)
        return int(lib().orc_bulk_delete(self._h, _p(t), t.size))

    def vacuum_repair(self):
        """hnswvacuum.c RepairGraph + MarkDeleted -> (elements marked deleted, elements re-linked)"""
        rep = C.c_int64()
        marked = int(lib().orc_vacuum_repair(self._h, C.byref(rep)))
        return marked, int(rep.value)

    def build_counters(self):
        c = Counters()
        lib().orc_counters(self._h, C.byref(c))
        return c.as_dict()

    def search_elements(self, q, ef):
        q = self._q(q)
        e = np.empty(ef, np.int32)
        d = np.empty(ef, np.float32)
        c = Counters()
        n = lib().orc_search_elements(self._h, _p(q), ef, _p(e), _p(d), C.byref(c))
        return e[:n], d[:n], c.as_dict()

    def search_tids(self, q, ef, k):
        q = self._q(q)
        t = np.empty(k, np.int64)
        d = np.empty(k, np.float32)
        n = lib().orc_search_tids(self._h, _p(q), ef, k, _p(t), _p(d), None)
        return t[:n], d[:n]

    def search_batch(self, qs, ef, threads=1):
        qs = self._q(qs)
        nq = qs.shape[0]
        e = np.empty((nq, ef), np.int32)
        d = np.empty((nq, ef), np.float32)
        cnt = np.empty(nq, np.int32)
        c = Counters()
        lib().orc_search_batch(self._h, _p(qs), nq, ef, _p(e), _p(d), _p(cnt), C.byref(c), threads)
        return e, d, cnt, c.as_dict()

    def search_layer(self, q, ep, ef, lc):
        q = self._q(q)
        ep = np.ascontiguousarray(ep, np.int32)
        cap = max(ef, len(ep)) + 2
        e = np.empty(cap, np.int32)
        d = np.empty(cap, np.float32)
        c = Counters()
        n = lib().orc_search_layer(self._h, _p(q), _p(ep), len(ep), ef, lc, _p(e), _p(d), C.byref(c))
        return e[:n], d[:n], c.as_dict()

    def iterate(self, q, ef, max_scan_tuples=20000, max_batches=1 << 30):
        """hnsw.iterative_scan: list of (elements, distances) batches, the first being GetScanItems'
        result and each later one a ResumeScanItems batch (or single leftover candidates once
        max_scan_tuples was reached).  Also returns (tuples, counters)."""
        q = self._q(q)
        it = lib().orc_iter_begin(self._h, _p(q), ef, max_scan_tuples)
        out = []
        e = np.empty(ef + 2, np.int32)
        d = np.empty(ef + 2, np.float32)
        while len(out) < max_batches:
            n = lib().orc_iter_next(it, _p(e), _p(d))
            if n == 0:
                break
            out.append((e[:n].copy(), d[:n].copy()))
        tuples = lib().orc_iter_tuples(it)
        c = Counters()
        lib().orc_iter_counters(it, C.byref(c))
        lib().orc_iter_end(it)
        return out, tuples, c.as_dict()

    def bruteforce(self, qs, k, threads=1):
        qs = self._q(qs)
        nq = qs.shape[0]
        e = np.empty((nq, k), np.int32)
        d = np.empty((nq, k), np.float64)
        lib().orc_bruteforce(self._h, _p(qs), nq, k, _p(e), _p(d), threads)
        return e, d

    def exact_topk(self, qs, k, threads=1):
        """top-k by the canonical fp32 distance and element id over every row (the exact scan's answer)"""
        qs = self._q(qs)
        nq = qs.shape[0]
        e = np.empty((nq, k), np.int32)
        d = np.empty((nq, k), np.float32)
        lib().orc_exact_topk(self._h, _p(qs), nq, k, _p(e), _p(d), threads)
        return e, d

    def export(self):
        n, ur, m = self.n, int(lib().orc_upper_rows(self._h)), self.m
        g = Graph(dim=self.dim, m=m, efc=self.efc, metric=self.metric, dtype=self.dtype, n=n, upper_rows=ur,
                  entry=self.entry[0], entry_level=self.entry[1],
                  vecs=np.empty((n, self.dim), _np_dtype(self.dtype)), level=np.empty(n, np.uint8),
                  nbr0=np.empty((n, 2 * m), np.int32), uoff=np.empty(n, np.int32),
                  nbru=np.empty((max(ur, 1), m), np.int32), ntids=np.empty(n, np.uint8),
                  tids=np.empty((n, HEAPTIDS), np.int64))
        g.nbru[:] = -1
        lib().orc_export(self._h, _p(g.vecs), _p(g.level), _p(g.nbr0), _p(g.uoff), _p(g.nbru), _p(g.ntids), _p(g.tids))
        return g

    @classmethod
    def from_graph(cls, g, mode=CANON):
        vecs = np.ascontiguousarray(g.vecs, _np_dtype(g.dtype))
        args = [np.ascontiguousarray(g.level, np.uint8), np.ascontiguousarray(g.nbr0, np.int32),
                np.ascontiguousarray(g.uoff, np.int32), np.ascontiguousarray(g.nbru, np.int32),
                np.ascontiguousarray(g.ntids, np.uint8), np.ascontiguousarray(g.tids, np.int64)]
        h = lib().orc_import(g.dim, g.m, g.efc, g.metric, g.dtype, mode, g.n, g.upper_rows, g.entry,
                             _p(vecs), *[_p(a) for a in args])
        return cls(g.dim, g.m, g.efc, g.metric, g.dtype, mode, 0, _h=h)
