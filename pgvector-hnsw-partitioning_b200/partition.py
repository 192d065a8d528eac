"""Hash-partitioned HNSW: ctypes mirror of the hb_part_* entry points (include/hnsw_b200.h, csrc/part.cu).

The reference mount has no source (/root/reference/README.md:1), so the partitioning contract is
the one BASELINE.json states: a row goes to partition splitmix64(heap_tid) mod P; a query is
broadcast to every partition; per-partition top-k lists are merged.  One process per GPU: rank r
owns partitions {p : p mod world == r}.  Everything on the data path -- the scans, the on-device
merges and the one ncclAllGather of nq x k (tid, distance) per rank -- happens inside the library;
the NCCL communicator belongs to the hb_part handle.  This module only carries pointers.

torch.distributed is used for one thing: handing rank 0's ncclUniqueId to the other ranks.
"""
import ctypes as C

import numpy as np

from .hnsw import HB_F32, OPCLASSES, Counters, HnswError, HnswIndex, _err, _np_dtype, _p, load_library, partition_route

HB_PART_ID_BYTES = 128
HB_PART_SLOTS = 4


def owned_partitions(n_partitions, rank, world):
    return [p for p in range(n_partitions) if p % world == rank]


def split_rows(heap_tids, n_partitions, rank, world):
    """Rows this rank indexes: {partition -> row indices}, for the partitions it owns (what hb_part_build does
    inside; kept for tests and callers that want to route themselves)."""
    part = partition_route(heap_tids, n_partitions)
    return {p: np.nonzero(part == p)[0] for p in owned_partitions(n_partitions, rank, world)}


def merge_rule(lists, k):
    """part_merge_kernel restated for tests: greedy head merge of lists [(tids, dist), ...], each sorted by
    (distance, tid) and -1 padded, ordered by (distance, tid).  For such lists the result is the k smallest pairs of
    their union, whatever the grouping; lists in another order (a scan's gettuple order) are merged as they come.
    Host-side test helper, never on the product path."""
    heads = [0] * len(lists)
    out_t, out_d = [], []
    for _ in range(k):
        best = None
        for li, (t, d) in enumerate(lists):
            h = heads[li]
            if h >= len(t) or t[h] < 0:
                continue
            key = (float(d[h]), int(t[h]))
            if best is None or key < best[0]:
                best = (key, li)
        if best is None:
            out_t.append(-1)
            out_d.append(float("inf"))
        else:
            out_t.append(best[0][1])
            out_d.append(best[0][0])
            heads[best[1]] += 1
    return out_t, out_d


def share_unique_id(rank, world, group=None):
    """rank 0 draws the ncclUniqueId (hb_part_unique_id), torch.distributed carries it to the other ranks."""
    if world == 1:
        return None
    import torch
    import torch.distributed as dist
    L = load_library()
    buf = np.zeros(HB_PART_ID_BYTES, np.uint8)
    if rank == 0 and L.hb_part_unique_id(_p(buf)) < 0:
        raise _err(L, "hb_part_unique_id")
    t = torch.from_numpy(buf)
    backend = dist.get_backend(group)
    if backend == "nccl":
        t = t.cuda()
    dist.broadcast(t, 0, group=group)
    return t.cpu().numpy().copy()


class PartitionedIndex:
    """hb_part handle: the partitions this rank owns + the communicator."""

    def __init__(self, dim, opclass="vector_l2_ops", n_partitions=8, m=16, ef_construction=64,
                 capacity_per_partition=1 << 20, rank=0, world=1, device=0, seed=0, group=None, unique_id=None):
        if opclass not in OPCLASSES:
            raise HnswError("operator class %r does not exist for access method hnsw" % (opclass,))
        self.dim, self.opclass, self.P, self.rank, self.world, self.device = dim, opclass, n_partitions, rank, world, device
        self.m, self.efc = m, ef_construction
        self.metric, self.dtype = OPCLASSES[opclass]
        self._L = load_library()
        if world > 1 and unique_id is None:
            unique_id = share_unique_id(rank, world, group)
        self._h = self._L.hb_part_create(device, dim, m, ef_construction, self.metric, self.dtype, n_partitions,
                                         capacity_per_partition, seed, rank, world, _p(unique_id))
        if not self._h:
            raise _err(self._L, "hb_part_create")
        own = np.empty(max(n_partitions, 1), np.int32)
        cnt = self._L.hb_part_owned(self._h, _p(own))
        self.owned = [int(p) for p in own[:cnt]]
        assert self.owned == owned_partitions(n_partitions, rank, world)
        self.parts = {p: HnswIndex._view(self._L.hb_part_index(self._h, p), dim, opclass, m, ef_construction, device, seed + p)
                      for p in self.owned}

    def close(self):
        if getattr(self, "_h", None):
            for ix in self.parts.values():
                ix._h = None
            self.parts = {}
            self._L.hb_part_free(self._h)
            self._h = None

    __del__ = close

    def _ck(self, rc, what):
        if rc < 0:
            raise _err(self._L, what)
        return rc

    def set_option(self, name, value):
        self._ck(self._L.hb_part_set_option(self._h, name.encode(), int(value)), "hb_part_set_option")

    def counters(self, reset=False):
        c = Counters()
        self._ck(self._L.hb_part_get_counters(self._h, C.byref(c), int(reset)), "hb_part_get_counters")
        return c.as_dict()

    # ---- build: every rank passes the same rows; each rank indexes the partitions it owns; no collective
    def build(self, vecs, heap_tids=None):
        vecs = np.ascontiguousarray(vecs, _np_dtype(self.dtype))
        if vecs.ndim != 2 or vecs.shape[1] != self.dim:
            raise HnswError("expected %d dimensions, not %d" % (self.dim, vecs.shape[-1]))
        t = None if heap_tids is None else np.ascontiguousarray(heap_tids, np.int64)
        return self._ck(self._L.hb_part_build(self._h, _p(vecs), vecs.shape[0], _p(t)), "hb_part_build")

    @property
    def n_local(self):
        return int(self._L.hb_part_size(self._h))

    # ---- search
    def search_async(self, slot, q_ptr, nq, k, ef_search, tids_ptr, dist_ptr, root=-1, q_on_device=False, out_on_device=False):
        """hb_part_search_async on raw pointers (ints); complete with search_wait(slot)."""
        self._ck(self._L.hb_part_search_async(self._h, slot, C.c_void_p(q_ptr), int(q_on_device), root, nq, ef_search, k,
                                              C.c_void_p(tids_ptr), C.c_void_p(dist_ptr), int(out_on_device)),
                 "hb_part_search_async")

    def search_wait(self, slot):
        self._ck(self._L.hb_part_search_wait(self._h, slot), "hb_part_search_wait")

    def search_dev(self, q_dev, k=10, ef_search=40, root=-1, slot=0):
        """q_dev: CUDA tensor nq x dim of the index dtype on this rank's GPU, holding the batch on every rank
        (root < 0) or on rank `root` only.  Returns merged nq x k CUDA tensors, identical on every rank."""
        import torch
        torch.cuda.current_stream(q_dev.device).synchronize()        # the library's streams do not know torch's
        nq = q_dev.shape[0]
        out_t = torch.empty((nq, k), dtype=torch.int64, device=q_dev.device)
        out_d = torch.empty((nq, k), dtype=torch.float32, device=q_dev.device)
        torch.cuda.current_stream(q_dev.device).synchronize()
        self.search_async(slot, q_dev.data_ptr(), nq, k, ef_search, out_t.data_ptr(), out_d.data_ptr(), root, True, True)
        self.search_wait(slot)
        return out_t, out_d

    def search(self, queries, k=10, ef_search=40, root=-1):
        """Host arrays in/out (H2D + D2H inside the library)."""
        q = np.ascontiguousarray(queries, _np_dtype(self.dtype))
        if q.ndim == 1:
            q = q[None, :]
        if q.shape[1] != self.dim:
            raise HnswError("expected %d dimensions, not %d" % (self.dim, q.shape[1]))
        nq = q.shape[0]
        tids = np.empty((nq, k), np.int64)
        dist = np.empty((nq, k), np.float32)
        self._ck(self._L.hb_part_search(self._h, _p(q), root, nq, ef_search, k, _p(tids), _p(dist)), "hb_part_search")
        return tids, dist
