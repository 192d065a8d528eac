"""The hash-partitioned index on one GPU (world = 1) against the CPU oracle, bit for bit.

Reference: tests/partition_ref.py on the graphs the partitions export -- the k smallest (distance, heap TID) pairs
over every heap TID of the elements each partition's scan returned.  Every comparison is exact: TIDs equal, distance
bits equal, each row ordered by (distance, TID).  The data is made for ties: integer-valued rows, byte copies folded
into shared elements (one row copied into several elements), heap TIDs that grow neither with row nor insertion
order."""
import os

import numpy as np
import pytest

import partition_ref as R
from conftest import sift_like

pytestmark = pytest.mark.gpu

THREADS = max(1, min(16, os.cpu_count() or 1))
KEF = ((1, 1), (10, 40), (100, 40), (255, 200), (40, 10))          # (100, 40) and (40, 10): k > ef_search
NQ_ALL = (1, 7, 148, 149, 2000)
# opclass, dim, rows, batch sizes.  768-d cosine: nq <= 148 takes the CTA-per-query kernel, more the warp kernels;
# 128-d: ef <= 104 the register-list kernel, ef = 200 the shared-memory list.
CASES = [("vector_l2_ops", 128, 6000, NQ_ALL), ("vector_ip_ops", 100, 3000, (7, 149)),
         ("vector_cosine_ops", 768, 2500, NQ_ALL), ("vector_l1_ops", 24, 3000, (1, 149)),
         ("halfvec_l2_ops", 24, 3000, (7, 149)), ("halfvec_ip_ops", 1536, 1200, (1, 149)),
         ("halfvec_cosine_ops", 100, 3000, (7, 148)), ("halfvec_l1_ops", 128, 3000, (7, 149))]


def _dt(pkg, opclass):
    return np.float16 if pkg.OPCLASSES[opclass][1] else np.float32


def queries(x, nq, seed):
    """The row with the most byte copies first, then other indexed rows (distance-0 ties), then fresh rows."""
    _, inv, cnt = np.unique(x, axis=0, return_inverse=True, return_counts=True)
    inv = inv.reshape(-1)
    order = np.argsort(-cnt[inv], kind="stable")
    head = x[order[:min(nq, 4)]]
    rest = sift_like(nq, x.shape[1], seed=seed).astype(x.dtype)
    rng = np.random.default_rng(seed)
    rest[::5] = x[rng.integers(0, len(x), len(rest[::5]))]
    return np.ascontiguousarray(np.concatenate([head, rest])[:nq])


def export_all(pix):
    return [pix.parts[p].export_graph() for p in pix.owned]


def check(t, d, rt, rd, what=""):
    """exact equality with the reference, and rows ordered by (distance, tid) with the pads last"""
    bad = np.nonzero((t != rt).any(axis=1) | (d.view(np.uint32) != rd.view(np.uint32)).any(axis=1))[0]
    assert len(bad) == 0, "%s: %d of %d rows differ, first %d: got %s / %s, want %s / %s" % (
        what, len(bad), len(t), bad[0], t[bad[0]][:12], d[bad[0]][:12], rt[bad[0]][:12], rd[bad[0]][:12])
    pad = t < 0
    assert (np.isinf(d) == pad).all() and (pad[:, :-1] <= pad[:, 1:]).all(), what
    a, b = (d[:, :-1], t[:, :-1]), (d[:, 1:], t[:, 1:])
    assert ((a[0] < b[0]) | ((a[0] == b[0]) & (a[1] < b[1])) | pad[:, 1:]).all(), what


def make(pkg, opclass, dim, P, x, tids, seed=5):
    pix = pkg.PartitionedIndex(dim, opclass, P, 16, 64, capacity_per_partition=len(x) + 64, rank=0, world=1, device=0,
                               seed=seed)
    assert pix.build(x, tids) == len(x)
    return pix


# ---- a. parity matrix: every operator class, P in {1, 3, 8} -----------------------------------------------------
@pytest.mark.parametrize("P", [1, 3, 8])
@pytest.mark.parametrize("opclass,dim,n,nqs", CASES, ids=[c[0] + "-%d" % c[1] for c in CASES])
def test_parity_matrix(oracle, pkg, opclass, dim, n, nqs, P):
    x, tids = R.tie_rows(n, dim, seed=dim + P, dtype=_dt(pkg, opclass))
    pix = make(pkg, opclass, dim, P, x, tids)
    graphs = export_all(pix)
    assert sum(g.n for g in graphs) == pix.n_local < n                    # byte copies folded
    assert max(int(g.ntids.max()) for g in graphs) >= 2
    q = queries(x, max(nqs), seed=dim + 100 + P)
    kmax = {}
    for k, ef in KEF:
        kmax[ef] = max(kmax.get(ef, 0), k)
    ref = {ef: R.answer(graphs, q, kk, ef, THREADS) for ef, kk in kmax.items()}
    ties = 0
    for k, ef in KEF:
        rt, rd, rc = ref[ef]
        for nq in sorted(nqs):
            if nq == max(nqs):
                pix.counters(reset=True)
            t, d = pix.search(q[:nq], k, ef)
            check(t, d, rt[:nq, :k], rd[:nq, :k], "%s P=%d k=%d ef=%d nq=%d" % (opclass, P, k, ef, nq))
        c = pix.counters()
        assert (c["n_dist"], c["n_hop0"], c["n_hopu"]) == (rc["n_dist"], rc["n_hop0"], rc["n_hopu"]), (k, ef, c, rc)
        ties += int((d[:, 1:] == d[:, :-1]).sum())
    assert ties > 0                       # the data exercised the (distance, tid) order
    pix.close()


# ---- b. edges -----------------------------------------------------------------------------------------------------
def test_many_partitions_mostly_empty(oracle, pkg):
    """P = 64 with 40 rows: most partitions are empty (their lists are padding), some hold a single element."""
    x, tids = R.tie_rows(100, 16, seed=3, copies=8)
    x, tids = x[:40], tids[:40]
    pix = make(pkg, "vector_l2_ops", 16, 64, x, tids)
    graphs = export_all(pix)
    sizes = [g.n for g in graphs]
    assert sizes.count(0) > 20 and sizes.count(1) > 0
    q = queries(x, 50, seed=4)
    for k, ef in KEF:
        pix.counters(reset=True)
        t, d = pix.search(q, k, ef)
        rt, rd, rc = R.answer(graphs, q, k, ef, THREADS)
        check(t, d, rt, rd, "P=64 k=%d ef=%d" % (k, ef))
        assert pix.counters()["n_dist"] == rc["n_dist"]
    pix.close()


@pytest.mark.parametrize("P", [1, 3])
def test_empty_handle_and_empty_batch(pkg, P):
    pix = pkg.PartitionedIndex(8, "vector_l2_ops", P, 8, 32, capacity_per_partition=16, rank=0, world=1, device=0)
    q = sift_like(5, 8, seed=1)
    t, d = pix.search(q, 7, 20)
    assert (t == -1).all() and np.isinf(d).all() and (d > 0).all()
    assert pix.build(q[:0]) == 0 and pix.n_local == 0
    # nq = 0: OK, and the output buffers are not written
    ot = np.full((1, 7), 12345, np.int64)
    od = np.full((1, 7), 2.5, np.float32)
    for slot in range(4):                      # HB_PART_SLOTS
        pix.search_async(slot, q.ctypes.data, 0, 7, 20, ot.ctypes.data, od.ctypes.data)
        pix.search_wait(slot)
    assert (ot == 12345).all() and (od == 2.5).all()
    t, d = pix.search(q[:0], 7, 20)
    assert t.shape == (0, 7)
    pix.close()


def test_argument_errors(pkg):
    x, tids = R.tie_rows(300, 8, seed=2, copies=4)
    pix = make(pkg, "vector_l2_ops", 8, 2, x, tids)
    q = x[:3].copy()
    ot = np.empty((3, 256), np.int64)
    od = np.empty((3, 256), np.float32)
    for slot, k, ef in ((4, 10, 40), (-1, 10, 40), (0, 0, 40), (0, 256, 40), (0, 10, 0), (0, 10, 1001)):
        with pytest.raises(pkg.HnswError):
            pix.search_async(slot, q.ctypes.data, 3, k, ef, ot.ctypes.data, od.ctypes.data)
    # a slot with a batch in flight refuses another one until its wait (HB_ESTATE); the other slots do not
    ot2, od2 = np.empty((3, 10), np.int64), np.empty((3, 10), np.float32)
    pix.search_async(1, q.ctypes.data, 3, 10, 40, ot.ctypes.data, od.ctypes.data)
    with pytest.raises(pkg.HnswError, match="in flight"):
        pix.search_async(1, q.ctypes.data, 3, 10, 40, ot.ctypes.data, od.ctypes.data)
    pix.search_async(2, q.ctypes.data, 3, 10, 40, ot2.ctypes.data, od2.ctypes.data)
    pix.search_wait(1)
    pix.search_wait(2)
    got = ot.reshape(-1)[:30].reshape(3, 10), od.reshape(-1)[:30].reshape(3, 10)
    t, d = pix.search(q, 10, 40)
    for a, b in (got, (ot2, od2)):
        assert (a == t).all() and (b.view(np.uint32) == d.view(np.uint32)).all()
    pix.close()


# ---- c. build -----------------------------------------------------------------------------------------------------
def graphs_equal(a, b, what=""):
    assert a.n == b.n and a.entry == b.entry and a.upper_rows == b.upper_rows, what
    assert (a.level == b.level).all() and (a.uoff == b.uoff).all(), what
    assert (a.vecs.view(np.uint8) == b.vecs.view(np.uint8)).all(), what
    bad = np.nonzero((a.nbr0 != b.nbr0).any(axis=1))[0]
    assert len(bad) == 0, "%s: layer-0 lists differ for %d elements, first %s" % (what, len(bad), bad[:5])
    if a.upper_rows:
        assert (a.nbru[:a.upper_rows] == b.nbru[:b.upper_rows]).all(), what
    assert (a.ntids == b.ntids).all(), what
    for e in range(a.n):
        assert (a.tids[e, :a.ntids[e]] == b.tids[e, :b.ntids[e]]).all(), (what, e)


def copies_routed(x, tids, P, rng, same, n):
    """n byte copies of indexed rows with new heap TIDs that route to the original's partition (same) or elsewhere"""
    part = R.route(tids, P)
    rows, new = [], []
    cand = int(tids.max()) + 1
    while len(rows) < n:
        i = int(rng.integers(0, len(x)))
        while (R.route([cand], P)[0] == part[i]) != same:
            cand += 1
        rows.append(x[i])
        new.append(cand)
        cand += 1
    return np.stack(rows), np.array(new, np.int64)


@pytest.mark.parametrize("opclass,metric,dtype,dim,P", [("vector_l2_ops", 0, 0, 32, 3), ("halfvec_cosine_ops", 2, 1, 24, 1),
                                                        ("vector_l1_ops", 3, 0, 20, 3)])
def test_sequential_build_and_inserts_equal_oracle(oracle, pkg, opclass, metric, dtype, dim, P):
    """build_batch = 1: every partition's graph is the oracle's sequential build of the rows routed to it, in row order,
    with seed + p -- for the first build and for two more calls, which insert: byte copies of indexed rows with TIDs of
    the same partition (they fold) and of other partitions, then rows without heap TIDs (TID = row number; with P = 1
    the rows are indexed in place)."""
    dt = np.float16 if dtype else np.float32
    x, tids = R.tie_rows(1200, dim, seed=dim, dtype=dt)
    rng = np.random.default_rng(dim)
    pix = pkg.PartitionedIndex(dim, opclass, P, 8, 32, capacity_per_partition=2000, rank=0, world=1, device=0, seed=9)
    pix.set_option("build_batch", 1)
    orcs = [oracle.Index(dim, 8, 32, metric, dtype, oracle.CANON, seed=9 + p) for p in range(P)]
    a, ta = copies_routed(x, tids, P, rng, True, 30)
    b, tb = copies_routed(x, tids, P, rng, False, 30) if P > 1 else (a[:0], ta[:0])
    y = np.concatenate([a, b, sift_like(60, dim, seed=dim + 1).astype(dt)])
    perm = rng.permutation(len(y))
    y, ty = y[perm], np.concatenate([ta, tb, np.zeros(60, np.int64)])[perm]
    fresh = ty == 0
    ty[fresh] = (1 << 41) + np.arange(fresh.sum())
    z = sift_like(40, dim, seed=dim + 2).astype(dt)
    z[:5] = x[:5]
    for step, (rows, t, given) in enumerate(((x, tids, True), (y, ty, True), (z, np.arange(len(z)), False))):
        got = pix.build(rows, t if given else None)
        assert got == len(rows), step
        part = R.route(t, P)
        for p in range(P):
            sel = np.nonzero(part == p)[0]
            orcs[p].build(rows[sel], t[sel])
        for p in range(P):
            graphs_equal(orcs[p].export(), pix.parts[p].export_graph(), "step %d partition %d" % (step, p))
        assert pix.n_local == sum(o.n for o in orcs)
    assert any((o.export().ntids > 1).any() for o in orcs)
    q = queries(x, 40, seed=1)
    t, d = pix.search(q, 30, 50)
    rt, rd, _ = R.answer(export_all(pix), q, 30, 50, THREADS)
    check(t, d, rt, rd, "after inserts")
    pix.close()


def test_concurrent_build_equals_standalone(oracle, pkg):
    """Default batching: the partitions are built concurrently, one host thread each; every graph equals a standalone
    HnswIndex (seed + p) given the same rows, for the build and for an insert."""
    dim, P = 64, 4
    x, tids = R.tie_rows(12000, dim, seed=8)
    y, ty = R.tie_rows(3000, dim, seed=9)
    ty += int(tids.max()) + 1
    pix = make(pkg, "vector_l2_ops", dim, P, x, tids, seed=11)
    assert pix.build(y, ty) == len(y)
    for p in range(P):
        ix = pkg.HnswIndex(dim, "vector_l2_ops", 16, 64, capacity=len(x) + 64, seed=11 + p)
        for rows, t in ((x, tids), (y, ty)):
            sel = R.route(t, P) == p
            ix.insert(rows[sel], t[sel])
        graphs_equal(ix.export_graph(), pix.parts[p].export_graph(), "partition %d" % p)
        ix.close()
    pix.close()


# ---- d. batches in flight -----------------------------------------------------------------------------------------
def test_four_slots_in_flight(oracle, pkg):
    """Four batches on slots 0..3 at once, each with its own nq, k and ef, host and device buffers mixed; each equals
    the synchronous search of that batch and the reference.  Then one slot is reused with a larger and a smaller batch."""
    import torch
    dim, P = 128, 8
    x, tids = R.tie_rows(8000, dim, seed=12)
    pix = make(pkg, "vector_l2_ops", dim, P, x, tids)
    graphs = export_all(pix)
    dev = torch.device("cuda", 0)
    # (nq, k, ef, queries on device, outputs on device)
    plan = [(300, 10, 40, False, False), (149, 255, 200, True, True), (1000, 100, 40, False, True), (7, 40, 10, True, False)]
    qs = [queries(x, nq, seed=20 + s) for s, (nq, _, _, _, _) in enumerate(plan)]
    want = [pix.search(qs[s], k, ef) for s, (_, k, ef, _, _) in enumerate(plan)]
    for s, (nq, k, ef, _, _) in enumerate(plan):
        rt, rd, _ = R.answer(graphs, qs[s], k, ef, THREADS)
        check(want[s][0], want[s][1], rt, rd, "slot %d synchronous" % s)

    def issue(slot, q, k, ef, qdev, odev):
        nq = len(q)
        if qdev:
            qb = torch.from_numpy(q).to(dev)
        else:
            qb = q
        if odev:
            ob = (torch.empty((nq, k), dtype=torch.int64, device=dev), torch.empty((nq, k), dtype=torch.float32, device=dev))
            ptrs = ob[0].data_ptr(), ob[1].data_ptr()
        else:
            ob = (np.empty((nq, k), np.int64), np.empty((nq, k), np.float32))
            ptrs = ob[0].ctypes.data, ob[1].ctypes.data
        torch.cuda.synchronize()
        pix.search_async(slot, qb.data_ptr() if qdev else qb.ctypes.data, nq, k, ef, ptrs[0], ptrs[1],
                         q_on_device=qdev, out_on_device=odev)
        return qb, ob

    def fetch(ob):
        return tuple(o.cpu().numpy() if hasattr(o, "cpu") else o for o in ob)

    keep = [issue(s, qs[s], k, ef, qd, od) for s, (nq, k, ef, qd, od) in enumerate(plan)]
    for s in (2, 0, 3, 1):
        pix.search_wait(s)
    for s in range(4):
        t, d = fetch(keep[s][1])
        check(t, d, want[s][0], want[s][1], "slot %d in flight" % s)
    # slot 2 again: a larger batch (buffers grow), then a smaller one
    for nq, k, ef in ((2000, 20, 60), (5, 255, 300)):
        q = queries(x, nq, seed=nq)
        _, ob = issue(2, q, k, ef, True, False)
        pix.search_wait(2)
        t, d = fetch(ob)
        rt, rd, _ = R.answer(graphs, q, k, ef, THREADS)
        check(t, d, rt, rd, "slot 2 reused, nq=%d" % nq)
    pix.close()


# ---- e. delete and vacuum through the partition views ---------------------------------------------------------------
def test_delete_and_vacuum_through_views(oracle, pkg):
    dim, P = 48, 4
    x, tids = R.tie_rows(6000, dim, seed=13)
    pix = make(pkg, "vector_l2_ops", dim, P, x, tids)
    rng = np.random.default_rng(13)
    part = R.route(tids, P)
    dead = set(rng.choice(tids, int(0.3 * len(tids)), replace=False).tolist()) | set(tids[part == 2].tolist())
    dead_arr = np.array(sorted(dead), np.int64)
    removed = sum(pix.parts[p].bulk_delete(dead_arr) for p in pix.owned)
    assert removed == len(dead)
    q = queries(x, 200, seed=14)
    for stage in ("deleted", "vacuumed"):
        if stage == "vacuumed":
            for p in pix.owned:
                pix.parts[p].vacuum_repair()
        graphs = export_all(pix)
        assert not (graphs[2].ntids > 0).any()
        if stage == "vacuumed":
            assert graphs[2].entry == -1
        for k, ef in ((10, 40), (255, 200), (40, 10)):
            t, d = pix.search(q, k, ef)
            rt, rd, _ = R.answer(graphs, q, k, ef, THREADS)
            check(t, d, rt, rd, "%s k=%d ef=%d" % (stage, k, ef))
            assert not (set(np.unique(t).tolist()) & dead)
            assert (t >= 0).any()
    pix.close()
