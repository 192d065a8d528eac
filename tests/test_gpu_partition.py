"""Hash-partitioned index on one GPU (world = 1): routing, per-partition scan, device merge."""
import numpy as np
import pytest

from conftest import clustered, sift_like

pytestmark = pytest.mark.gpu


def test_partitioned_search_matches_exact_scan(oracle, pkg):
    n, dim, nq, k, P = 20000, 64, 300, 10, 4
    x = sift_like(n, dim, seed=1)
    q = sift_like(nq, dim, seed=2)
    tids = np.arange(n, dtype=np.int64) * 3 + 11
    pix = pkg.PartitionedIndex(dim, "vector_l2_ops", P, 16, 64, capacity_per_partition=n, rank=0, world=1, device=0, seed=5)
    assert pix.build(x, tids) == n
    part = pkg.partition_route(tids, P)
    for p, ix in pix.parts.items():
        assert ix.n <= (part == p).sum()          # duplicates fold into one element
    t, d = pix.search(q, k, 60)
    # exact answer over the whole set
    full = oracle.Index(dim, 8, 32, oracle.L2)
    full.build(x[:10])
    d2 = ((q[:, None, :].astype(np.float64) - x[None, :, :].astype(np.float64)) ** 2).sum(-1)
    order = np.argsort(d2, axis=1, kind="stable")[:, :k]
    hits = 0
    for i in range(nq):
        assert np.all(np.diff(d[i]) >= 0)
        got = t[i][t[i] >= 0]
        # distances reported are the true squared distances of the returned rows
        rows = (got - 11) // 3
        assert np.allclose(d[i][:len(got)], d2[i, rows], rtol=1e-5)
        kth = d2[i, order[i, -1]]
        hits += np.sum(d2[i, rows] <= kth * (1 + 1e-6))
    assert hits / (nq * k) >= 0.95
    # merged result == merge of the per-partition results (device merge kernel vs numpy)
    import torch
    qd = torch.tensor(q).cuda()
    per = []
    for p, ix in pix.parts.items():
        pt, pd, _ = ix.search(q, k, 60)
        per.append((pt, pd))
    for i in range(0, nq, 17):
        mt, md = pkg.merge_rule([(pt[i], pd[i]) for pt, pd in per], k)
        assert mt == list(t[i]) and md == [float(v) for v in d[i]]
    pix.close()


# ---- two NCCL ranks (needs two visible devices; skipped on a machine with one GPU) ------------------------
def _nccl_worker(rank, world, port, outq):
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    import torch.distributed as dist
    import pgvector_hnsw_partitioning_b200 as pkg
    from oracle import oracle as O
    from conftest import sift_like
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)      # carries the ncclUniqueId only
    torch.cuda.set_device(rank)
    n, dim, nq, k, P, ef = 12000, 64, 257, 10, 4, 40
    x = sift_like(n, dim, seed=1)                                     # integer-valued: exact distance ties happen
    tids = np.arange(n, dtype=np.int64) * 5 + 2
    pix = pkg.PartitionedIndex(dim, "vector_l2_ops", P, 16, 64, capacity_per_partition=n, rank=rank, world=world,
                               device=rank, seed=5)
    built = pix.build(x, tids)
    assert built == sum(int((pkg.partition_route(tids, P) == p).sum()) for p in pix.owned)
    # three batches in flight; batch b is also searched with the broadcast path (queries on rank 0 only)
    qs = [sift_like(nq, dim, seed=20 + b) for b in range(3)]
    outs = [(np.empty((nq, k), np.int64), np.empty((nq, k), np.float32)) for _ in range(3)]
    for b in range(3):
        pix.search_async(b, qs[b].ctypes.data, nq, k, ef, outs[b][0].ctypes.data, outs[b][1].ctypes.data, root=-1)
    for b in range(3):
        pix.search_wait(b)
    outs_b = [(np.empty((nq, k), np.int64), np.empty((nq, k), np.float32)) for _ in range(3)]
    for b in range(3):
        qp = qs[b].ctypes.data if rank == 0 else 0
        pix.search_async(b, qp, nq, k, ef, outs_b[b][0].ctypes.data, outs_b[b][1].ctypes.data, root=0)
    for b in range(3):
        pix.search_wait(b)
    for b in range(3):
        assert (outs[b][0] == outs_b[b][0]).all() and (outs[b][1] == outs_b[b][1]).all()
    # the exchange over peer memory (default) and the ncclAllGather fallback give the same answer; two rounds per slot so
    # that the epoch / acknowledge flags of a reused slot are exercised
    for exchange in (0, 1):
        pix.set_option("exchange", exchange)
        for rnd in range(2):
            outs_x = [(np.empty((nq, k), np.int64), np.empty((nq, k), np.float32)) for _ in range(3)]
            for b in range(3):
                pix.search_async(b, qs[b].ctypes.data, nq, k, ef, outs_x[b][0].ctypes.data, outs_x[b][1].ctypes.data, root=-1)
            for b in range(3):
                pix.search_wait(b)
            for b in range(3):
                assert (outs[b][0] == outs_x[b][0]).all() and (outs[b][1] == outs_x[b][1]).all(), (exchange, rnd, b)
    # a larger batch re-allocates (and re-maps) the exchange buffers
    qbig = np.concatenate(qs)
    ob = (np.empty((3 * nq, k), np.int64), np.empty((3 * nq, k), np.float32))
    pix.search_async(1, qbig.ctypes.data, 3 * nq, k, ef, ob[0].ctypes.data, ob[1].ctypes.data, root=-1)
    pix.search_wait(1)
    assert (ob[0] == np.concatenate([o[0] for o in outs])).all()
    # the oracle's answer for the partitions this rank owns, on the very graphs the GPU built
    per = {}
    for p, ix in pix.parts.items():
        g = ix.export_graph()
        orc = O.Index.from_graph(g, O.CANON)
        lists = []
        for b in range(3):
            oe, od, oc, _ = orc.search_batch(qs[b], ef, threads=2)
            t = np.full((nq, k), -1, np.int64)
            d = np.full((nq, k), np.inf, np.float32)
            for i in range(nq):
                c = min(int(oc[i]), k)
                t[i, :c] = g.tids[oe[i, :c], 0]
                d[i, :c] = od[i, :c]
            lists.append((t, d))
        per[p] = lists
    outq.put((rank, per, [(t.copy(), d.copy()) for t, d in outs]))
    pix.close()
    dist.destroy_process_group()


def test_two_nccl_ranks_match_oracle_merge(pkg):
    import socket
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    outq = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, outq)) for r in range(2)]
    for p in procs:
        p.start()
    got = [outq.get(timeout=600) for _ in range(2)]
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    per, res = {}, {}
    for rank, pp, outs in got:
        per.update(pp)
        res[rank] = outs
    assert sorted(per) == [0, 1, 2, 3]
    nq, k = res[0][0][0].shape
    ties = 0
    for b in range(3):
        # every rank holds the same answer
        assert (res[0][b][0] == res[1][b][0]).all() and (res[0][b][1] == res[1][b][1]).all()
        for i in range(nq):
            mt, md = pkg.merge_rule([(per[p][b][0][i], per[p][b][1][i]) for p in range(4)], k)
            assert mt == list(res[0][b][0][i]), (b, i)
            assert md == [float(v) for v in res[0][b][1][i]]
            ties += len(md) - len(set(md))
    assert ties > 0          # the data did exercise the (distance, tid) tie rule
