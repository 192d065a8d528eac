"""The reference answer of the partitioned search (tests/partition_ref.py) on the CPU: its routing equals the library's,
its answer equals a plain restatement built from the oracle's own gettuple stream, and it is the k smallest
(distance, heap TID) pairs whatever order a partition emits tied TIDs in -- which the greedy merge of gettuple lists
is not."""
import numpy as np
import pytest

import partition_ref as R
from conftest import sift_like


def test_route_equals_library(pkg):
    rng = np.random.default_rng(1)
    tids = np.concatenate([np.arange(1000), rng.integers(0, 1 << 62, 5000), [(1 << 63) - 1, 1 << 32, (1 << 32) - 1]])
    for P in (1, 2, 3, 8, 13, 64):
        assert (R.route(tids, P) == pkg.partition_route(tids, P)).all(), P
    assert pkg.partition_of(12345, 7) == R.route([12345], 7)[0]


def brute(orcs, q, k, ef):
    """Per partition the oracle's gettuple stream of every TID of its ef nearest elements; their union sorted by
    (distance, tid), cut at k."""
    out = []
    for i in range(len(q)):
        pairs = []
        for orc in orcs:
            if orc is None:
                continue
            t, d = orc.search_tids(q[i], ef, ef * R.O.HEAPTIDS)
            pairs += [(float(dd), int(tt)) for tt, dd in zip(t, d)]
        pairs.sort()
        pairs = pairs[:k] + [(float("inf"), -1)] * (k - min(k, len(pairs)))
        out.append(pairs)
    return out


def build_parts(x, tids, P, metric=0, dtype=0, m=8, efc=32, seed=3):
    part = R.route(tids, P)
    orcs = []
    for p in range(P):
        rows = np.nonzero(part == p)[0]
        if len(rows) == 0:
            orcs.append(None)
            continue
        orc = R.O.Index(x.shape[1], m, efc, metric, dtype, R.O.CANON, seed=seed + p)
        orc.build(x[rows], tids[rows])
        orcs.append(orc)
    return orcs


@pytest.mark.parametrize("P,metric,dtype,n", [(1, 0, 0, 600), (3, 1, 0, 600), (5, 2, 0, 600), (4, 3, 1, 600), (64, 0, 1, 80)])
def test_answer_equals_brute_force(oracle, pkg, P, metric, dtype, n):
    dim = 12
    x, tids = R.tie_rows(n, dim, seed=P + metric, copies=25)
    x = x.astype(np.float16 if dtype else np.float32)
    orcs = build_parts(x, tids, P, metric, dtype)
    if P == 64:
        assert any(o is None for o in orcs)           # empty partitions
    # deleted, not vacuumed: elements without heap TIDs stay in the graphs and in the scans
    dead = tids[np.random.default_rng(7).choice(n, n // 5, replace=False)]
    for o in orcs:
        if o is not None:
            o.bulk_delete(dead)
    graphs = [None if o is None else o.export() for o in orcs]
    assert any(((g.ntids == 0).any()) for g in graphs if g is not None)
    assert any(((g.ntids > 1).any()) for g in graphs if g is not None)
    q = np.concatenate([x[:12], sift_like(12, dim, seed=99).astype(x.dtype)])
    for k, ef in ((1, 1), (10, 40), (60, 20), (5, 5)):
        t, d, ctr = R.answer(graphs, q, k, ef)
        want = brute(orcs, q, k, ef)
        for i in range(len(q)):
            assert [(float(a), int(b)) for a, b in zip(d[i], t[i])] == want[i], (k, ef, i)
            assert not set(t[i].tolist()) & set(dead.tolist())
        assert ctr["n_dist"] > 0
        # per-partition answers merged greedily (what the device does) give the same lists, in any grouping
        per = [R.answer([g], q, k, ef)[:2] for g in graphs]
        for i in range(len(q)):
            lists = [(pt[i], pd[i]) for pt, pd in per]
            mt, md = pkg.merge_rule(lists, k)
            assert mt == t[i].tolist() and md == d[i].tolist()
            for world in (2, 3):
                ranks = [pkg.merge_rule([lists[p] for p in range(P) if p % world == r], k) for r in range(world)]
                assert pkg.merge_rule([(np.array(a), np.array(b, np.float32)) for a, b in ranks], k) == (mt, md)


def test_counters_are_summed(oracle):
    x, tids = R.tie_rows(400, 8, seed=5)
    orcs = build_parts(x, tids, 3)
    graphs = [o.export() for o in orcs]
    q = x[:20]
    _, _, ctr = R.answer(graphs, q, 10, 30)
    want = {"n_dist": 0, "n_hop0": 0, "n_hopu": 0}
    for g in graphs:
        c = R.O.Index.from_graph(g).search_batch(q, 30)[3]
        for key in want:
            want[key] += c[key]
    assert ctr == want


def test_empty_inputs(oracle):
    x, tids = R.tie_rows(100, 8, seed=6)
    g = build_parts(x, tids, 1)[0].export()
    t, d, ctr = R.answer([None, g], x[:0], 5, 10)
    assert t.shape == (0, 5) and d.shape == (0, 5)
    t, d, ctr = R.answer([None], x[:3], 5, 10)
    assert (t == -1).all() and np.isinf(d).all() and ctr["n_dist"] == 0


def test_tie_order_is_by_tid_not_by_gettuple(oracle, pkg):
    """Row 10 and two byte copies of it hold TIDs 31, 151 and 154 in one partition (pgvector's gettuple returns them
    154, 151, 31: an element's TIDs last to first); another partition holds a copy with TID 155.  The answer at
    distance 0 is 31, 151, 154, 155; the greedy merge of the gettuple lists gives 154, 151, 31, 155, and with k = 2
    {154, 151} instead of {31, 151}."""
    x = sift_like(60, 8, seed=4)
    a_rows = np.concatenate([x, x[[10, 10]]])
    a_tids = np.concatenate([np.arange(60) * 2 + 1000, [151, 154]])
    a_tids[10] = 31
    A = oracle.Index(8, 8, 32, oracle.L2, 0, oracle.CANON, seed=1)
    A.build(a_rows, a_tids)
    B = oracle.Index(8, 8, 32, oracle.L2, 0, oracle.CANON, seed=2)
    b_tids = np.arange(31, dtype=np.int64) * 2 + 5000          # the last row, a copy of row 10, gets TID 155
    b_tids[30] = 155
    B.build(np.concatenate([sift_like(30, 8, seed=5), x[[10]]]), b_tids)
    q = x[10:11]
    ga, gb = A.export(), B.export()
    t, d, _ = R.answer([ga, gb], q, 4, 20)
    assert t[0].tolist() == [31, 151, 154, 155] and (d[0] == 0).all()
    t2, _, _ = R.answer([ga, gb], q, 2, 20)
    assert t2[0].tolist() == [31, 151]
    # gettuple order of each partition, merged greedily
    ta, da = A.search_tids(q[0], 20, 4)
    tb, db = B.search_tids(q[0], 20, 4)
    assert ta[:3].tolist() == [154, 151, 31] and tb[0] == 155
    assert pkg.merge_rule([(ta, da), (tb, db)], 4)[0] == [154, 151, 31, 155]
    assert pkg.merge_rule([(ta[:2], da[:2]), (tb[:2], db[:2])], 2)[0] == [154, 151]
    # the reference's per-partition lists are sorted by (distance, tid): merging them gives the answer
    per = [R.answer([g], q, 4, 20)[:2] for g in (ga, gb)]
    assert pkg.merge_rule([(pt[0], pd[0]) for pt, pd in per], 4)[0] == [31, 151, 154, 155]
