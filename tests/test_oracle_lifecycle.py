"""The delete -> vacuum -> insert lifecycle on the CPU oracle alone (the reference the GPU lifecycle tests compare
against): after every step the graph keeps the invariants of hnswvacuum.c's MarkDeleted, and a graph exported and
imported again searches exactly like the one it came from."""
import numpy as np
import pytest

from lifecycle import Rows, check_invariants, live_tids, run_rounds

CASES = [(0, 0, 24, 8), (1, 0, 32, 8), (2, 0, 40, 12), (0, 1, 24, 8), (1, 1, 48, 8), (2, 1, 20, 8), (3, 0, 28, 8), (3, 1, 36, 8)]


@pytest.mark.parametrize("metric,dtype,dim,m", CASES)
def test_oracle_rounds_keep_invariants(oracle, metric, dtype, dim, m):
    rows = Rows(dim, np.float16 if dtype else np.float32, "clustered", seed=dim + metric)
    x = rows.fresh(1500)
    orc = oracle.Index(dim, m, 2 * m if 2 * m >= 32 else 32, metric, dtype, oracle.CANON, seed=7)
    orc.build(x, rows.tids(x))
    q = rows.fresh(40)
    deleted = set()

    def apply(op, *args):
        if op == "delete":
            deleted.update(int(t) for t in args[0])

    def check(step, marked, after_vacuum):
        g = orc.export()
        check_invariants(g, marked, after_vacuum)
        # the scan returns live heap TIDs only
        have = live_tids(g)
        for i in range(len(q)):
            t, _ = orc.search_tids(q[i], 40, 10)
            assert set(t.tolist()) <= have and not (set(t.tolist()) & deleted), step
        # export -> import: same searches, results and counters
        imp = oracle.Index.from_graph(g)
        a = orc.search_batch(q, 40, threads=2)
        b = imp.search_batch(q, 40, threads=2)
        assert (a[2] == b[2]).all() and (a[0] == b[0]).all() and (a[1].view(np.uint32) == b[1].view(np.uint32)).all(), step
        assert a[3] == b[3], step

    marked = run_rounds(orc, rows, dim, metric == oracle.COSINE, apply, check)
    assert marked and orc.n > 1500


def test_oracle_vacuum_of_everything_then_insert(oracle):
    """Every element vacuumed away: the next insert is a first element at slot n with no neighbours; an imported copy
    of the emptied graph (entry -1) inserts exactly like the original."""
    rows = Rows(16, np.float32, "clustered", seed=3)
    x = rows.fresh(300)
    orc = oracle.Index(16, 8, 32, oracle.L2, 0, oracle.CANON, seed=0)
    orc.build(x, rows.tids(x))
    orc.bulk_delete(np.array(list(rows.by_tid), np.int64))
    assert orc.vacuum_repair()[0] == 300
    assert orc.entry == (-1, -1)
    g0 = orc.export()
    imp = oracle.Index.from_graph(g0)
    assert imp.entry == (-1, -1)
    y = rows.fresh(60)
    t = rows.tids(y)
    assert imp.insert(y[0], int(t[0])) == 300
    g = imp.export()
    lv = int(g.level[300])
    assert g.entry == 300 and g.entry_level == lv
    assert g.uoff[300] == (g0.upper_rows if lv > 0 else -1) and g.upper_rows == g0.upper_rows + lv
    assert (g.nbr0[300] == -1).all()
    for i in range(1, 60):
        assert imp.insert(y[i], int(t[i])) == 300 + i
    g = imp.export()
    check_invariants(g, set(range(300)), True)
    assert g.entry >= 300 and g.level[g.entry] == g.level[300:].max()
    assert (g.nbr0[300] >= 0).any()                  # later elements linked back to the first one
