"""The mutation path ambulkdelete / aminsert call -- hb_bulk_delete -> hb_vacuum_repair -> hb_insert -- over several
rounds, against the CPU oracle in lock-step.  build_batch = 1 and vacuum_batch = 1 make the GPU path the sequential
algorithm, so after every step the graph must be IDENTICAL to the oracle's and every scan kernel must return the
oracle's ids, distances and counters bit for bit.  Batched repair is held to structural invariants and recall."""
import numpy as np
import pytest

from conftest import clustered
from lifecycle import Rows, check_invariants, live_tids, run_rounds
from pgpages_writer import write_pages
from test_gpu_build import OPC, graphs_equal

pytestmark = pytest.mark.gpu

OPC_ALL = {**OPC, (3, 0): "vector_l1_ops", (3, 1): "halfvec_l1_ops"}


def sequential_pair(oracle, pkg, x, tids, metric, dtype, m, efc, seed):
    orc = oracle.Index(x.shape[1], m, efc, metric, dtype, oracle.CANON, seed=seed)
    orc.build(x, tids)
    ix = pkg.HnswIndex(x.shape[1], OPC_ALL[(metric, dtype)], m, efc, capacity=x.shape[0], seed=seed)
    ix.set_option("build_batch", 1)
    ix.set_option("vacuum_batch", 1)
    if len(x):
        assert ix.build(x, tids) == orc.n
    return orc, ix


def scans_equal(orc, ix, q, ef=40, variants=(0, 7, 9), step=""):
    """search_elements under each kernel variant: ids, distances and counters bit-equal to the oracle's"""
    oe, od, oc, octr = orc.search_batch(q, ef, threads=4)
    for v in variants:
        ix.set_option("variant", v)
        ix.counters(reset=True)
        e, d, c = ix.search_elements(q, ef)
        ctr = ix.counters()
        assert (c == oc).all(), (step, v)
        assert (e == oe).all(), (step, v, int((e != oe).any(axis=1).sum()))
        assert (d.view(np.uint32) == od.view(np.uint32)).all(), (step, v)
        assert all(ctr[k] == octr[k] for k in ("n_dist", "n_hop0", "n_hopu")), (step, v, ctr, octr)
    ix.set_option("variant", 0)


def iterate_equal(orc, ix, q, ef=20, max_tuples=300, step=""):
    want = [orc.iterate(q[i], ef, max_scan_tuples=max_tuples) for i in range(len(q))]
    it = ix.iterate(q, ef, max_tuples)
    nb = 0
    while True:
        r = it.next()
        if r is None:
            break
        e, d, c = r
        for i in range(len(q)):
            batches = want[i][0]
            if nb < len(batches):
                we, wd = batches[nb]
                assert c[i] == len(we) and (e[i, :c[i]] == we).all(), (step, i, nb)
                assert (d[i, :c[i]].view(np.uint32) == wd.view(np.uint32)).all(), (step, i, nb)
            else:
                assert c[i] == 0, (step, i, nb)
        nb += 1
        assert nb < 10000
    assert nb == max([len(w[0]) for w in want] + [0]), step
    assert (it.tuples() == np.array([w[1] for w in want])).all(), step
    it.close()


def same_everything(orc, ix, q, marked, after_vacuum, deleted, step):
    go, gg = orc.export(), ix.export_graph()
    graphs_equal(go, gg)
    assert ix.entry == orc.entry, step
    check_invariants(gg, marked, after_vacuum)
    scans_equal(orc, ix, q, step=step)
    iterate_equal(orc, ix, q[:6], step=step)
    t, _, c = ix.search(q, 10, 40)
    got = set(t[t >= 0].tolist())
    assert got <= live_tids(gg) and not (got & deleted), step


# (metric, dtype, dim, m, generator): all eight operator classes; 128-d integer-valued rows take the register-list scan
# kernel and tie exactly; 384-d fp32 rows (1536 bytes) are what the four-warps-per-query kernel is chosen for on its own
ROUND_CASES = [(0, 0, 24, 8, "clustered"), (1, 0, 32, 8, "clustered"), (2, 0, 40, 12, "clustered"), (0, 1, 24, 8, "clustered"),
               (1, 1, 48, 8, "clustered"), (2, 1, 20, 8, "clustered"), (3, 0, 28, 8, "clustered"), (3, 1, 36, 8, "clustered"),
               (0, 0, 128, 16, "sift"), (2, 0, 384, 16, "clustered")]


@pytest.mark.parametrize("metric,dtype,dim,m,gen", ROUND_CASES)
def test_rounds_identical_to_oracle(oracle, pkg, metric, dtype, dim, m, gen):
    """four rounds of insert (fresh rows, byte copies of live and of emptied rows, a zero vector under cosine) -> bulk
    delete (10 / 40 / 0 / 70 % of the live TIDs, always the entry point's, some TIDs of multi-TID elements, a missing
    TID) -> vacuum (skipped in round 1)"""
    rows = Rows(dim, np.float16 if dtype else np.float32, gen, seed=dim + metric)
    x = rows.fresh(1500)
    orc, ix = sequential_pair(oracle, pkg, x, rows.tids(x), metric, dtype, m, max(2 * m, 32), seed=5)
    q = rows.fresh(50)
    deleted = set()

    def apply(op, *args):
        if op == "insert":
            xs, ts, want = args
            assert ix.insert(xs, ts) == want
        elif op == "delete":
            dead, want = args
            assert ix.bulk_delete(dead) == want
            deleted.update(dead.tolist())
        else:
            got = ix.vacuum_repair()
            assert got == args[0]

    def check(step, marked, after_vacuum):
        same_everything(orc, ix, q, marked, after_vacuum, deleted, step)

    same_everything(orc, ix, q, set(), True, deleted, "build")
    run_rounds(orc, rows, dim, metric == oracle.COSINE, apply, check)
    ix.close()


def exact_tids(x, tids, q, metric, k=10):
    """exact top-k heap TIDs by a float64 scan (ties are negligible on these rows)"""
    a, b = x.astype(np.float64), q.astype(np.float64)
    if metric == 2:
        a = a / np.linalg.norm(a, axis=1, keepdims=True)
        b = b / np.linalg.norm(b, axis=1, keepdims=True)
    if metric == 0:
        s = (b * b).sum(1)[:, None] - 2 * b @ a.T + (a * a).sum(1)[None, :]
    else:
        s = -(b @ a.T)
    return tids[np.argsort(s, axis=1, kind="stable")[:, :k]]


def recall(t, gt):
    return float(np.mean([len(set(t[i].tolist()) & set(gt[i].tolist())) / gt.shape[1] for i in range(len(gt))]))


@pytest.mark.parametrize("metric,dtype,dim", [(0, 0, 16), (2, 0, 24), (1, 1, 32)])
def test_insert_after_vacuum_of_everything(oracle, pkg, metric, dtype, dim):
    dt = np.float16 if dtype else np.float32
    rows = Rows(dim, dt, "clustered", seed=dim)
    x = rows.fresh(300)
    tx = rows.tids(x)
    orc, ix = sequential_pair(oracle, pkg, x, tx, metric, dtype, 8, 32, seed=4)
    q = rows.fresh(30)
    deleted = set(tx.tolist())
    assert ix.bulk_delete(tx) == orc.bulk_delete(tx) == 300
    assert ix.vacuum_repair() == orc.vacuum_repair()
    assert ix.entry == orc.entry == (-1, -1)
    t, _, c = ix.search(q, 10, 40)
    assert (c == 0).all()
    same_everything(orc, ix, q, set(range(300)), True, deleted, "emptied")
    up0 = ix.export_graph().upper_rows
    # one row at a time: the first lands at slot 300 with its level, its upper rows after the old ones, empty lists
    y = rows.fresh(60)
    ty = rows.tids(y)
    for i in range(60):
        assert ix.insert(y[i:i + 1], ty[i:i + 1]) == 1
        assert orc.insert(y[i], int(ty[i])) == 300 + i
        if i == 0:
            g = ix.export_graph()
            lv = int(g.level[300])
            assert ix.entry == (300, lv) and g.n == 301
            assert g.uoff[300] == (up0 if lv > 0 else -1) and g.upper_rows == up0 + lv
            assert (g.nbr0[300] == -1).all() and g.ntids[300] == 1 and g.tids[300, 0] == ty[0]
    same_everything(orc, ix, q, set(range(300)), False, deleted, "refilled")
    # a second round of delete everything + vacuum + insert
    assert ix.bulk_delete(ty) == orc.bulk_delete(ty) == 60
    deleted |= set(ty.tolist())
    assert ix.vacuum_repair() == orc.vacuum_repair()
    same_everything(orc, ix, q, set(range(360)), True, deleted, "emptied again")
    z = rows.fresh(40)
    tz = rows.tids(z)
    assert ix.insert(z, tz) == 40
    for i in range(40):
        orc.insert(z[i], int(tz[i]))
    same_everything(orc, ix, q, set(range(360)), False, deleted, "refilled again")
    ix.close()
    # default batching on a fresh copy of the emptied index: a valid graph with good recall over the new rows
    ix2 = pkg.HnswIndex(dim, OPC_ALL[(metric, dtype)], 8, 32, capacity=300, seed=4)
    assert ix2.build(x, tx) == 300
    assert ix2.bulk_delete(tx) == 300 and ix2.vacuum_repair()[0] == 300
    y2 = rows.fresh(1000)
    t2 = rows.tids(y2)
    assert ix2.insert(y2, t2) == 1000
    g = ix2.export_graph()
    check_invariants(g, set(range(300)), True)
    q2 = rows.fresh(200)
    got, _, _ = ix2.search(q2, 10, 64)
    r = recall(got, exact_tids(y2, t2, q2, metric))
    assert r >= 0.95, r
    ix2.close()


def test_insert_between_delete_of_everything_and_vacuum(oracle, pkg):
    """every TID deleted, rows inserted while the emptied elements (and the emptied entry point) are still in the graph,
    then vacuum: the entry point moves from an emptied element to a live one"""
    rows = Rows(20, np.float32, "clustered", seed=21)
    x = rows.fresh(300)
    tx = rows.tids(x)
    orc, ix = sequential_pair(oracle, pkg, x, tx, 0, 0, 8, 32, seed=6)
    q = rows.fresh(30)
    assert ix.bulk_delete(tx) == orc.bulk_delete(tx) == 300
    y = rows.fresh(40)
    ty = rows.tids(y)
    assert ix.insert(y, ty) == 40
    for i in range(40):
        orc.insert(y[i], int(ty[i]))
    old = orc.entry[0]
    same_everything(orc, ix, q, set(), False, set(tx.tolist()), "inserted")
    assert ix.vacuum_repair() == orc.vacuum_repair()
    assert orc.entry[0] >= 300 and orc.entry[0] != old
    same_everything(orc, ix, q, set(range(300)), True, set(tx.tolist()), "vacuumed")
    ix.close()


def cluster_labels(n, d, n_centres, seed):
    """the centre each row of conftest.clustered(n, d, n_centres, seed) was drawn around"""
    return np.random.default_rng(seed).integers(0, n_centres, n)


@pytest.mark.parametrize("case", ["random90", "random99", "densest60"])
def test_vacuum_after_heavy_deletes(oracle, pkg, case):
    """Emptied elements stay in the search list of the repair search without counting towards ef_construction, so the
    list grows with the emptied elements a search meets -- well past ef_construction + the tie allowance after heavy
    deletes.  Elements whose list outgrows the per-warp list are searched again with a larger one."""
    n, dim, m, efc = 20000, 16, 8, 32
    x = clustered(n, dim, 32, seed=61)
    rng = np.random.default_rng(62)
    gone_centres = []
    if case == "densest60":
        lab = cluster_labels(n, dim, 32, 61)
        dead_rows = []
        for c in np.argsort(-np.bincount(lab, minlength=32), kind="stable"):
            if len(dead_rows) >= 0.6 * n:
                break
            dead_rows.extend(np.nonzero(lab == c)[0].tolist())
            gone_centres.append(int(c))
        dead = np.array(sorted(dead_rows), np.int64)
    else:
        dead = np.sort(rng.choice(n, int(n * (0.90 if case == "random90" else 0.99)), replace=False)).astype(np.int64)
    orc = oracle.Index(dim, m, efc, 0, 0, oracle.CANON, seed=8)
    orc.build(x)
    g0 = orc.export()
    ix = pkg.HnswIndex(dim, "vector_l2_ops", m, efc, capacity=n, seed=8)
    ix.load_graph(g0)
    ix.set_option("vacuum_batch", 1)
    assert ix.bulk_delete(dead) == orc.bulk_delete(dead) == len(dead)
    got, want = ix.vacuum_repair(), orc.vacuum_repair()
    assert got == want and got[0] == len(dead)
    nq = 300
    q = clustered(nq, dim, 32, seed=63)
    graphs_equal(orc.export(), ix.export_graph())
    check_invariants(ix.export_graph(), set(dead.tolist()), True)
    scans_equal(orc, ix, q, variants=(0, 7))
    ix.close()
    # default batches on a fresh copy: invariants, and recall against the exact answer over the live rows
    ix = pkg.HnswIndex(dim, "vector_l2_ops", m, efc, capacity=n, seed=8)
    ix.load_graph(g0)
    assert ix.bulk_delete(dead) == len(dead)
    marked, repaired = ix.vacuum_repair()
    assert marked == len(dead) and repaired > 0
    check_invariants(ix.export_graph(), set(dead.tolist()), True)
    alive = np.ones(n, bool)
    alive[dead] = False
    live = np.nonzero(alive)[0]
    gt = exact_tids(x[live], live, q, 0)
    t, _, _ = ix.search(q, 10, 64)
    per_query = lambda ids: np.array([len(set(ids[i].tolist()) & set(gt[i].tolist())) / 10 for i in range(nq)])
    r_gpu = per_query(t)
    # the sequential repair (the oracle's graph) on the same queries
    r_seq = per_query(np.array([np.pad(orc.search_tids(q[i], 64, 10)[0], (0, 10), constant_values=-1)[:10] for i in range(nq)]))
    assert r_gpu.mean() >= r_seq.mean() - 0.02, (r_gpu.mean(), r_seq.mean())
    # queries drawn around a centre whose rows all left have no near neighbours: their nearest live rows lie about
    # equally far in every surviving cluster, and a graph search finds ~2/3 of them -- the oracle's sequentially repaired
    # graph and a fresh build of the live rows alike (0.64 and 0.63 at ef_search 64 on these rows).  Queries among the
    # live rows must be answered well.
    near_live = ~np.isin(cluster_labels(nq, dim, 32, 63), gone_centres)
    assert near_live.sum() >= 100
    assert r_gpu[near_live].mean() >= 0.95, (r_gpu[near_live].mean(), r_seq[near_live].mean())
    ix.close()


@pytest.mark.parametrize("survivor", ["entry", "level0"])
def test_single_live_element(oracle, pkg, survivor):
    """one element left: the entry point itself, or a level-0 element that then becomes the entry point; then the
    survivor goes too"""
    rows = Rows(16, np.float32, "clustered", seed=71)
    x = rows.fresh(400)
    tx = rows.tids(x)
    orc, ix = sequential_pair(oracle, pkg, x, tx, 0, 0, 8, 32, seed=9)
    q = rows.fresh(20)
    g = orc.export()
    keep = g.entry if survivor == "entry" else int(next(e for e in range(g.n) if g.level[e] == 0 and e != g.entry))
    dead = tx[np.arange(400) != keep]
    assert ix.bulk_delete(dead) == orc.bulk_delete(dead) == 399
    assert ix.vacuum_repair() == orc.vacuum_repair()
    assert orc.entry == (keep, int(g.level[keep]))
    gone = set(range(400)) - {keep}
    same_everything(orc, ix, q, gone, True, set(dead.tolist()), "one left")
    t, d, c = ix.search(q, 10, 40)
    assert (c == 1).all() and (t[:, 0] == tx[keep]).all()
    assert ix.bulk_delete(tx[keep:keep + 1]) == orc.bulk_delete(tx[keep:keep + 1]) == 1
    assert ix.vacuum_repair() == orc.vacuum_repair() == (1, 0)
    assert ix.entry == orc.entry == (-1, -1)
    same_everything(orc, ix, q, set(range(400)), True, set(tx.tolist()), "none left")
    ix.close()


@pytest.mark.parametrize("emptied", ["partly", "fully"])
def test_vacuumed_graph_round_trip(oracle, pkg, emptied):
    """A vacuumed graph through export_graph -> load_graph and through pgvector index pages (deleted elements flagged;
    no entry point when nothing is left) loads and searches like the oracle's import of it; inserts after the load equal
    the imported oracle's (both start their level draws at seq = n with seed 0)."""
    dim, m, efc = 24, 8, 32
    rows = Rows(dim, np.float32, "clustered", seed=81)
    x = rows.fresh(600)
    tx = rows.tids(x)
    orc, ix = sequential_pair(oracle, pkg, x, tx, 2, 0, m, efc, seed=3)
    g = orc.export()
    dead = tx if emptied == "fully" else np.unique(np.concatenate([np.random.default_rng(82).choice(tx, 300, replace=False),
                                                                  g.tids[g.entry, :g.ntids[g.entry]]]))
    assert ix.bulk_delete(dead) == orc.bulk_delete(dead)
    assert ix.vacuum_repair() == orc.vacuum_repair()
    gg = ix.export_graph()
    graphs_equal(orc.export(), gg)
    marked = set(np.nonzero(gg.ntids == 0)[0].tolist())
    q = rows.fresh(40)
    y = rows.fresh(80)
    ty = rows.tids(y)
    ix.close()
    for how in ("graph", "pages"):
        imp = oracle.Index.from_graph(orc.export())
        ix2 = pkg.HnswIndex(dim, "vector_cosine_ops", m, efc, capacity=600, seed=0)
        if how == "graph":
            ix2.load_graph(gg)
        else:
            ix2.load_pgvector_pages(write_pages(gg, m, efc, dim, deleted=marked))
        ix2.set_option("build_batch", 1)
        ix2.set_option("vacuum_batch", 1)
        assert ix2.entry == imp.entry
        same_everything(imp, ix2, q, marked, True, set(dead.tolist()), how)
        assert ix2.insert(y, ty) == 80
        for i in range(80):
            imp.insert(y[i], int(ty[i]))
        same_everything(imp, ix2, q, marked, False, set(dead.tolist()), how + " + inserts")
        ix2.close()

