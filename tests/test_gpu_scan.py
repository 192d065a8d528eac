"""Parity of the CUDA scan path with the CPU oracle, through the C ABI, on oracle-built graphs.

Bar: neighbour ids AND distances bit-identical to the oracle in canonical summation order (the
oracle restates the kernels' fp32 order, oracle/hnsw_oracle.c canon_*); against pgvector's natural
scalar-loop order the ids agree except where distances tie within 1e-5 relative (north_star)."""
import numpy as np
import pytest

from conftest import clustered, sift_like

pytestmark = pytest.mark.gpu

OPC = {(0, 0): "vector_l2_ops", (1, 0): "vector_ip_ops", (2, 0): "vector_cosine_ops",
       (0, 1): "halfvec_l2_ops", (1, 1): "halfvec_ip_ops", (2, 1): "halfvec_cosine_ops"}


def make(oracle, pkg, x, metric, dtype=0, m=16, efc=64, seed=1):
    orc = oracle.Index(x.shape[1], m, efc, metric, dtype, oracle.CANON, seed=seed)
    orc.build(x)
    ix = pkg.HnswIndex(x.shape[1], OPC[(metric, dtype)], m, efc, capacity=max(orc.n, 1), seed=seed)
    ix.load_graph(orc.export())
    return orc, ix


@pytest.mark.parametrize("dim", [3, 8, 100, 128, 130, 768, 1100])
@pytest.mark.parametrize("metric", [0, 1, 2])
def test_distance_kernel_bit_exact(oracle, pkg, dim, metric):
    """rows a1-a3: query-vs-candidate-list distances (opclass FUNCTION 1)."""
    x = clustered(300, dim, 8, seed=dim)
    q = clustered(9, dim, 8, seed=dim + 1)
    ix = pkg.HnswIndex(dim, OPC[(metric, 0)], 8, 32, capacity=300)
    orc = oracle.Index(dim, 8, 32, metric)
    orc.build(x[:1])      # only to get normalisation semantics; distances use stored rows below
    xs = x
    if metric == oracle.COSINE:
        xs = np.stack([oracle.normalize(r)[0] for r in x])
    g = oracle.Graph(dim=dim, m=8, efc=32, metric=metric, dtype=0, n=300, upper_rows=0, entry=0, vecs=xs,
                     level=np.zeros(300, np.uint8), nbr0=np.full((300, 16), -1, np.int32), uoff=np.full(300, -1, np.int32),
                     nbru=np.full((1, 8), -1, np.int32), ntids=np.ones(300, np.uint8), tids=np.zeros((300, 10), np.int64))
    ix.load_graph(g)
    rng = np.random.default_rng(0)
    cand = rng.integers(0, 300, (9, 45)).astype(np.int32)
    cand[0, 3] = -1
    got = ix.distance(q, cand)
    for i in range(9):
        qi = oracle.normalize(q[i])[0] if metric == oracle.COSINE else q[i]
        for j in range(45):
            if cand[i, j] < 0:
                assert np.isinf(got[i, j])
                continue
            want = oracle.distance(qi, xs[cand[i, j]], oracle.L2 if metric == 0 else oracle.IP, 0, oracle.CANON)
            assert got[i, j] == np.float32(want), (i, j, got[i, j], want)
            nat = oracle.distance(qi, xs[cand[i, j]], oracle.L2 if metric == 0 else oracle.IP, 0, oracle.NATURAL)
            # 1e-5 relative to the magnitude of the summed terms (an inner product can cancel)
            a64, b64 = qi.astype(np.float64), xs[cand[i, j]].astype(np.float64)
            scale = ((a64 - b64) ** 2).sum() if metric == 0 else np.abs(a64 * b64).sum()
            assert abs(got[i, j] - nat) <= 1e-5 * scale
    ix.close()


@pytest.mark.parametrize("dim", [8, 64, 1536])
def test_halfvec_distance_bit_exact(oracle, pkg, dim):
    """row a4: halfvec storage, fp32 accumulate."""
    x = clustered(200, dim, 8, seed=dim, dtype=np.float16)
    q = clustered(5, dim, 8, seed=dim + 1, dtype=np.float16)
    for metric in (0, 1):
        ix = pkg.HnswIndex(dim, OPC[(metric, 1)], 8, 32, capacity=200)
        g = oracle.Graph(dim=dim, m=8, efc=32, metric=metric, dtype=1, n=200, upper_rows=0, entry=0, vecs=x,
                         level=np.zeros(200, np.uint8), nbr0=np.full((200, 16), -1, np.int32), uoff=np.full(200, -1, np.int32),
                         nbru=np.full((1, 8), -1, np.int32), ntids=np.ones(200, np.uint8), tids=np.zeros((200, 10), np.int64))
        ix.load_graph(g)
        cand = np.random.default_rng(1).integers(0, 200, (5, 33)).astype(np.int32)
        got = ix.distance(q, cand)
        for i in range(5):
            for j in range(33):
                want = oracle.distance(q[i], x[cand[i, j]], metric, oracle.F16, oracle.CANON)
                assert got[i, j] == np.float32(want)
        ix.close()


@pytest.mark.parametrize("dtype", [0, 1])
def test_normalize_bit_exact(oracle, pkg, dtype):
    dim = 200
    x = clustered(64, dim, 4, seed=3, dtype=np.float16 if dtype else np.float32)
    x[5] = 0
    ix = pkg.HnswIndex(dim, OPC[(2, dtype)], 8, 32, capacity=8)
    out, ok = ix.normalize(x)
    for i in range(64):
        w, wok = oracle.normalize(x[i], dtype, oracle.CANON)
        assert ok[i] == wok
        assert (out[i].view(np.uint16 if dtype else np.uint32) == w.view(np.uint16 if dtype else np.uint32)).all()
    ix.close()


def check_scan(oracle, orc, ix, q, ef, natural_check=True):
    ix.set_option("per_query_counters", 1)
    ix.counters(reset=True)
    elem, dist, cnt = ix.search_elements(q, ef)
    oe, od, oc, octr = orc.search_batch(q, ef, threads=4)
    assert (cnt == oc).all()
    assert (elem == oe).all(), "ids differ in %d of %d queries" % ((elem != oe).any(axis=1).sum(), len(q))
    assert (dist.view(np.uint32) == od.view(np.uint32)).all()
    c = ix.counters()
    assert c["n_dist"] == octr["n_dist"] and c["n_hop0"] == octr["n_hop0"] and c["n_hopu"] == octr["n_hopu"]
    if natural_check:
        # against pgvector's natural summation order: identical ids except within-tolerance ties
        orc.set_mode(oracle.NATURAL)
        ne, nd, _, _ = orc.search_batch(q, ef, threads=4)
        orc.set_mode(oracle.CANON)
        k = min(10, ef)
        for i in range(len(q)):
            if (ne[i, :k] == elem[i, :k]).all():
                continue
            # every mismatch must be explained by a tie within 1e-5 relative
            a, b = set(ne[i, :k]), set(elem[i, :k])
            dmap = dict(zip(elem[i], dist[i]))
            dmap.update(dict(zip(ne[i], nd[i])))
            edge = max(dist[i, k - 1], nd[i, k - 1])
            for e in a ^ b:
                assert abs(dmap[e] - edge) <= 1e-5 * max(abs(edge), 1e-3), (i, e, dmap[e], edge)
            for j in range(k):
                if ne[i, j] != elem[i, j]:
                    assert abs(nd[i, j] - dist[i, j]) <= 1e-5 * max(abs(dist[i, j]), 1e-3)
    return c


@pytest.mark.parametrize("ef", [1, 10, 40, 100])
def test_scan_l2_sift_like_ties(oracle, pkg, ef):
    """C1-shaped: integer-valued 128-d vectors, L2, exact distance ties are frequent."""
    x = sift_like(6000, 128, seed=1)
    q = sift_like(300, 128, seed=2)
    orc, ix = make(oracle, pkg, x, oracle.L2)
    check_scan(oracle, orc, ix, q, ef)
    ix.close()


def test_scan_cosine_768(oracle, pkg):
    """C2-shaped: 768-d cosine."""
    x = clustered(2500, 768, 64, seed=5)
    q = clustered(200, 768, 64, seed=6)
    orc, ix = make(oracle, pkg, x, oracle.COSINE)
    for ef in (40, 200):
        check_scan(oracle, orc, ix, q, ef)
    ix.close()


def test_scan_halfvec_ip_1536(oracle, pkg):
    """C4-shaped: 1536-d halfvec inner product."""
    x = clustered(1500, 1536, 32, seed=7, dtype=np.float16)
    q = clustered(100, 1536, 32, seed=8, dtype=np.float16)
    orc, ix = make(oracle, pkg, x, oracle.IP, dtype=1)
    check_scan(oracle, orc, ix, q, 40, natural_check=False)
    ix.close()


@pytest.mark.parametrize("dim,m", [(5, 4), (37, 8), (200, 24), (1030, 16), (48, 40)])
def test_scan_odd_shapes(oracle, pkg, dim, m):
    """generic row lengths (padding, run-time chunk loop) and degrees beyond one warp (2m > 32)."""
    x = clustered(2000, dim, 16, seed=dim)
    q = clustered(100, dim, 16, seed=dim + 1)
    for metric in (0, 1):
        orc, ix = make(oracle, pkg, x, metric, m=m, efc=max(2 * m, 32))
        check_scan(oracle, orc, ix, q, 30, natural_check=False)
        ix.close()


def test_scan_edge_cases(oracle, pkg):
    """empty index, one element, fewer elements than ef, k beyond the result count."""
    ix = pkg.HnswIndex(16, "vector_l2_ops", 8, 32, capacity=64)
    q = clustered(4, 16, 2, seed=1)
    elem, dist, cnt = ix.search_elements(q, 10)
    assert (cnt == 0).all() and (elem == -1).all() and np.isinf(dist).all()
    t, d, c = ix.search(q, 5, 10)
    assert (c == 0).all() and (t == -1).all()
    x = clustered(7, 16, 2, seed=2)
    for n in (1, 7):
        orc = oracle.Index(16, 8, 32, oracle.L2)
        orc.build(x[:n])
        ix.load_graph(orc.export())
        elem, dist, cnt = ix.search_elements(q, 10)
        oe, od, oc, _ = orc.search_batch(q, 10)
        assert (cnt == n).all() and (elem == oe).all() and (dist == od).all()
    ix.close()


@pytest.mark.parametrize("slots", [64, 256])
def test_visited_overflow_table(oracle, pkg, slots):
    """a shared-memory visited table too small for the query spills into the per-warp overflow table
    in HBM (and, past that, to the bitmap path); results unchanged."""
    x = sift_like(5000, 32, seed=3)
    q = sift_like(200, 32, seed=4)
    orc, ix = make(oracle, pkg, x, oracle.L2)
    ix.set_option("slots", slots)
    check_scan(oracle, orc, ix, q, 100, natural_check=False)
    ix.close()


def test_many_exact_ties(oracle, pkg):
    """very low-entropy data: long runs of equal distances at the ef boundary (tail overflow ->
    large-list path)."""
    rng = np.random.default_rng(5)
    x = rng.integers(0, 2, (3000, 8)).astype(np.float32)
    q = rng.integers(0, 2, (100, 8)).astype(np.float32)
    orc, ix = make(oracle, pkg, x, oracle.L2, m=8, efc=32)
    c = check_scan(oracle, orc, ix, q, 20, natural_check=False)
    ix.close()


def test_tie_tail_overflow_uses_long_list_path(oracle, pkg):
    """all points of the {0,1}^12 lattice: dozens of distinct elements tie exactly at the ef boundary;
    with ef=64 more than 16 of them are pushed past position ef (21 in a host emulation), which the
    shared-memory tie tail cannot hold, so those queries re-run on the long-list / bitmap path."""
    rng = np.random.default_rng(6)
    x = np.array([[(i >> b) & 1 for b in range(12)] for i in range(4096)], np.float32)[rng.permutation(4096)]
    q = x[rng.integers(0, 4096, 60)]
    orc, ix = make(oracle, pkg, x, oracle.L2, m=8, efc=32)
    c = check_scan(oracle, orc, ix, q, 64, natural_check=False)
    assert c["n_slow"] > 0
    ix.close()


def test_search_layer_parity(oracle, pkg):
    """row a5 on its own: one HnswSearchLayer call from explicit entry points, upper and base layers."""
    x = clustered(4000, 24, 16, seed=9)
    q = clustered(64, 24, 16, seed=10)
    orc, ix = make(oracle, pkg, x, oracle.L2, m=8, efc=32, seed=4)
    ent, lvl = orc.entry
    assert lvl >= 2
    g = orc.export()
    lvl1 = np.nonzero(g.level >= 1)[0]
    for layer, ef, eps in ((lvl, 1, np.full((64, 1), ent)), (1, 1, np.tile(lvl1[:1], (64, 1))),
                           (1, 8, np.tile(lvl1[:5], (64, 1))), (0, 16, np.tile(np.arange(7), (64, 1)))):
        elem, dist, cnt = ix.search_layer(q, eps.astype(np.int32), ef, layer)
        for i in range(64):
            oe, od, _ = orc.search_layer(q[i], eps[i].astype(np.int32), ef, layer)
            assert cnt[i] == len(oe)
            assert (elem[i, :cnt[i]] == oe).all() and (dist[i, :cnt[i]] == od).all()
    ix.close()


def test_gettuple_streams_like_hnswgettuple(oracle, pkg):
    """rows a6/a11: amrescan + amgettuple order, duplicate heap TIDs, exhaustion."""
    x = clustered(500, 16, 4, seed=11)
    orc = oracle.Index(16, 8, 32, oracle.L2)
    orc.build(x)
    for j in range(3):
        orc.insert(x[10], 1000 + j)           # duplicates of row 10 share its element
    ix = pkg.HnswIndex(16, "vector_l2_ops", 8, 32, capacity=600)
    ix.load_graph(orc.export())
    scan = ix.beginscan()
    with pytest.raises(pkg.HnswError):
        scan.gettuple()                        # "cannot scan hnsw index without order"
    for qi in (10, 77):
        scan.rescan(x[qi], 25)
        got = []
        while True:
            t = scan.gettuple()
            if t is None:
                break
            got.append(t)
        wt, wd = orc.search_tids(x[qi], 25, 1000)
        assert [g[0] for g in got] == list(wt)
        assert [np.float32(g[1]) for g in got] == list(wd)
    assert scan.gettuple() is None
    # batched form agrees with the stream
    t, d, c = ix.search(x[[10, 77]], 6, 25)
    wt, wd = orc.search_tids(x[10], 25, 6)
    assert list(t[0]) == list(wt)
    scan.endscan()
    with pytest.raises(pkg.HnswError):
        ix.search(np.zeros((1, 15), np.float32))     # expected 16 dimensions, not 15
    ix.close()


def test_merge_topk(pkg):
    import torch
    rng = np.random.default_rng(0)
    P, nq, k = 5, 300, 10
    d = np.sort(rng.random((P, nq, k)).astype(np.float32), axis=2)
    t = rng.integers(0, 1 << 40, (P, nq, k)).astype(np.int64)
    d[2, :, 7:] = np.inf
    t[2, :, 7:] = -1
    dt, dd = torch.tensor(t).cuda(), torch.tensor(d).cuda()
    ot = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    od = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    pkg.merge_topk_dev(0, dt.data_ptr(), dd.data_ptr(), P, nq, k, ot.data_ptr(), od.data_ptr(),
                       torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for i in range(nq):
        allp = sorted((d[p, i, j], p, t[p, i, j]) for p in range(P) for j in range(k) if t[p, i, j] >= 0)[:k]
        assert [a[2] for a in allp] == ot[i].tolist()


def test_c1_config_on_gpu_built_graph(oracle, pkg):
    """configs[0] (the reference's own CPU-runnable case): 100k x 128 SIFT-shaped L2, m=16,
    ef_construction=64, ef_search=40, k=10, one partition.  The graph is built on the GPU (the
    single-threaded oracle build of 100k rows takes minutes); the oracle then searches that same graph
    on the CPU and must return the same ids, distances and counters."""
    n, nq = 100000, 1000
    x = sift_like(n, 128, seed=21)
    q = sift_like(nq, 128, seed=22)
    ix = pkg.HnswIndex(128, "vector_l2_ops", 16, 64, capacity=n, seed=3)
    assert ix.build(x) == n
    orc = oracle.Index.from_graph(ix.export_graph())
    check_scan(oracle, orc, ix, q, 40)
    gt, _ = ix.bruteforce(q, 10)
    elem, _, _ = ix.search_elements(q, 40)
    rec = np.mean([len(set(elem[i, :10]) & set(gt[i])) / 10 for i in range(nq)])
    assert rec >= 0.9, rec
    ix.close()


@pytest.mark.parametrize("dim,dtype,m,ef", [(2000, 0, 8, 20), (4000, 1, 8, 20), (16, 0, 100, 300), (32, 0, 16, 1000), (64, 1, 16, 500)])
def test_limits(oracle, pkg, dim, dtype, m, ef):
    """pgvector's limits: 2000 dims (vector) / 4000 (halfvec) in hnsw, m = 100, ef_search = 1000."""
    dt = np.float16 if dtype else np.float32
    x = clustered(1200, dim, 8, seed=dim, dtype=dt)
    q = clustered(40, dim, 8, seed=dim + 1, dtype=dt)
    orc, ix = make(oracle, pkg, x, oracle.L2, dtype=dtype, m=m, efc=max(2 * m, 32))
    check_scan(oracle, orc, ix, q, ef, natural_check=False)
    ix.close()
    with pytest.raises(pkg.HnswError):
        ix2 = pkg.HnswIndex(8, "vector_l2_ops", 8, 32, capacity=10)
        ix2.search(np.zeros((1, 8), np.float32), 5, 1001)       # hnsw.ef_search is capped at 1000


# ---- the register-list scan kernel (csrc/scan_reg.cuh): rows of 32 or 64 chunks --------------------
@pytest.mark.parametrize("dim,dtype,metric,m,ef", [
    (128, 0, 0, 16, 48), (128, 0, 0, 16, 49), (128, 0, 1, 16, 104), (128, 0, 2, 16, 105), (128, 0, 0, 24, 40),
    (256, 0, 0, 16, 40), (256, 0, 2, 12, 90), (256, 1, 0, 16, 40), (512, 1, 1, 16, 64), (256, 1, 2, 16, 30)])
def test_register_list_scan(oracle, pkg, dim, dtype, metric, m, ef):
    """ef at the edges of the 64- and 128-entry register lists (48|49, 104|105), degrees beyond one warp (m = 24),
    fp32 and halfvec rows, all metrics; integer-valued data so that exact ties sit at the ef boundary.  The
    forced shared-memory-list kernel (variant 9) must agree as well."""
    dt = np.float16 if dtype else np.float32
    x = sift_like(5000, dim, seed=dim + ef).astype(dt)
    q = sift_like(200, dim, seed=dim + ef + 1).astype(dt)
    orc, ix = make(oracle, pkg, x, metric, dtype=dtype, m=m, efc=max(2 * m, 64))
    check_scan(oracle, orc, ix, q, ef, natural_check=False)
    e1, d1, c1 = ix.search_elements(q, ef)
    ix.set_option("variant", 9)
    e2, d2, c2 = ix.search_elements(q, ef)
    assert (e1 == e2).all() and (d1.view(np.uint32) == d2.view(np.uint32)).all() and (c1 == c2).all()
    ix.close()


def test_register_list_scan_l1(oracle, pkg):
    x = sift_like(4000, 128, seed=3)
    q = sift_like(150, 128, seed=4)
    orc = oracle.Index(128, 16, 64, oracle.L1, 0, oracle.CANON, seed=2)
    orc.build(x)
    ix = pkg.HnswIndex(128, "vector_l1_ops", 16, 64, capacity=4000, seed=2)
    ix.load_graph(orc.export())
    check_scan(oracle, orc, ix, q, 40, natural_check=False)
    ix.close()


def test_register_list_tail_and_table_overflow(oracle, pkg):
    """128-d rows whose distances tie massively (lattice points padded with zeros): the tie tail outgrows the
    64 register slots -> those queries re-run on the long-list path; a tiny visited table spills to HBM."""
    rng = np.random.default_rng(6)
    lat = np.array([[(i >> b) & 1 for b in range(12)] for i in range(4096)], np.float32)[rng.permutation(4096)]
    x = np.zeros((4096, 128), np.float32)
    x[:, :12] = lat
    q = x[rng.integers(0, 4096, 60)]
    orc, ix = make(oracle, pkg, x, oracle.L2, m=8, efc=32)
    c = check_scan(oracle, orc, ix, q, 48, natural_check=False)         # 48 + 16 = 64 slots: room for 16 ties only
    assert c["n_slow"] > 0
    ix.set_option("slots", 64)
    check_scan(oracle, orc, ix, q, 30, natural_check=False)
    ix.close()


# ---- the CTA-per-query kernel (csrc/scan_cta.cuh): batches of at most one query per SM ---------------
@pytest.mark.parametrize("dim,dtype,metric,m,ef", [
    (128, 0, 0, 16, 40), (96, 0, 2, 16, 64), (768, 0, 2, 16, 90), (256, 1, 1, 12, 200), (48, 1, 0, 8, 30), (384, 0, 0, 24, 100)])
def test_cta_per_query_scan(oracle, pkg, dim, dtype, metric, m, ef):
    """Small batches of long rows take the four-warps-per-query kernels on their own (>= 1536-byte rows); variant 7
    forces them for every shape (register list + look-ahead row staging when ef <= 104, shared-memory list above), 17
    forces the shared-memory list, 27 the register list without row staging, 6 forbids the CTA kernels.  All must
    equal the oracle bit for bit, counters included."""
    dt = np.float16 if dtype else np.float32
    x = sift_like(5000, dim, seed=dim + ef + 7).astype(dt)
    q = sift_like(100, dim, seed=dim + ef + 8).astype(dt)
    orc, ix = make(oracle, pkg, x, metric, dtype=dtype, m=m, efc=max(2 * m, 64))
    ix.set_option("variant", 7)
    check_scan(oracle, orc, ix, q, ef, natural_check=False)
    e1, d1, c1 = ix.search_elements(q, ef)
    e3, d3, c3 = ix.search_elements(q[:1], ef)                     # a single scan
    assert (e3[0] == e1[0]).all() and c3[0] == c1[0]
    for v in (17, 27, 6):
        ix.set_option("variant", v)
        e2, d2, c2 = ix.search_elements(q, ef)
        assert (e1 == e2).all() and (d1.view(np.uint32) == d2.view(np.uint32)).all() and (c1 == c2).all(), v
    ix.close()


def test_cta_per_query_tie_tail(oracle, pkg):
    """Massive exact ties (see test_register_list_tail_and_table_overflow) under the forced CTA-per-query kernel:
    queries whose tie tail outgrows the list re-run on the long-list path and still match the oracle."""
    rng = np.random.default_rng(9)
    lat = np.array([[(i >> b) & 1 for b in range(12)] for i in range(4096)], np.float32)[rng.permutation(4096)]
    x = np.zeros((4096, 128), np.float32)
    x[:, :12] = lat
    q = x[rng.integers(0, 4096, 60)]
    orc, ix = make(oracle, pkg, x, oracle.L2, m=8, efc=32)
    for v in (7, 17, 27):
        ix.set_option("variant", v)
        check_scan(oracle, orc, ix, q, 48, natural_check=False)
        check_scan(oracle, orc, ix, q, 10, natural_check=False)
    ix.close()


def test_scan_variant_values(pkg):
    """The variant option takes only the values that force a production scan path; the removed tuning variants and
    the unfused neighbour selection are refused instead of silently ignored."""
    ix = pkg.HnswIndex(128, "vector_l2_ops", 16, 64, capacity=10)
    for v in (1, 2, 3, 4, 5, 8, 10, 20):
        with pytest.raises(pkg.HnswError):
            ix.set_option("variant", v)
    for v in (0, 6, 7, 9, 17, 27):
        ix.set_option("variant", v)
    with pytest.raises(pkg.HnswError):
        ix.set_option("fused_select", 0)
    ix.close()
