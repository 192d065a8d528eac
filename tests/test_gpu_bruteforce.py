"""Exact per-partition scan (config 5): bf16 tcgen05 GEMM candidate generation + fp32 re-rank,
against numpy (raw scores), the oracle's double-precision brute force, and bit for bit against the oracle's
exhaustive top-k of the canonical fp32 distance (the exact scan's contract), whether a query was certified or
re-scanned."""
import math
import os

import numpy as np
import pytest

from conftest import clustered, sift_like
from exact import flat_graph

pytestmark = pytest.mark.gpu


def bf16_round(a):
    """round-to-nearest-even fp32 -> bf16 -> fp32 in numpy"""
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


@pytest.mark.parametrize("n,dim,nq", [(1000, 64, 37), (3000, 128, 300), (2500, 768, 130), (700, 100, 129),
                                     (257, 1, 5), (513, 65, 128), (300, 2000, 129)])
def test_gemm_scores_match_bf16_reference(pkg, n, dim, nq):
    """the tensor-core stage on its own: S = bf16(Q) . bf16(X)^T accumulated in fp32"""
    x = clustered(n, dim, 16, seed=n)
    q = clustered(nq, dim, 16, seed=n + 1)
    ix = pkg.HnswIndex(dim, "vector_ip_ops", 8, 32, capacity=n)
    g = type("G", (), {})()
    g.dim, g.m, g.efc, g.n, g.upper_rows, g.entry = dim, 8, 32, n, 0, 0
    g.vecs, g.level, g.nbr0 = x, np.zeros(n, np.uint8), np.full((n, 16), -1, np.int32)
    g.uoff, g.nbru, g.ntids, g.tids = np.full(n, -1, np.int32), np.full((1, 8), -1, np.int32), np.ones(n, np.uint8), np.zeros((n, 10), np.int64)
    ix.load_graph(g)
    elem, dist, scores, st = ix.bruteforce(q, 10, debug_scores=True, stats=True)
    want = bf16_round(q).astype(np.float64) @ bf16_round(x).astype(np.float64).T
    scale = np.abs(bf16_round(q)).astype(np.float64) @ np.abs(bf16_round(x)).astype(np.float64).T
    # fp32 accumulation only: 2e-6 of sum |q^_i x^_i| up to 768 terms (12 K-chunks), growing with the terms above;
    # far inside the kpad 2^-23 the certificate allows for it
    kpad = -(-dim // 64) * 64
    assert np.max(np.abs(scores - want) / (scale + 1e-6)) < 2e-6 * max(1.0, kpad / 768)
    assert st["certified"] + st["rescanned"] == nq
    ix.close()


@pytest.mark.parametrize("metric,opclass,dtype", [(0, "vector_l2_ops", 0), (1, "vector_ip_ops", 0), (2, "vector_cosine_ops", 0),
                                                   (1, "halfvec_ip_ops", 1), (0, "halfvec_l2_ops", 1),
                                                   (2, "halfvec_cosine_ops", 1)])
def test_exact_topk_matches_oracle(oracle, pkg, metric, opclass, dtype):
    n, dim, nq, k = 6000, 96, 400, 10
    dt = np.float16 if dtype else np.float32
    x = clustered(n, dim, 32, seed=3, dtype=dt)
    q = clustered(nq, dim, 32, seed=4, dtype=dt)
    orc = oracle.Index(dim, 8, 32, metric, dtype)
    orc.build(x[:50])                                   # any small graph: only the vectors matter below
    g = orc.export()
    xs = x if metric != 2 else np.stack([oracle.normalize(r, dtype)[0] for r in x])
    g.n, g.vecs = n, xs
    g.level, g.nbr0 = np.zeros(n, np.uint8), np.full((n, 16), -1, np.int32)
    g.uoff, g.nbru, g.upper_rows, g.entry = np.full(n, -1, np.int32), np.full((1, 8), -1, np.int32), 0, 0
    g.ntids, g.tids = np.ones(n, np.uint8), np.zeros((n, 10), np.int64)
    ix = pkg.HnswIndex(dim, opclass, 8, 32, capacity=n)
    ix.load_graph(g)
    full = oracle.Index.from_graph(g)
    gt, gd = full.bruteforce(q, k, threads=8)
    elem, dist, st = ix.bruteforce(q, k, stats=True)
    assert st["certified"] + st["rescanned"] == nq
    for i in range(nq):
        if list(elem[i]) == list(gt[i]):
            continue
        # any difference must be an fp32-vs-double near tie
        for j in range(k):
            assert abs(dist[i, j] - gd[i, j]) <= 1e-5 * max(abs(gd[i, j]), 1e-3), (i, j, elem[i], gt[i])
    same = np.mean([list(elem[i]) == list(gt[i]) for i in range(nq)])
    assert same > 0.98
    # and bit for bit the canonical fp32 top-k
    st = check_exact(oracle, ix, q, k)
    assert st["certified"] > nq // 2
    ix.close()


def test_uncertifiable_queries_are_rescanned(oracle, pkg):
    """nearly uniform data: bf16 cannot separate the candidates, the certificate fails and the fp32
    exhaustive path takes over; results stay exact."""
    rng = np.random.default_rng(0)
    n, dim, nq, k = 3000, 64, 20, 10
    x = (1.0 + 1e-3 * rng.standard_normal((n, dim))).astype(np.float32)
    q = (1.0 + 1e-3 * rng.standard_normal((nq, dim))).astype(np.float32)
    g = type("G", (), {})()
    g.dim, g.m, g.efc, g.metric, g.dtype, g.n, g.upper_rows, g.entry = dim, 8, 32, 1, 0, n, 0, 0
    g.vecs, g.level, g.nbr0 = x, np.zeros(n, np.uint8), np.full((n, 16), -1, np.int32)
    g.uoff, g.nbru, g.ntids, g.tids = np.full(n, -1, np.int32), np.full((1, 8), -1, np.int32), np.ones(n, np.uint8), np.zeros((n, 10), np.int64)
    ix = pkg.HnswIndex(dim, "vector_ip_ops", 8, 32, capacity=n)
    ix.load_graph(g)
    elem, dist, st = ix.bruteforce(q, k, stats=True)
    assert st["rescanned"] > 0
    full = oracle.Index.from_graph(g)
    for i in range(nq):
        want = sorted((oracle.distance(q[i], x[e], oracle.IP), e) for e in range(n))[:k]
        assert [e for _, e in want] == list(elem[i])
    ix.close()


# ---- bit for bit against the oracle's exhaustive canonical fp32 top-k ---------------------------------------------

OPS = {"vector_l2_ops": (0, 0), "vector_ip_ops": (1, 0), "vector_cosine_ops": (2, 0),
       "halfvec_l2_ops": (0, 1), "halfvec_ip_ops": (1, 1), "halfvec_cosine_ops": (2, 1)}


def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def decomposition(nq, n, grid_opt=0):
    """the host's work split of hb_bruteforce_ex: query tiles of 128 x slices of S runs of 256-row tiles, one work
    item per (query tile, slice), items run by min(items, SMs, grid option) persistent CTAs"""
    sms = num_sms()
    n_mtiles, ntiles = -(-nq // 128), -(-n // 256)
    best_s, best_eff = 1, -1.0
    for s in range(1, min(16, ntiles) + 1):
        items = n_mtiles * s
        eff = items / (-(-items // sms) * sms)
        if eff > best_eff + 1e-9 or (abs(eff - best_eff) <= 1e-9 and s > best_s and s <= 8):
            best_eff, best_s = eff, s
    tps = -(-ntiles // best_s)
    s = -(-ntiles // tps)
    items = n_mtiles * s
    grid = min(items, sms, grid_opt) if grid_opt > 0 else min(items, sms)
    return {"n_mtiles": n_mtiles, "ntiles": ntiles, "S": s, "tiles_per_split": tps, "items": items, "grid": grid,
            "candidates": 2 * s * 16}


def rows(opclass, x, oracle):
    metric, dtype = OPS[opclass]
    x = np.ascontiguousarray(x, np.float16 if dtype else np.float32)
    if metric == 2:
        x = np.stack([oracle.normalize(r, dtype)[0] for r in x])
    return x


def flat_index(pkg, oracle, opclass, x):
    metric, dtype = OPS[opclass]
    x = rows(opclass, x, oracle)
    ix = pkg.HnswIndex(x.shape[1], opclass, 8, 32, capacity=max(len(x), 1))
    ix.load_graph(flat_graph(x, metric, dtype))
    return ix


def check_exact(oracle, ix, q, k):
    """the exact scan's answer equals the oracle's canonical top-k of the index's own (exported) rows, ids and
    distance bits; returns the certified / rescanned counts"""
    ref = oracle.Index.from_graph(ix.export_graph())
    want_e, want_d = ref.exact_topk(q, k, threads=os.cpu_count() or 8)
    elem, dist, st = ix.bruteforce(q, k, stats=True)
    assert st["certified"] + st["rescanned"] == len(q)
    bad = np.nonzero((elem != want_e).any(axis=1) | (dist.view(np.uint32) != want_d.view(np.uint32)).any(axis=1))[0]
    assert bad.size == 0, ("%d of %d queries differ, first %d: got %s %s want %s %s" %
                           (bad.size, len(q), bad[0], elem[bad[0]], dist[bad[0]], want_e[bad[0]], want_d[bad[0]]))
    return st


@pytest.mark.parametrize("opclass", ["vector_l2_ops", "vector_ip_ops", "vector_cosine_ops"])
def test_several_work_items_per_cta(oracle, pkg, opclass):
    """tiles_per_split odd and CTAs capped below the item count: every CTA carries the TMA ring, the accumulator
    phase, the L2 norm buffers and the threshold seeds from one item to the next; any cap gives the same answer"""
    n, dim, nq, k = 39 * 256 - 17, 128, 300, 10
    x = clustered(n, dim, 32, seed=21)
    q = rows(opclass, clustered(nq, dim, 32, seed=22), oracle)
    ix = flat_index(pkg, oracle, opclass, x)
    first = None
    for grid in (1, 3, 7, 0):
        dec = decomposition(nq, n, grid)
        assert dec["tiles_per_split"] % 2 == 1
        if grid:
            assert dec["items"] > dec["grid"] == grid
        ix.set_option("grid", grid)
        st = check_exact(oracle, ix, q, k)
        assert st["certified"] > nq // 2
        out = ix.bruteforce(q, k)
        if first is None:
            first = out
        assert np.array_equal(out[0], first[0]) and np.array_equal(out[1].view(np.uint32), first[1].view(np.uint32))
    ix.close()


@pytest.mark.parametrize("opclass,gen", [("vector_l2_ops", "sift"), ("vector_cosine_ops", "clustered")])
def test_recall_ground_truth_shape(oracle, pkg, opclass, gen):
    """10 000 queries: the shape the recall tests use as ground truth, with several items per CTA uncapped"""
    n, dim, nq, k = 9967, 128, 10000, 10
    dec = decomposition(nq, n)
    assert dec["items"] > dec["grid"]
    assert dec["tiles_per_split"] % 2 == 1
    mk = (lambda m, s: sift_like(m, dim, seed=s)) if gen == "sift" else (lambda m, s: clustered(m, dim, 32, seed=s))
    ix = flat_index(pkg, oracle, opclass, mk(n, 31))
    st = check_exact(oracle, ix, rows(opclass, mk(nq, 32), oracle), k)
    assert st["certified"] > 0
    ix.close()


RAGGED = ([("n", v, 129, 65) for v in (1, 5, 16, 17, 255, 256, 257, 511, 513)] +
          [("nq", 513, v, 100) for v in (1, 127, 128, 129)] +
          [("dim", 257, 128, v) for v in (1, 63, 64, 65, 100, 2000)])


@pytest.mark.parametrize("what,n,nq,dim", RAGGED)
def test_ragged_shapes(oracle, pkg, what, n, nq, dim):
    """rows around the 256-row tiles and 128-column halves, queries around the 128-row tiles, dims around the
    64-wide K-chunks up to the vector maximum; the metric rotates with the case"""
    opclass = ("vector_l2_ops", "vector_ip_ops", "vector_cosine_ops")[(n + nq + dim) % 3]
    if dim == 1 and opclass == "vector_cosine_ops":
        opclass = "vector_l2_ops"                      # a 1-d unit vector is +-1: nothing to rank
    ix = flat_index(pkg, oracle, opclass, clustered(n, dim, 8, seed=n + dim))
    q = rows(opclass, clustered(nq, dim, 8, seed=n + dim + 1), oracle)
    check_exact(oracle, ix, q, 10)
    ix.close()


@pytest.mark.parametrize("opclass", ["halfvec_l2_ops", "halfvec_ip_ops", "halfvec_cosine_ops"])
def test_halfvec_max_dim(oracle, pkg, opclass):
    """4000 dimensions (the halfvec maximum): 63 K-chunks"""
    n, dim, nq = 300, 4000, 129
    ix = flat_index(pkg, oracle, opclass, clustered(n, dim, 8, seed=41, dtype=np.float16))
    q = rows(opclass, clustered(nq, dim, 8, seed=42, dtype=np.float16), oracle)
    check_exact(oracle, ix, q, 10)
    ix.close()


@pytest.mark.parametrize("k", [1, 10, 16, 17, 32, 33, 100, 128])
def test_k(oracle, pkg, k):
    n, dim, nq = 5000, 64, 129
    ix = flat_index(pkg, oracle, "vector_l2_ops", clustered(n, dim, 16, seed=51))
    q = clustered(nq, dim, 16, seed=52)
    st = check_exact(oracle, ix, q, k)
    if k > decomposition(nq, n)["candidates"]:
        assert st["rescanned"] == nq
    ix.close()


@pytest.mark.parametrize("n,k", [(5, 10), (16, 128), (40, 100), (256, 33), (256, 128), (700, 128)])
def test_k_beyond_rows_or_candidates(oracle, pkg, n, k):
    """k > n pads with -1 / +inf; k above the 2 * S * 16 candidates the GEMM keeps cannot be certified and goes
    through the fp32 re-scan"""
    dim, nq = 48, 3
    ix = flat_index(pkg, oracle, "vector_ip_ops", clustered(n, dim, 4, seed=n))
    q = clustered(nq, dim, 4, seed=n + 1)
    st = check_exact(oracle, ix, q, k)
    dec = decomposition(nq, n)
    if n < 16:
        assert st["certified"] == nq                   # no slice filled its list: every row is a candidate
    elif n > k > dec["candidates"]:
        assert st["rescanned"] == nq
    ix.close()


@pytest.mark.parametrize("opclass", ["vector_l2_ops", "vector_ip_ops"])
def test_exact_ties(oracle, pkg, opclass):
    """integer rows are exact in bf16, so GEMM scores tie exactly across slices (the strict > at the threshold, the
    seeds from other slices); byte copies of one row at ids in different slices come back in id order"""
    n, dim, nq = 7000, 128, 200
    x = sift_like(n, dim, seed=61)
    copies = [5, 300, 2100, 4000, 6999]
    x[copies] = x[1234]
    q = sift_like(nq, dim, seed=62)
    q[:20] = x[1234]
    q[20:40] = x[1234] + 1
    ix = flat_index(pkg, oracle, opclass, x)
    assert decomposition(nq, n)["S"] > 1
    check_exact(oracle, ix, q, 10)
    if opclass == "vector_l2_ops":
        e, _ = ix.bruteforce(q[:1], 10)
        assert list(e[0][:6]) == sorted(copies + [1234])
    ix.close()


@pytest.mark.parametrize("spread", [1e-7, 1e-6, 1e-5])
def test_certificate_l2_query_near_origin(oracle, pkg, spread):
    """rows on a thin shell and queries at or near the origin: the scores are -|x|^2/2 and differ from the
    re-rank's distances only by fp32 rounding of |x|^2, which the certificate has to cover"""
    rng = np.random.default_rng(71)
    n, dim = 2000, 128
    d = rng.standard_normal((n, dim))
    x = (d / np.linalg.norm(d, axis=1, keepdims=True) * (1 + spread * rng.random((n, 1)))).astype(np.float32)
    q = np.zeros((40, dim), np.float32)
    q[10:] = (1e-3 * rng.standard_normal((30, dim)) / math.sqrt(dim)).astype(np.float32)
    ix = flat_index(pkg, oracle, "vector_l2_ops", x)
    check_exact(oracle, ix, q, 10)
    ix.close()


def test_certificate_bf16_rounding_of_both_operands(oracle, pkg):
    """the bf16 copies of q and x each perturb q.x by up to 2^-8 |q||x|, together about 2^-7: a row that both
    roundings pull down (G) is dropped behind rows whose scores are exact in one operand, and a bound below 2^-7
    would certify the wrong top-1"""
    dim = 33
    a = 1 + 2.0 ** -8                                  # halfway between two bf16 values: rounds down to 1
    q = np.zeros(dim, np.float32)
    q[:32], q[32] = a, 1.0
    filler = np.zeros(dim, np.float32)
    filler[:32], filler[32] = 1.0, 2.0 ** -5           # bf16 score 32.03125, exact q.x 32.15625
    top = filler.copy()
    top[32] = 3 * 2.0 ** -5                            # bf16 score 32.09375, exact q.x 32.21875
    g = np.zeros(dim, np.float32)
    g[:32] = a                                         # bf16 score 32, exact q.x 32.2501: the true top-1
    x = np.zeros((300, dim), np.float32)
    x[:20] = filler
    x[20], x[21] = top, g
    x[22:] = 0.01 * np.random.default_rng(81).standard_normal((278, dim))
    ix = flat_index(pkg, oracle, "vector_ip_ops", x)
    qs = np.stack([q] * 4)
    check_exact(oracle, ix, qs, 1)
    e, _ = ix.bruteforce(qs, 1)
    assert (e[:, 0] == 21).all()
    ix.close()


def test_certificate_halfvec_ip_max_dim_near_ties(oracle, pkg):
    """4000-d halfvec inner product on rows one fp16 ulp apart in a few components: the GEMM's fp32 accumulation
    error over 4032 terms is as large as the gaps"""
    rng = np.random.default_rng(91)
    n, dim, nq = 600, 4000, 16
    base = rng.standard_normal(dim).astype(np.float16)
    x = np.repeat(base[None, :], n, axis=0)
    for i in range(n):
        j = rng.integers(0, dim, 4)
        x[i, j] = np.nextafter(x[i, j], np.float16(np.inf) * np.sign(rng.standard_normal(4)).astype(np.float16))
    q = (base[None, :] + 0.01 * rng.standard_normal((nq, dim))).astype(np.float16)
    ix = flat_index(pkg, oracle, "halfvec_ip_ops", x)
    st = check_exact(oracle, ix, q, 10)
    assert st["rescanned"] > 0
    ix.close()


def test_cached_image_follows_the_index(oracle, pkg):
    """the bf16 image is rebuilt after every change of the index: inserted rows are found, a different graph with
    the same n replaces the old rows, and rows emptied by bulk delete + vacuum are scanned as the exported image
    holds them"""
    n, dim, k = 3000, 64, 10
    x = clustered(n, dim, 16, seed=101)
    ix = pkg.HnswIndex(dim, "vector_l2_ops", 8, 32, capacity=2 * n)
    ix.build(x)
    q = clustered(50, dim, 16, seed=102)
    check_exact(oracle, ix, q, k)
    new = clustered(200, dim, 16, seed=103)
    ix.insert(new, np.arange(n, n + 200))
    check_exact(oracle, ix, q, k)
    e, d = ix.bruteforce(new, 1)
    assert (e[:, 0] >= n).all() and (d[:, 0] == 0).all()
    # another graph with the same number of rows
    other = flat_graph(clustered(ix.n, dim, 16, seed=104), 0, 0)
    ix.load_graph(other)
    check_exact(oracle, ix, q, k)
    check_exact(oracle, ix, other.vecs[::37], k)
    # delete half the heap TIDs and vacuum
    assert ix.bulk_delete(np.arange(0, ix.n, 2)) > 0
    ix.vacuum_repair()
    check_exact(oracle, ix, q, k)
    ix.close()
