"""The oracle's exact top-k (the reference the GPU exact scan must equal bit for bit) against a plain sort of the
canonical fp32 distance over every row, and against the double-precision brute force used for recall."""
import numpy as np
import pytest

from conftest import clustered, sift_like
from exact import flat_graph


def rows_for(oracle, gen, n, dim, metric, dtype, seed):
    dt = np.float16 if dtype else np.float32
    x = sift_like(n, dim, seed=seed).astype(dt) if gen == "sift" else clustered(n, dim, 8, seed=seed, dtype=dt)
    if metric == oracle.COSINE:
        x = np.stack([oracle.normalize(r, dtype)[0] for r in x])
    return x


CASES = [(m, dt, gen, dim) for m in (0, 1, 2) for dt in (0, 1) for gen, dim in (("clustered", 5), ("clustered", 100), ("sift", 64))]


@pytest.mark.parametrize("metric,dtype,gen,dim", CASES)
@pytest.mark.parametrize("n,k", [(1, 3), (37, 10), (300, 17), (300, 128)])
def test_exact_topk_is_the_sorted_canonical_distance(oracle, metric, dtype, gen, dim, n, k):
    x = rows_for(oracle, gen, n, dim, metric, dtype, seed=n + dim)
    # byte copies of one row at several ids: the tie must resolve by element id
    if n > 20:
        x[[3, 11, n - 1]] = x[7]
    q = rows_for(oracle, gen, 6, dim, oracle.COSINE if metric == oracle.COSINE else oracle.L2, dtype, seed=n + dim + 1)
    if n > 20:
        q[0] = x[7]
    ix = oracle.Index.from_graph(flat_graph(x, metric, dtype))
    e, d = ix.exact_topk(q, k, threads=4)
    code = oracle.L2 if metric == oracle.L2 else oracle.IP
    for i in range(len(q)):
        qi = oracle.normalize(q[i], dtype)[0] if metric == oracle.COSINE else q[i]
        want = sorted((oracle.distance(qi, x[r], code, dtype), r) for r in range(n))[:k]
        got_e = [int(v) for v in e[i]]
        assert got_e[:len(want)] == [r for _, r in want], i
        assert np.array_equal(d[i, :len(want)], np.array([w for w, _ in want], np.float32)), i
        assert (e[i, len(want):] == -1).all() and np.isinf(d[i, len(want):]).all()
    if n > 20:
        # the copies of x[7] come back in id order, right after one another
        pos = [list(e[0]).index(r) for r in (3, 7, 11) if r in e[0]]
        assert pos == sorted(pos)


@pytest.mark.parametrize("metric,dtype", [(0, 0), (1, 0), (2, 0), (0, 1), (1, 1), (2, 1)])
def test_exact_topk_agrees_with_double_bruteforce(oracle, metric, dtype):
    """ids may differ from the double-precision answer only where the double distances of the swapped rows lie within
    fp32 rounding of the k-th distance"""
    n, dim, k = 2000, 96, 10
    x = rows_for(oracle, "clustered", n, dim, metric, dtype, seed=5)
    q = rows_for(oracle, "clustered", 50, dim, metric, dtype, seed=6)
    ix = oracle.Index.from_graph(flat_graph(x, metric, dtype))
    e, d = ix.exact_topk(q, k, threads=4)
    ge, gd = ix.bruteforce(q, k, threads=4)
    xs = x.astype(np.float64)
    for i in range(len(q)):
        if list(e[i]) == list(ge[i]):
            continue
        qi = (oracle.normalize(q[i], dtype)[0] if metric == oracle.COSINE else q[i]).astype(np.float64)
        scale = np.linalg.norm(qi) * np.max(np.linalg.norm(xs, axis=1))
        if metric == oracle.L2:
            scale = scale + float(qi @ qi) + float(np.max(np.sum(xs * xs, axis=1)))
        tol = 4 * dim * 2.0 ** -24 * scale
        for r in set(e[i].tolist()) ^ set(ge[i].tolist()):
            dr = float(np.sum((qi - xs[r]) ** 2)) if metric == oracle.L2 else -float(qi @ xs[r])
            assert abs(dr - gd[i, k - 1]) <= tol, (i, r, dr, gd[i, k - 1])
        # the fp32 distances agree with the double ones to fp32 rounding
        assert np.all(np.abs(d[i].astype(np.float64) - gd[i]) <= tol)
