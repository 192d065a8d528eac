"""The partitioned search restated on the CPU oracle: what hb_part_search must return for the graphs its partitions
hold.  Test helper shared by the oracle-only tests (test_oracle_partition_ref.py) and the GPU tests of the partitioned
index (test_gpu_partition_world1.py, test_gpu_partition.py).

The answer of a query is the k smallest (distance, heap TID) pairs over every heap TID of the elements each
partition's scan returned (at most ef_search elements per partition), at that element's distance, nearest first and
padded with -1 / +inf.  It does not depend on the order a scan emits TIDs in, on how partitions are grouped into ranks,
or on the number of ranks."""
import numpy as np

from conftest import sift_like
from oracle import oracle as O


def route(tids, P):
    """splitmix64(tid) mod P: the partition of each heap TID (hb_partition_route restated in numpy)."""
    x = np.ascontiguousarray(tids, np.int64).astype(np.uint64)
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    return (x % np.uint64(P)).astype(np.int32)


def tie_rows(n, dim, seed, copies=40, dtype=np.float32):
    """Rows made for exact ties: integer-valued (SIFT-shaped), about 5 % of them byte copies of one of the first 40
    rows, and row 3 copied `copies` more times (more than HEAPTIDS copies fill several elements of one partition, and
    the copies land in several partitions).  Heap TIDs: a random permutation of sparse values, so they neither grow
    with row order nor with insertion order.  Returns (rows in random order, their TIDs)."""
    rng = np.random.default_rng(seed)
    x = sift_like(n, dim, seed=seed)
    dup = rng.choice(n - 40 - copies, n // 20, replace=False) + 40
    x[dup] = x[rng.integers(0, 40, len(dup))]
    x[n - copies:] = x[3]
    tids = np.unique(rng.integers(1 << 20, 1 << 40, 2 * n))[:n]
    return x[rng.permutation(n)].astype(dtype), rng.permutation(tids)


def expand(g, elem, dist, cnt):
    """Every heap TID of the elements one partition's scan returned: (query, distance, tid) arrays."""
    nq, ef = elem.shape
    valid = np.arange(ef)[None, :] < np.asarray(cnt)[:, None]
    qi, j = np.nonzero(valid)
    e = elem[qi, j]
    nt = g.ntids[e].astype(np.int64)
    rep = np.repeat(np.arange(len(e)), nt)
    slot = np.arange(len(rep)) - np.repeat(np.cumsum(nt) - nt, nt)
    return qi[rep], dist[qi, j][rep], g.tids[e[rep], slot]


def select(parts, nq, k):
    """The k smallest (distance, tid) pairs per query of the union of expand() outputs, padded with -1 / +inf."""
    qi = np.concatenate([p[0] for p in parts] + [np.zeros(0, np.int64)]).astype(np.int64)
    d = np.concatenate([p[1] for p in parts] + [np.zeros(0, np.float32)]).astype(np.float32)
    t = np.concatenate([p[2] for p in parts] + [np.zeros(0, np.int64)]).astype(np.int64)
    order = np.lexsort((t, d, qi))
    qi, d, t = qi[order], d[order], t[order]
    start = np.searchsorted(qi, np.arange(nq))
    rank = np.arange(len(qi)) - start[qi]
    keep = rank < k
    out_t = np.full((nq, k), -1, np.int64)
    out_d = np.full((nq, k), np.inf, np.float32)
    out_t[qi[keep], rank[keep]] = t[keep]
    out_d[qi[keep], rank[keep]] = d[keep]
    return out_t, out_d


def answer(graphs, queries, k, ef, threads=4):
    """graphs: the graph each partition exports (None or n = 0 for an empty partition).  Returns (tids, dist, counters):
    nq x k heap TIDs and distances, and the oracle's scan counters summed over the partitions."""
    queries = np.asarray(queries)
    nq = queries.shape[0]
    parts = []
    ctr = {"n_dist": 0, "n_hop0": 0, "n_hopu": 0}
    for g in graphs:
        if g is None or g.n == 0 or nq == 0:
            continue
        orc = O.Index.from_graph(g, O.CANON)
        e, d, c, oc = orc.search_batch(queries, ef, threads=threads)
        parts.append(expand(g, e, d, c))
        for key in ctr:
            ctr[key] += oc[key]
    t, d = select(parts, nq, k)
    return t, d, ctr
