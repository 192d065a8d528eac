"""Rows as a graph without edges: the exact scan reads only the vectors, so its tests load raw rows this way.  Test
helper shared by the oracle-only test of the exact top-k reference (test_oracle_exact.py) and the GPU exact-scan
tests (test_gpu_bruteforce.py)."""
import numpy as np

HEAPTIDS = 10


class Graph:
    pass


def flat_graph(x, metric, dtype, m=8, efc=32):
    """n rows, each its own heap TID, every element on layer 0 with no neighbours, element 0 the entry point.
    Rows are used as given: a cosine caller passes rows that are already normalised."""
    n, dim = x.shape
    g = Graph()
    g.dim, g.m, g.efc, g.metric, g.dtype, g.n, g.upper_rows = dim, m, efc, metric, dtype, n, 0
    g.entry, g.entry_level = (0 if n else -1), 0
    g.vecs = np.ascontiguousarray(x, np.float16 if dtype else np.float32)
    g.level = np.zeros(n, np.uint8)
    g.nbr0 = np.full((n, 2 * m), -1, np.int32)
    g.uoff = np.full(n, -1, np.int32)
    g.nbru = np.full((1, m), -1, np.int32)
    g.ntids = np.ones(n, np.uint8)
    g.tids = np.zeros((n, HEAPTIDS), np.int64)
    g.tids[:, 0] = np.arange(n)
    return g
