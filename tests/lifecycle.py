"""Round scripts of the index lifecycle: insert -> bulk delete (ambulkdelete's RemoveHeapTids) -> vacuum (RepairGraph +
MarkDeleted), repeated on a graph that has been repaired before.  Test helper shared by the oracle-only test
(test_oracle_lifecycle.py) and the GPU-against-oracle test (test_gpu_lifecycle.py): every plan is drawn from the
oracle's graph, so both sides of a comparison receive the same operations."""
import numpy as np

from conftest import clustered, sift_like

HEAPTIDS = 10
MISSING_TID = (1 << 40) + 1             # a heap TID no index ever holds
# per round: share of the live heap TIDs deleted, and whether VACUUM runs (round 1 leaves its emptied elements in the
# graph through the inserts of round 2)
ROUNDS = ((0.10, True), (0.40, False), (0.0, True), (0.70, True))


def heap_tid(k):
    """k-th heap TID: (block k // 200, offset k % 200 + 1); offsets start at 1 as ItemPointers' do"""
    return ((k // 200) << 16) | (k % 200 + 1)


class Rows:
    """Input rows by heap TID (cosine indexes store them normalised; byte copies must be made of the input)."""

    def __init__(self, dim, dtype, gen, seed):
        self.dim, self.dtype, self.gen, self.seed = dim, dtype, gen, seed
        self.by_tid = {}
        self.k = 0
        self.drawn = 0
        self.deleted_from = {}          # element -> a heap TID it held before bulk delete emptied it

    def fresh(self, n):
        self.drawn += 1
        if self.gen == "sift":
            return sift_like(n, self.dim, seed=self.seed * 100 + self.drawn).astype(self.dtype)
        return clustered(n, self.dim, 16, seed=self.seed * 100 + self.drawn, dtype=self.dtype)

    def tids(self, rows):
        out = np.array([heap_tid(self.k + i) for i in range(len(rows))], np.int64)
        self.k += len(rows)
        for t, r in zip(out.tolist(), rows):
            self.by_tid[t] = np.array(r, copy=True)
        return out


def insert_plan(g, rows, rng, metric_is_cosine, n_fresh=170):
    """~200 rows: fresh ones, byte copies of live rows (one of them 12 times: it fills an element's HEAPTIDS and spills
    into a new element), byte copies of rows whose TIDs were deleted but not vacuumed yet (they fold into the emptied
    element), and a zero vector under cosine (dropped).  Returns (rows, heap TIDs)."""
    parts = [rows.fresh(n_fresh)]
    live = np.nonzero(g.ntids > 0)[0]
    if len(live):
        pick = rng.choice(live, min(8, len(live)), replace=False)
        copies = [rows.by_tid[int(g.tids[e, 0])] for e in pick]
        copies += [rows.by_tid[int(g.tids[pick[0], 0])]] * 11
        parts.append(np.stack(copies))
    emptied = [e for e in range(g.n) if g.ntids[e] == 0 and g.vecs[e].any()]
    if emptied:
        pick = rng.choice(emptied, min(10, len(emptied)), replace=False)
        parts.append(np.stack([rows.by_tid[rows.deleted_from[int(e)]] for e in pick]))
    if metric_is_cosine:
        parts.append(np.zeros((1, rows.dim), rows.dtype))
    x = np.concatenate(parts).astype(rows.dtype)
    x = x[rng.permutation(len(x))]
    return x, rows.tids(x)


def delete_plan(g, rng, frac):
    """TIDs to delete: `frac` of the live heap TIDs at random, every TID of the entry point, the first (not every) TID of
    up to three multi-TID elements, and a TID that is not in the index."""
    live_tids = np.array([int(t) for e in range(g.n) for t in g.tids[e, :g.ntids[e]]], np.int64)
    dead = set(rng.choice(live_tids, int(round(frac * len(live_tids))), replace=False).tolist()) if len(live_tids) else set()
    if g.entry >= 0:
        dead |= set(int(t) for t in g.tids[g.entry, :g.ntids[g.entry]])
    multi = [e for e in range(g.n) if g.ntids[e] >= 2 and e != g.entry]
    for e in multi[:3]:
        keep = [int(t) for t in g.tids[e, 1:g.ntids[e]]]
        dead.discard(keep[0])           # at least one TID of the element survives
        dead.add(int(g.tids[e, 0]))
    out = np.array(sorted(dead) + [MISSING_TID], np.int64)
    return out[rng.permutation(len(out))]


def note_deleted(g, rows, dead):
    """remember, per element about to be emptied, one of its TIDs (for byte copies of it later)"""
    dead = set(dead.tolist())
    for e in range(g.n):
        ts = [int(t) for t in g.tids[e, :g.ntids[e]]]
        if ts and all(t in dead for t in ts):
            rows.deleted_from[e] = ts[0]


def check_invariants(g, marked, after_vacuum):
    """marked: elements MarkDeleted has removed.  Lists of the other elements never point at one of them; they have no
    lists, a zero vector and no TIDs; the entry point is not one of them, and after a vacuum it is -1 exactly when no
    element is live."""
    marked = np.array(sorted(marked), np.int64)
    gone = np.zeros(g.n, bool)
    gone[marked] = True
    assert (g.ntids[gone] == 0).all()
    assert (g.nbr0[gone] == -1).all()
    assert not g.vecs[gone].any()
    for e in marked:
        for lc in range(1, int(g.level[e]) + 1):
            assert (g.nbru[int(g.uoff[e]) + lc - 1] == -1).all()
    nb0 = g.nbr0[~gone]
    assert not gone[nb0[nb0 >= 0]].any(), "a layer-0 list points at a deleted element"
    for e in np.nonzero(~gone & (g.level > 0))[0]:
        rowsu = g.nbru[int(g.uoff[e]):int(g.uoff[e]) + int(g.level[e])]
        assert not gone[rowsu[rowsu >= 0]].any(), "an upper-layer list points at a deleted element"
    if g.entry >= 0:
        assert not gone[g.entry]
        assert g.entry_level == g.level[g.entry]
    if after_vacuum:
        assert (g.entry == -1) == (not (g.ntids > 0).any())


def live_tids(g):
    return set(int(t) for e in range(g.n) for t in g.tids[e, :g.ntids[e]])


def run_rounds(orc, rows, seed, cosine, apply, check):
    """The ROUNDS on the oracle `orc`.  apply(op, *args) repeats each operation on the side under test: ("insert", rows,
    tids, count indexed by the oracle), ("delete", tids, TIDs removed by the oracle), ("vacuum", (marked, repaired) of
    the oracle).  check(step, marked, after_vacuum) runs after every step; `marked` = the elements vacuumed away."""
    rng = np.random.default_rng(seed)
    marked = set()
    for r, (frac, vacuum) in enumerate(ROUNDS):
        x, t = insert_plan(orc.export(), rows, rng, cosine)
        got = [orc.insert(x[i], int(t[i])) for i in range(len(x))]
        apply("insert", x, t, sum(1 for e in got if e >= 0))
        check("round %d insert" % r, marked, False)
        g = orc.export()
        dead = delete_plan(g, rng, frac)
        note_deleted(g, rows, dead)
        apply("delete", dead, orc.bulk_delete(dead))
        check("round %d delete" % r, marked, False)
        if vacuum:
            res = orc.vacuum_repair()
            g = orc.export()
            marked |= set(np.nonzero(g.ntids == 0)[0].tolist())
            apply("vacuum", res)
            check("round %d vacuum" % r, marked, True)
    return marked
