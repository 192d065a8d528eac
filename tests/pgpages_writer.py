"""Writer of pgvector HNSW index pages in the layout csrc/pgpages.cu reads (pgvector 0.7-0.8 hnsw.h +
PostgreSQL page format AS RECALLED; there is no PostgreSQL here to produce a real file).  Test helper."""
import struct

import numpy as np

BLCKSZ = 8192
INVALID_BLK = 0xFFFFFFFF


def _maxalign(n):
    return (n + 7) & ~7


def _tid(blk, off):
    return struct.pack("<HHH", (blk >> 16) & 0xffff, blk & 0xffff, off)


class _Page:
    def __init__(self):
        self.buf = bytearray(BLCKSZ)
        self.items = []
        self.upper = BLCKSZ - 8

    def free(self):
        return self.upper - (24 + 4 * (len(self.items) + 1))

    def add(self, tup):
        size = _maxalign(len(tup))
        self.upper -= size
        self.buf[self.upper:self.upper + len(tup)] = tup
        self.items.append((self.upper, len(tup)))
        return len(self.items)          # offset number (1-based)

    def finish(self, nextblk):
        lower = 24 + 4 * len(self.items)
        struct.pack_into("<QHHHHHHI", self.buf, 0, 0, 0, 0, lower, self.upper, BLCKSZ - 8, BLCKSZ | 4, 0)
        for i, (off, ln) in enumerate(self.items):
            struct.pack_into("<I", self.buf, 24 + 4 * i, off | (1 << 15) | (ln << 17))
        struct.pack_into("<IHH", self.buf, BLCKSZ - 8, nextblk, 0, 0xFF90)
        return bytes(self.buf)


def write_pages(g, m, efc, dim, half=False, scatter=False, deleted=()):
    """g: flat graph (oracle.Graph / export()); returns the relation file's bytes.  scatter: neighbour
    tuples go to pages of their own (exercises the neighbortid indirection); deleted: element ids to
    mark deleted."""
    n = g.n
    esz = 2 if half else 4
    vec_hdr = lambda: struct.pack("<ihh", (8 + dim * esz) << 2, dim, 0)
    pages = [_Page()]
    where = {}            # element -> (blk, off)
    nwhere = {}           # element -> (blk, off) of its neighbour tuple
    pending = []          # (page index, item index, element) of neighbour tuples to patch
    esize = _maxalign(72 + 8 + dim * esz)

    def nsize(e):
        return _maxalign(4 + 6 * (int(g.level[e]) + 2) * m)

    # placement first (tuples reference each other by position)
    plan = []
    cur, used = 0, [24]   # rough accounting: header + line pointers + tuples
    def fits(pi, size, nitems):
        return used[pi] + size + 4 * nitems <= BLCKSZ - 8
    spill = []
    for e in range(n):
        need = esize + (0 if scatter else nsize(e))
        if not fits(cur, need, 1 if scatter else 2):
            cur += 1
            used.append(24)
        used[cur] += need + (4 if scatter else 8)
        plan.append(cur)
    blk_of_page = lambda pi: pi + 1
    # materialise: elements (and their neighbour tuples when not scattered) page by page
    pages = [_Page() for _ in range(cur + 1)]
    for e in range(n):
        pg = pages[plan[e]]
        off = len(pg.items) + 1
        where[e] = (blk_of_page(plan[e]), off)
        pg.items.append(None)
        if not scatter:
            nwhere[e] = (blk_of_page(plan[e]), off + 1)
            pg.items.append(None)
    if scatter:
        pi = len(pages)
        pages.append(_Page())
        room = BLCKSZ - 8 - 24
        for e in range(n):
            if room < nsize(e) + 4:
                pages.append(_Page())
                pi += 1
                room = BLCKSZ - 8 - 24
            room -= nsize(e) + 4
            nwhere[e] = (blk_of_page(pi), len(pages[pi].items) + 1)
            pages[pi].items.append(None)
    for p in pages:
        p.items = []
    # now write the tuples in the planned order
    order = {}
    for e in range(n):
        order.setdefault(where[e][0], []).append(("e", where[e][1], e))
        order.setdefault(nwhere[e][0], []).append(("n", nwhere[e][1], e))
    for blk, lst in order.items():
        pg = pages[blk - 1]
        for kind, off, e in sorted(lst, key=lambda t: t[1]):
            if kind == "e":
                t = bytearray()
                t += struct.pack("<BBBB", 1, int(g.level[e]), 1 if e in deleted else 0, 0)
                nt = int(g.ntids[e])
                for k in range(10):
                    if k < nt:
                        tid = int(g.tids[e, k])
                        t += _tid(tid >> 16, tid & 0xffff)
                    else:
                        t += _tid(INVALID_BLK, 0)
                t += _tid(*nwhere[e])
                t += struct.pack("<H", 0)
                t += vec_hdr()
                t += np.ascontiguousarray(g.vecs[e]).tobytes()
            else:
                lv = int(g.level[e])
                t = bytearray(struct.pack("<BBH", 2, 0, (lv + 2) * m))
                for lc in range(lv, -1, -1):
                    lst_ = g.nbr0[e] if lc == 0 else g.nbru[int(g.uoff[e]) + lc - 1]
                    for j in range(2 * m if lc == 0 else m):
                        x = int(lst_[j])
                        t += _tid(*where[x]) if x >= 0 else _tid(INVALID_BLK, 0)
            got = pg.add(bytes(t))
            assert got == off, (got, off)
    meta = bytearray(BLCKSZ)
    # no entry point (an empty index, or one whose every element was vacuumed away): InvalidBlockNumber, offset 0
    has_entry = n > 0 and int(g.entry) >= 0
    eb, eo = where[int(g.entry)] if has_entry else (INVALID_BLK, 0)
    struct.pack_into("<QHHHHHHI", meta, 0, 0, 0, 0, 24 + 28, BLCKSZ - 8, BLCKSZ - 8, BLCKSZ | 4, 0)
    struct.pack_into("<IIIHHIHhI", meta, 24, 0xA953A953, 1, dim, m, efc, eb, eo, int(g.level[int(g.entry)]) if has_entry else -1, len(pages))
    struct.pack_into("<IHH", meta, BLCKSZ - 8, INVALID_BLK, 0, 0xFF90)
    out = bytes(meta)
    for i, p in enumerate(pages):
        out += p.finish(i + 2 if i + 1 < len(pages) else INVALID_BLK)
    return out
