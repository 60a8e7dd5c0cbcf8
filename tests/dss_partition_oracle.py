"""tests/dss_partition_oracle.py — TEST INFRASTRUCTURE ONLY.

The DSS and ``neighbor_minmax`` across partitioned handles (``caar_set_partition``, ``caar_dss_pack`` /
``caar_dss_unpack``, ``caar_neighbor_minmax_pack`` / ``caar_neighbor_minmax_unpack`` in include/caar_b200.h),
transcribed in numpy from the header's text: each ``Part`` knows only the global-id map and its own block. ``pack``
builds, for every other part q, the records of the local copies of points q also holds (spheremp and the values), or
the bound rows of the local elements with a neighbour in q; ``exchange`` moves segment p->q to part q; ``unpack`` sums
every point's copies, local and received, in (global e, p) order with dss_oracle's sequential-by-rank numpy transcription
(or widens the bounds over N(e) in ascending global element order). The record order inside a segment is this module's
own (the global sort by (gid, global e, p)); only the segment sizes have to agree with the library's.

``Part(..., defect="remote_after_local")`` sums a point's received copies after its local ones: a deliberately wrong
variant the CPU tests must catch.
"""
from __future__ import annotations

import numpy as np

import dss_oracle as do


def block_partition(E, nparts, rng, one_element_block=True):
    """part_start [nparts + 1]: nparts contiguous non-empty blocks of E elements at random cuts; with nparts > 1 and
    one_element_block, the first block is one element"""
    assert 1 <= nparts <= E
    if nparts == 1:
        return np.array([0, E], dtype=np.int32)
    fixed = [1] if one_element_block else []
    pool = np.setdiff1d(np.arange(1, E), fixed)
    cuts = np.sort(np.concatenate([fixed, rng.choice(pool, nparts - 1 - len(fixed), replace=False)]))
    return np.concatenate([[0], cuts, [E]]).astype(np.int32)


class Part:
    def __init__(self, gid, part_start, part, defect=None):
        assert defect in (None, "remote_after_local")
        flat = np.asarray(gid, dtype=np.int64).reshape(-1)
        self.ps = np.asarray(part_start, dtype=np.int64)
        self.nparts = len(self.ps) - 1
        self.part = part
        self.e0, self.e1 = int(self.ps[part]), int(self.ps[part + 1])
        self.nl = self.e1 - self.e0
        order = np.lexsort((np.arange(flat.size), flat))              # by (gid, global e*16 + p)
        g = flat[order]
        starts = np.flatnonzero(np.r_[True, g[1:] != g[:-1]])
        ends = np.r_[starts[1:], flat.size]
        part_of = np.searchsorted(self.ps, np.arange(self.ps[-1]), side="right") - 1
        self.groups = []                                    # every point with a local copy: its global copies in order
        self.send = [[] for _ in range(self.nparts)]         # local copies (global index) each part receives
        self.recv = [[] for _ in range(self.nparts)]         # copies of each part received here
        nb = {}
        for a, b in zip(starts, ends):
            cps = [int(x) for x in order[a:b]]
            els = [c // 16 for c in cps]
            if not any(self.e0 <= e < self.e1 for e in els):
                continue
            self.groups.append(cps)
            others = sorted({int(part_of[e]) for e in els} - {part})
            for c, e in zip(cps, els):
                if self.e0 <= e < self.e1:
                    for q in others:
                        self.send[q].append(c)
                    nb.setdefault(e, set()).update(x for x in els if x != e)
                else:
                    self.recv[int(part_of[e])].append(c)
        self.neighbours = [sorted(nb.get(e, ())) for e in range(self.e0, self.e1)]   # global, ascending
        self.send_el = [[] for _ in range(self.nparts)]
        self.recv_el = [[] for _ in range(self.nparts)]
        for i, ns in enumerate(self.neighbours):
            for q in sorted({int(part_of[x]) for x in ns} - {part}):
                self.send_el[q].append(self.e0 + i)
            for x in ns:
                if not self.e0 <= x < self.e1:
                    self.recv_el[int(part_of[x])].append(x)
        self.recv_el = [sorted(set(r)) for r in self.recv_el]
        if defect == "remote_after_local":
            loc = lambda c: self.e0 <= c // 16 < self.e1
            self.groups = [[c for c in g if loc(c)] + [c for c in g if not loc(c)] for g in self.groups]

    # -- the DSS: f is the part's [16 nl, ...] values (points leading), s its [16 nl] spheremp --
    def pack(self, f, s):
        """-> [segment q: (spheremp [n_q], values [n_q, ...])]"""
        return [(s[np.array(c, dtype=np.int64) - 16 * self.e0], f[np.array(c, dtype=np.int64) - 16 * self.e0])
                if c else None for c in self.send]

    def unpack(self, f, s, segments, weighting):
        """segments[q]: what part q packed for this part -> the assembled f (a new array)"""
        rem_index, rs, rf = {}, [], []
        n = 16 * self.nl
        for q, c in enumerate(self.recv):
            if not c:
                continue
            sq, fq = segments[q]
            assert len(sq) == len(c)
            for k, cp in enumerate(c):
                rem_index[cp] = n + len(rs)
                rs.append(sq[k])
                rf.append(fq[k])
        s_ext = np.concatenate([s, np.array(rs, dtype=np.float64)])
        f_ext = np.concatenate([f, np.array(rf).reshape((-1,) + f.shape[1:])]) if rf else f.copy()
        ext = lambda c: c - 16 * self.e0 if self.e0 <= c // 16 < self.e1 else rem_index[c]

        class Conn:
            pass
        conn = Conn()
        conn.mult = np.array([len(g) for g in self.groups], dtype=np.int64)
        conn.M = int(conn.mult.max())
        conn.idx = np.full((len(self.groups), conn.M), -1, dtype=np.int64)
        for i, g in enumerate(self.groups):
            conn.idx[i, :len(g)] = [ext(c) for c in g]
        return do.dss_np(f_ext, s_ext, conn, weighting)[:n]

    # -- neighbor_minmax: b is the part's bounds [nl][qsize_d][L][2] --
    def pack_bounds(self, b, qsize):
        return [b[np.array(r, dtype=np.int64) - self.e0, :qsize] if r else None for r in self.send_el]

    def unpack_bounds(self, b, segments, qsize):
        rows, index = [b], {}
        n = self.nl
        for q, r in enumerate(self.recv_el):
            if not r:
                continue
            seg = segments[q]
            assert seg.shape[0] == len(r)
            full = np.zeros((len(r),) + b.shape[1:])
            full[:, :qsize] = seg
            rows.append(full)
            for k, x in enumerate(r):
                index[x] = n
                n += 1
        b_ext = np.concatenate(rows)

        class Conn:
            pass
        conn = Conn()
        conn.E = b_ext.shape[0]
        loc = lambda x: x - self.e0 if self.e0 <= x < self.e1 else index[x]
        conn.neighbours = [[loc(x) for x in ns] for ns in self.neighbours] + [[]] * (conn.E - self.nl)
        return do.neighbor_minmax_np(b_ext, conn, qsize)[:self.nl]


def exchange(parts, packed):
    """packed[p]: part p's segments -> received[q][p] = segment p->q"""
    return [[packed[p][q] for p in range(len(parts))] for q in range(len(parts))]


def dss_partitioned(gid, part_start, f, s, weighting, defect=None):
    """f [16 E, ...], s [16 E] of the whole mesh: pack on every part, exchange, unpack -> the concatenated result"""
    ps = np.asarray(part_start)
    parts = [Part(gid, ps, p, defect) for p in range(len(ps) - 1)]
    sl = [slice(16 * ps[p], 16 * ps[p + 1]) for p in range(len(parts))]
    rec = exchange(parts, [pt.pack(f[sl[p]], s[sl[p]]) for p, pt in enumerate(parts)])
    return np.concatenate([pt.unpack(f[sl[p]], s[sl[p]], rec[p], weighting) for p, pt in enumerate(parts)])


def neighbor_minmax_partitioned(gid, part_start, b, qsize):
    ps = np.asarray(part_start)
    parts = [Part(gid, ps, p) for p in range(len(ps) - 1)]
    sl = [slice(ps[p], ps[p + 1]) for p in range(len(parts))]
    rec = exchange(parts, [pt.pack_bounds(b[sl[p]], qsize) for p, pt in enumerate(parts)])
    return np.concatenate([pt.unpack_bounds(b[sl[p]], rec[p], qsize) for p, pt in enumerate(parts)])
