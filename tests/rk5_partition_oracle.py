"""tests/rk5_partition_oracle.py — TEST INFRASTRUCTURE ONLY.

caar_dss_interior / caar_dss_boundary (include/caar_b200.h) transcribed in numpy on top of dss_partition_oracle's
``Part``: the local groups split into interior groups (every copy on this part) and boundary groups (at least one
copy on another part). ``interior`` assembles the interior groups without the receive buffer: its remote slots hold NaN,
as if the segments had not arrived. ``boundary`` assembles the boundary groups from the received segments and writes
only the local copies. Each pass is dss_oracle.dss_np restricted to its groups, so a point's sum runs in copy order.

Deliberately wrong variants the CPU tests must catch: ``defect="boundary_in_interior"`` moves one boundary group into
the interior set; ``defect="boundary_writes_remote"`` lets the boundary pass write its result into the received
records too.
"""
from __future__ import annotations

import numpy as np

import dss_oracle as do
import dss_partition_oracle as dpo

DEFECTS = ("boundary_in_interior", "boundary_writes_remote")


class SplitPart(dpo.Part):
    def __init__(self, gid, part_start, part, defect=None):
        assert defect in (None,) + DEFECTS
        super().__init__(gid, part_start, part)
        self.defect = defect
        local = lambda c: self.e0 <= c // 16 < self.e1
        self.interior = [i for i, g in enumerate(self.groups) if all(local(c) for c in g)]
        self.boundary = [i for i, g in enumerate(self.groups) if not all(local(c) for c in g)]
        if defect == "boundary_in_interior" and self.boundary:
            self.interior = sorted(self.interior + self.boundary[:1])
            self.boundary = self.boundary[1:]
        self.remote = {}                                   # global copy -> its slot in the receive buffer
        for q, c in enumerate(self.recv):
            for cp in c:
                self.remote[cp] = len(self.remote)

    def receive(self, segments):
        """segments[q]: what part q packed for this part -> the receive buffer (spheremp [R], values [R, ...])"""
        rs, rf = [], []
        for q, c in enumerate(self.recv):
            if c:
                sq, fq = segments[q]
                assert len(sq) == len(c)
                rs.extend(sq)
                rf.extend(fq)
        return np.array(rs, dtype=np.float64), np.array(rf)

    def _pass(self, which, f, s, rs, rf, weighting):
        n = 16 * self.nl
        ids = self.interior if which == "interior" else self.boundary
        if not ids:
            return
        rf = rf.reshape((-1,) + f.shape[1:])
        f_ext, s_ext = np.concatenate([f, rf]), np.concatenate([s, rs])

        class Conn:
            pass
        conn = Conn()
        grps = [self.groups[i] for i in ids]
        conn.mult = np.array([len(g) for g in grps], dtype=np.int64)
        conn.M = int(conn.mult.max())
        conn.idx = np.full((len(grps), conn.M), -1, dtype=np.int64)
        for i, g in enumerate(grps):
            conn.idx[i, :len(g)] = [c - 16 * self.e0 if self.e0 <= c // 16 < self.e1 else n + self.remote[c] for c in g]
        out = do.dss_np(f_ext, s_ext, conn, weighting)
        f[:] = out[:n]
        if which == "boundary" and self.defect == "boundary_writes_remote" and len(rf):
            rf[:] = out[n:]

    def interior_pass(self, f, s, weighting):
        """in place on f [16 nl, ...]; the receive buffer is not read: its slots are NaN here"""
        R = len(self.remote)
        self._pass("interior", f, s, np.full(R, np.nan), np.full((R,) + f.shape[1:], np.nan), weighting)

    def boundary_pass(self, f, s, rs, rf, weighting):
        """in place on f; rs, rf the receive buffer"""
        self._pass("boundary", f, s, rs, rf, weighting)

    def unpack_split(self, f, s, segments, weighting, order="interior_first"):
        """-> (the assembled f, the receive buffer's values after both passes)"""
        rs, rf = self.receive(segments)
        f = f.copy()
        rf = rf.reshape((-1,) + f.shape[1:]) if len(rf) else np.zeros((0,) + f.shape[1:])
        if order == "interior_first":
            self.interior_pass(f, s, weighting)
            self.boundary_pass(f, s, rs, rf, weighting)
        else:
            self.boundary_pass(f, s, rs, rf, weighting)
            self.interior_pass(f, s, weighting)
        return f, rf


def dss_split(gid, part_start, f, s, weighting, order="interior_first", defect=None):
    """f [16 E, ...], s [16 E] of the whole mesh: pack on every part, exchange, interior and boundary in `order` ->
    (the concatenated result, whether every receive buffer still holds what was received)"""
    ps = np.asarray(part_start)
    parts = [SplitPart(gid, ps, p, defect) for p in range(len(ps) - 1)]
    sl = [slice(16 * ps[p], 16 * ps[p + 1]) for p in range(len(parts))]
    rec = dpo.exchange(parts, [pt.pack(f[sl[p]], s[sl[p]]) for p, pt in enumerate(parts)])
    out, kept = [], True
    for p, pt in enumerate(parts):
        got, rf = pt.unpack_split(f[sl[p]], s[sl[p]], rec[p], weighting, order)
        _, want_rf = pt.receive(rec[p])
        kept = kept and np.array_equal(np.ascontiguousarray(rf).view(np.uint64).reshape(-1),
                                       np.ascontiguousarray(want_rf).view(np.uint64).reshape(-1))
        out.append(got)
    return np.concatenate(out), kept
