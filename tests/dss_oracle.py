"""tests/dss_oracle.py — TEST INFRASTRUCTURE ONLY.

HOMME's direct stiffness summation (DSS) and ``neighbor_minmax`` as specified in include/caar_b200.h (``caar_dss``,
``caar_neighbor_minmax``), transcribed twice:

  * ``dss_scalar`` / ``neighbor_minmax_scalar``: literal loops over points, copies and neighbours on Python floats (IEEE
    double, every operation rounded separately), following the header's text line by line;
  * ``dss_np`` / ``neighbor_minmax_np``: numpy, vectorised over groups (or bound pairs) but sequential over the rank of a
    copy in its group (or of a neighbour in its list). No ``np.sum`` or ``np.add.at``: their order is not the header's.

``dss_arrays`` applies the numpy transcription to handle-shaped arrays, as caar_dss does (the neighbor_minmax transcriptions
take the handle-shaped bounds themselves), and ``rk5_dss_step`` composes ``rk5_oracle.schedule`` / ``rotate`` with a single-call oracle and the DSS after every
stage (``caar_run_rk5_dss``).

Meshes: ``cubed_sphere_gid`` builds HOMME's cubed sphere exactly, on integers; ``random_gid`` builds groups of any size
that no sphere has, including two points of one element with one id.

``dss_np`` takes ``defect`` (one of ``DEFECTS``) and ``Connectivity`` takes ``defect="edges_only"``: deliberately wrong
variants that the CPU tests must catch.
"""
from __future__ import annotations

import numpy as np

import rk5_oracle as ro

ASSEMBLE, PROJECT = 0, 1
DEFECTS = ("descending", "local_r", "inplace")
STATE = ("elem_state_v", "elem_state_T", "elem_state_dp3d")


# ---- meshes ---------------------------------------------------------------------------------------------------------

D4 = [(k, t) for t in (False, True) for k in range(4)]   # rotations by k quarter turns, optionally after a transpose


def cubed_sphere_gid(ne, rng=None):
    """gid [6 ne^2][4][4] (int64) of the cubed sphere with ne x ne elements per face. Face f lies on the surface of the
    cube [0, 3ne]^3; element (f, a, b) covers the lattice points 3a..3a+3 x 3b..3b+3 of its face, and the id of a point is
    its integer position (x, y, z) packed into one integer: points on the edges and corners of the cube are shared between
    faces exactly. With rng, the elements are put in a random order and each element's 4x4 block gets a random dihedral
    orientation, as HOMME's panels are rotated against each other."""
    N = 3 * ne
    ids = []
    for axis in range(3):
        for side in (0, N):
            u_ax, v_ax = [a for a in range(3) if a != axis]
            for a in range(ne):
                for b in range(ne):
                    i = 3 * a + np.arange(4)[:, None]
                    j = 3 * b + np.arange(4)[None, :]
                    xyz = [None, None, None]
                    xyz[axis] = np.full((4, 4), side)
                    xyz[u_ax] = np.broadcast_to(i, (4, 4))
                    xyz[v_ax] = np.broadcast_to(j, (4, 4))
                    ids.append((xyz[0] * (N + 1) + xyz[1]) * (N + 1) + xyz[2])
    gid = np.array(ids, dtype=np.int64)
    if rng is not None:
        gid = gid[rng.permutation(len(gid))]
        for e in range(len(gid)):
            k, t = D4[rng.integers(8)]
            blk = gid[e].T if t else gid[e]
            gid[e] = np.rot90(blk, k)
    return np.ascontiguousarray(gid)


def random_gid(E, rng, max_mult):
    """gid [E][4][4] of a mesh that is no sphere: the 16 E points are cut into groups of 1 .. max_mult copies at random,
    each with a random 64-bit id of either sign; points 0 and 5 of element 0 always form one group (two points of one
    element with one id)."""
    slots = np.concatenate([[0, 5], rng.permutation(np.setdiff1d(np.arange(16 * E), [0, 5]))])
    sizes = [2]
    while sum(sizes) < 16 * E:
        sizes.append(int(min(16 * E - sum(sizes), rng.integers(1, max_mult + 1))))
    ids = rng.choice(1 << 62, size=len(sizes), replace=False) * rng.choice([-1, 1], size=len(sizes))
    gid = np.empty(16 * E, dtype=np.int64)
    o = 0
    for n, g in zip(sizes, ids):
        gid[slots[o:o + n]] = g
        o += n
    return gid.reshape(E, 4, 4)


class Connectivity:
    """The groups of copies of a gid map, as the header defines them: copies (e, p), p = 4*igp + jgp, ordered by (e, p);
    groups in the order of their owners. idx [G][M] holds the flat copy e*16 + p by rank (-1 beyond mult[g]);
    neighbours[e] is N(e), ascending."""

    def __init__(self, gid, defect=None):
        gid = np.asarray(gid, dtype=np.int64).reshape(-1, 16)
        self.E = gid.shape[0]
        flat = gid.reshape(-1)
        order = np.lexsort((np.arange(flat.size), flat))          # by (gid, e*16 + p)
        g_sorted = flat[order]
        starts = np.flatnonzero(np.r_[True, g_sorted[1:] != g_sorted[:-1]])
        ends = np.r_[starts[1:], flat.size]
        owner = order[starts]
        by_owner = np.argsort(owner, kind="stable")
        starts, ends = starts[by_owner], ends[by_owner]
        self.mult = (ends - starts).astype(np.int64)
        self.G, self.M = len(starts), int(self.mult.max())
        self.idx = np.full((self.G, self.M), -1, dtype=np.int64)
        for c in range(self.M):
            has = self.mult > c
            self.idx[has, c] = order[starts[has] + c]
        self.groups = [list(order[a:b]) for a, b in zip(starts, ends)]   # for the scalar transcription
        nb = [set() for _ in range(self.E)]
        for grp in self.groups:
            if defect == "edges_only" and len(grp) != 2:
                continue
            els = {int(c) // 16 for c in grp}
            for e in els:
                nb[e] |= els - {e}
        self.neighbours = [sorted(s) for s in nb]


# ---- the DSS ----------------------------------------------------------------------------------------------------------

def dss_scalar(f, s, conn, weighting):
    """The header's text on one level of one field: f, s are lists of 16 E floats (flat e*16 + p) -> the new f."""
    out = list(f)
    for grp in conn.groups:
        m = s[grp[0]]
        for c in grp[1:]:
            m = m + s[c]
        r = 1.0 / m
        S = f[grp[0]] if weighting == ASSEMBLE else s[grp[0]] * f[grp[0]]
        for c in grp[1:]:
            S = S + (f[c] if weighting == ASSEMBLE else s[c] * f[c])
        for c in grp:
            out[c] = S * r
    return out


def dss_scalar_inplace_defect(f, s, conn, weighting):
    """A wrong DSS: each copy in turn sums its group from the array it is updating, so later copies see new values."""
    out = list(f)
    for grp in conn.groups:
        m = s[grp[0]]
        for c in grp[1:]:
            m = m + s[c]
        r = 1.0 / m
        for tgt in grp:
            S = out[grp[0]] if weighting == ASSEMBLE else s[grp[0]] * out[grp[0]]
            for c in grp[1:]:
                S = S + (out[c] if weighting == ASSEMBLE else s[c] * out[c])
            out[tgt] = S * r
    return out


def dss_np(f, s, conn, weighting, defect=None):
    """Numpy transcription: f [16 E, ...] (points leading, any trailing shape), s [16 E] -> a new array. Rank c of every
    group is added in step c, so each sum runs in copy order."""
    assert defect in (None,) + DEFECTS
    if defect == "inplace":
        flat = f.reshape(f.shape[0], -1)
        cols = [dss_scalar_inplace_defect(flat[:, j].tolist(), s.tolist(), conn, weighting) for j in range(flat.shape[1])]
        return np.array(cols).T.reshape(f.shape)
    tail = (slice(None),) + (None,) * (f.ndim - 1)
    idx = conn.idx
    if defect == "descending":   # copy c of a group in place c-th from its end
        idx = idx.copy()
        for c in range(conn.M):
            has = conn.mult > c
            idx[has, c] = conn.idx[has, conn.mult[has] - 1 - c]

    def term(i):
        return f[i] if weighting == ASSEMBLE else s[i][tail] * f[i]
    m = s[idx[:, 0]]
    S = term(idx[:, 0])
    for c in range(1, conn.M):
        has = conn.mult > c
        m[has] = m[has] + s[idx[has, c]]
        S[has] = S[has] + term(idx[has, c])
    r = 1.0 / m
    out = f.copy()
    for c in range(conn.M):
        has = conn.mult > c
        i = idx[has, c]
        rr = 1.0 / s[i] if defect == "local_r" else r[has]
        out[i] = S[has] * rr[tail]
    return out


def dss_arrays(arrays, conn, names, tl=0, qtl=0, qsize=0, weighting=ASSEMBLE, defect=None):
    """caar_dss on handle-shaped numpy arrays (harness field shapes), in place: dp3d, v, T at time level tl, Qdp(qtl) of
    tracers < qsize."""
    E = conn.E
    s = arrays["elem_spheremp"].reshape(E * 16)
    for n in names:
        A = arrays[n]
        if n == "elem_state_Qdp" and qsize == 0:
            continue
        sl = np.s_[:, :qsize, qtl] if n == "elem_state_Qdp" else np.s_[:, tl]
        blk = A[sl]
        comp = (2,) if n == "elem_state_v" else ()
        x = blk.reshape((E, -1, 16) + comp)                      # [E][X][16](2)
        X = x.shape[1]
        pts = np.moveaxis(x, 2, 1).reshape((E * 16, X) + comp)   # [16 E][X](2)
        y = dss_np(pts, s, conn, weighting, defect)
        A[sl] = np.moveaxis(y.reshape((E, 16, X) + comp), 1, 2).reshape(blk.shape)
    return arrays


# ---- neighbor_minmax --------------------------------------------------------------------------------------------------

def neighbor_minmax_scalar(b, conn, qsize):
    """The header's text: b [E][qsize_d][L][2] -> a new array."""
    out = b.copy()
    E, _, L, _ = b.shape
    for e in range(E):
        for iq in range(qsize):
            for k in range(L):
                qmin, qmax = float(b[e, iq, k, 0]), float(b[e, iq, k, 1])
                for n in conn.neighbours[e]:
                    if b[n, iq, k, 0] < qmin:
                        qmin = float(b[n, iq, k, 0])
                    if b[n, iq, k, 1] > qmax:
                        qmax = float(b[n, iq, k, 1])
                out[e, iq, k] = (qmin, qmax)
    return out


def neighbor_minmax_np(b, conn, qsize):
    out = b.copy()
    if qsize == 0:
        return out
    deg = np.array([len(x) for x in conn.neighbours])
    D = int(deg.max()) if len(deg) else 0
    nb = np.zeros((conn.E, max(D, 1)), dtype=np.int64)
    for e, x in enumerate(conn.neighbours):
        nb[e, :len(x)] = x
    lo, hi = b[:, :qsize, :, 0].copy(), b[:, :qsize, :, 1].copy()
    for j in range(D):
        ok = (deg > j)[:, None, None]
        cand = b[nb[:, j], :qsize]
        lo = np.where(ok & (cand[..., 0] < lo), cand[..., 0], lo)
        hi = np.where(ok & (cand[..., 1] > hi), cand[..., 1], hi)
    out[:, :qsize, :, 0], out[:, :qsize, :, 1] = lo, hi
    return out


# ---- RK5 with the DSS after every stage -------------------------------------------------------------------------------

def rk5_dss_step(orc, state, dt, conn, hybi=None):
    """caar_run_rk5_dss's step on a harness.State, in place: rk5_oracle's schedule with dss_arrays(v, T, dp3d, the
    stage's np1, ASSEMBLE) after each stage. state.ctl's levels come back rotated; dt2 and eta_ave_w restored."""
    n0, np1, nm1 = (int(x) for x in state.ctl[2:5])
    assert len({n0, np1, nm1}) == 3 and (int(state.ctl[0]), int(state.ctl[1])) == (0, state.nelem)
    dt2, w = state.dt2, float(state.consts[1])
    for st in ro.schedule(n0, np1, nm1, float(dt), w):
        if st == "combine":
            for name in ro.COMBINED:
                X = state.arrays[name]
                X[:, nm1] = (5 * X[:, nm1] - X[:, n0]) / 4
            continue
        state.ctl[2:5] = st[:3]
        state.dt2, state.consts[1] = st[3], st[4]
        if hybi is None:
            orc.run(state)
        else:
            orc.run_eulerian(state, hybi)
        dss_arrays(state.arrays, conn, STATE, tl=st[1], weighting=ASSEMBLE)
    state.ctl[2:5] = ro.rotate(n0, np1, nm1)
    state.dt2, state.consts[1] = dt2, w
    return state
