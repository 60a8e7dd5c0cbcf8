"""tests/remap_oracle.py — TEST INFRASTRUCTURE ONLY.

HOMME's vertical remap for ``rsplit > 0`` (``vertical_remap`` with ``remap1`` = ``remap_Q_ppm`` and
``vert_remap_q_alg = 1``: PPM with mirrored ghost cells), as specified in include/caar_b200.h
(``caar_vertical_remap``). The header's restatement is the contract; this file transcribes it twice:

  * ``remap_column``: a literal scalar transcription on Python floats (IEEE double, every operation rounded
    separately), in HOMME's 1-based indices, loop for loop;
  * ``remap_np``: numpy, vectorised over columns (and over levels wherever the restatement has no sum), sequential in
    k wherever it sums. No ``np.sum`` / ``np.cumsum``: the sums are written out.

``vertical_remap`` applies the numpy transcription to handle-shaped arrays, as the C-API call does. ``coordinate``
and ``columns`` build the tests' inputs: a hybrid coordinate with positive layers, and source thicknesses in three
deformation regimes (none, under one cell, over one cell).

``remap_np`` also takes ``defect``: one of ``DEFECTS``, each a deliberately wrong remap that the CPU tests must tell
from the scalar transcription (a ghost mirror of dp_star shifted by one cell at the top, no pin(nlev+1) = pio(nlev+1) override,
no reset of the edge values at a local extremum).
"""
from __future__ import annotations

import math

import numpy as np

OFF = 2                                   # index of level i in the ghosted lists / arrays is i + OFF (i >= -1)
DEFECTS = ("ghost", "top", "no_extremum")
REGIMES = ("identity", "under", "over")


# ---- scalar transcription -------------------------------------------------------------------------------------------

def _ghosted(x, L):
    """x (L floats, C level k-1 = Fortran level k) -> list g with g[i + OFF] = x(i) for i = -1..L+2, mirrored."""
    g = [0.0] * (L + OFF + 3)
    for i in range(1, L + 1):
        g[i + OFF] = float(x[i - 1])
    for i in (1, 2):
        g[1 - i + OFF] = g[i + OFF]
        g[L + i + OFF] = g[L + 1 - i + OFF]
    return g


def _min3(a, b, c):
    m = a
    if b < m:
        m = b
    if c < m:
        m = c
    return m


def remap_column(dpo, dpn, fields):
    """One column: dpo (dp_star) and dpn (dp) are L floats, fields a list of L-float lists (the values to remap) ->
    list of the remapped fields. Literal restatement of include/caar_b200.h."""
    L = len(dpo)
    pio = [0.0] * (L + 3)                 # pio[i], i = 1..L+2
    pin = [0.0] * (L + 2)                 # pin[i], i = 1..L+1
    for k in range(1, L + 1):
        pio[k + 1] = pio[k] + dpo[k - 1]
        pin[k + 1] = pin[k] + dpn[k - 1]
    pio[L + 2] = pio[L + 1] + 1.0
    pin[L + 1] = pio[L + 1]
    dx = _ghosted(dpo, L)
    kid, z2 = [0] * (L + 1), [0.0] * (L + 1)
    for k in range(1, L + 1):
        kk = k
        while pio[kk] <= pin[k + 1]:
            kk = kk + 1
            if kk == L + 2:
                break
        kk = kk - 1
        if kk == L + 1:
            kk = L
        kk = min(max(kk, 1), L)           # no effect inside the contract (dpo > 0, dpn > 0)
        kid[k] = kk
        z2[k] = (pin[k + 1] - (pio[kk] + pio[kk + 1]) * 0.5) / dx[kk + OFF]
    D = lambda j: dx[j + OFF]
    r = [[0.0] * (L + 2) for _ in range(11)]   # r[n][j], n = 1..10, j = 0..L+1
    for j in range(0, L + 2):
        r[1][j] = D(j) / ((D(j - 1) + D(j)) + D(j + 1))
        r[2][j] = (2.0 * D(j - 1) + D(j)) / (D(j + 1) + D(j))
        r[3][j] = (D(j) + 2.0 * D(j + 1)) / (D(j - 1) + D(j))
    for j in range(0, L + 1):
        r[4][j] = D(j) / (D(j) + D(j + 1))
        r[5][j] = 1.0 / (((D(j - 1) + D(j)) + D(j + 1)) + D(j + 2))
        r[6][j] = ((2.0 * D(j + 1)) * D(j)) / (D(j) + D(j + 1))
        r[7][j] = (D(j - 1) + D(j)) / (2.0 * D(j) + D(j + 1))
        r[8][j] = (D(j + 2) + D(j + 1)) / (2.0 * D(j + 1) + D(j))
        r[9][j] = (D(j) * (D(j - 1) + D(j))) / (2.0 * D(j) + D(j + 1))
        r[10][j] = (D(j + 1) * (D(j + 1) + D(j + 2))) / (D(j) + 2.0 * D(j + 1))
    out = []
    for f in fields:
        masso = [0.0] * (L + 2)
        ao = [0.0] * L
        for k in range(1, L + 1):
            masso[k + 1] = masso[k] + f[k - 1]
            ao[k - 1] = f[k - 1] / dpo[k - 1]
        ag = _ghosted(ao, L)
        a = lambda j: ag[j + OFF]
        dma = [0.0] * (L + 2)
        for j in range(0, L + 2):
            da = r[1][j] * (r[2][j] * (a(j + 1) - a(j)) + r[3][j] * (a(j) - a(j - 1)))
            dma[j] = _min3(abs(da), 2.0 * abs(a(j) - a(j - 1)), 2.0 * abs(a(j + 1) - a(j))) * math.copysign(1.0, da)
            if (a(j + 1) - a(j)) * (a(j) - a(j - 1)) <= 0.0:
                dma[j] = 0.0
        ai = [0.0] * (L + 1)
        for j in range(0, L + 1):
            ai[j] = (a(j) + r[4][j] * (a(j + 1) - a(j))) + r[5][j] * (
                ((r[6][j] * (r[7][j] - r[8][j])) * (a(j + 1) - a(j)) - r[9][j] * dma[j + 1]) + r[10][j] * dma[j])
        c0, c1, c2 = [0.0] * (L + 1), [0.0] * (L + 1), [0.0] * (L + 1)
        for j in range(1, L + 1):
            al, ar, aj = ai[j - 1], ai[j], a(j)
            if (ar - aj) * (aj - al) <= 0.0:
                al, ar = aj, aj
            if (ar - al) * (aj - (al + ar) / 2.0) > ((ar - al) * (ar - al)) / 6.0:
                al = 3.0 * aj - 2.0 * ar
            if (ar - al) * (aj - (al + ar) / 2.0) < -(((ar - al) * (ar - al)) / 6.0):
                ar = 3.0 * aj - 2.0 * al
            c0[j] = 1.5 * aj - (al + ar) / 4.0
            c1[j] = ar - al
            c2[j] = -6.0 * aj + 3.0 * (al + ar)
        new = [0.0] * L
        massn1 = 0.0
        for k in range(1, L + 1):
            kk, x2, x1 = kid[k], z2[k], -0.5
            integral = (c0[kk] * (x2 - x1) + (c1[kk] * (x2 * x2 - x1 * x1)) / 2.0) + (
                c2[kk] * ((x2 * x2) * x2 - (x1 * x1) * x1)) / 3.0
            massn2 = masso[kk] + integral * dx[kk + OFF]
            new[k - 1] = massn2 - massn1
            massn1 = massn2
        out.append(new)
    return out


# ---- numpy transcription --------------------------------------------------------------------------------------------

def _ghosted_np(x, defect=None):
    """x (N, L) -> (N, L + OFF + 3) with column i + OFF holding level i = -1..L+2, mirrored."""
    N, L = x.shape
    g = np.zeros((N, L + OFF + 3))
    g[:, 1 + OFF:L + 1 + OFF] = x
    for i in (1, 2):
        g[:, 1 - i + OFF] = g[:, i + OFF]
        src = L - i if defect == "ghost" else L + 1 - i    # the defect mirrors dp_star through the centre of cell L
        g[:, L + i + OFF] = g[:, src + OFF]
    return g


def grid_np(dpo, dpn, defect=None):
    """The grid terms of a set of columns: dict(kid (N, L+1) int, z2 (N, L+1), r (11, N, L+2), dx ghosted)."""
    N, L = dpo.shape
    pio, pin = np.zeros((N, L + 3)), np.zeros((N, L + 2))
    for k in range(1, L + 1):
        pio[:, k + 1] = pio[:, k] + dpo[:, k - 1]
        pin[:, k + 1] = pin[:, k] + dpn[:, k - 1]
    pio[:, L + 2] = pio[:, L + 1] + 1.0
    if defect != "top":
        pin[:, L + 1] = pio[:, L + 1]
    dx = _ghosted_np(dpo, defect)
    rows = np.arange(N)
    kid, z2 = np.zeros((N, L + 1), np.int64), np.zeros((N, L + 1))
    for k in range(1, L + 1):
        kk = np.full(N, k)
        run = np.ones(N, bool)
        while run.any():
            step = run & (pio[rows, kk] <= pin[:, k + 1])
            kk = np.where(step, kk + 1, kk)
            run = step & (kk != L + 2)
        kk = kk - 1
        kk = np.where(kk == L + 1, L, kk)
        kk = np.clip(kk, 1, L)
        kid[:, k] = kk
        z2[:, k] = (pin[:, k + 1] - (pio[rows, kk] + pio[rows, kk + 1]) * 0.5) / dx[rows, kk + OFF]
    D = lambda j0, j1: dx[:, j0 + OFF:j1 + OFF]      # levels j0 .. j1-1
    r = np.zeros((11, N, L + 2))
    J = L + 2                                       # j = 0..L+1
    dm, d0, dp = D(-1, J - 1), D(0, J), D(1, J + 1)
    r[1] = d0 / ((dm + d0) + dp)
    r[2] = (2.0 * dm + d0) / (dp + d0)
    r[3] = (d0 + 2.0 * dp) / (dm + d0)
    J = L + 1                                       # j = 0..L
    dm, d0, dp, dpp = D(-1, J - 1), D(0, J), D(1, J + 1), D(2, J + 2)
    r[4, :, :J] = d0 / (d0 + dp)
    r[5, :, :J] = 1.0 / (((dm + d0) + dp) + dpp)
    r[6, :, :J] = ((2.0 * dp) * d0) / (d0 + dp)
    r[7, :, :J] = (dm + d0) / (2.0 * d0 + dp)
    r[8, :, :J] = (dpp + dp) / (2.0 * dp + d0)
    r[9, :, :J] = (d0 * (dm + d0)) / (2.0 * d0 + dp)
    r[10, :, :J] = (dp * (dp + dpp)) / (d0 + 2.0 * dp)
    return dict(kid=kid, z2=z2, r=r, dx=dx)


def remap_field_np(g, dpo, f, defect=None):
    """One field of every column: f (N, L) the values to remap -> (N, L) the remapped values."""
    N, L = f.shape
    r, dx, kid, z2 = g["r"], g["dx"], g["kid"], g["z2"]
    masso = np.zeros((N, L + 2))
    for k in range(1, L + 1):
        masso[:, k + 1] = masso[:, k] + f[:, k - 1]
    ag = _ghosted_np(f / dpo)
    A = lambda j0, j1: ag[:, j0 + OFF:j1 + OFF]
    J = L + 2
    am, a0, ap = A(-1, J - 1), A(0, J), A(1, J + 1)
    da = r[1] * (r[2] * (ap - a0) + r[3] * (a0 - am))
    m = np.abs(da)
    b = 2.0 * np.abs(a0 - am)
    m = np.where(b < m, b, m)
    c = 2.0 * np.abs(ap - a0)
    m = np.where(c < m, c, m)
    dma = m * np.copysign(1.0, da)
    dma = np.where((ap - a0) * (a0 - am) <= 0.0, 0.0, dma)
    J = L + 1
    a0, ap = A(0, J), A(1, J + 1)
    R = lambda n: r[n, :, :J]
    ai = (a0 + R(4) * (ap - a0)) + R(5) * (((R(6) * (R(7) - R(8))) * (ap - a0) - R(9) * dma[:, 1:J + 1]) + R(10) * dma[:, :J])
    al, ar, aj = ai[:, :L].copy(), ai[:, 1:L + 1].copy(), A(1, L + 1)
    flat = (ar - aj) * (aj - al) <= 0.0
    if defect != "no_extremum":
        al, ar = np.where(flat, aj, al), np.where(flat, aj, ar)
    hi = (ar - al) * (aj - (al + ar) / 2.0) > ((ar - al) * (ar - al)) / 6.0
    al = np.where(hi, 3.0 * aj - 2.0 * ar, al)
    lo = (ar - al) * (aj - (al + ar) / 2.0) < -(((ar - al) * (ar - al)) / 6.0)
    ar = np.where(lo, 3.0 * aj - 2.0 * al, ar)
    c0 = np.zeros((N, L + 1))
    c1, c2 = c0.copy(), c0.copy()
    c0[:, 1:] = 1.5 * aj - (al + ar) / 4.0
    c1[:, 1:] = ar - al
    c2[:, 1:] = -6.0 * aj + 3.0 * (al + ar)
    rows = np.arange(N)[:, None]
    kk, x2, x1 = kid[:, 1:], z2[:, 1:], -0.5
    integral = (c0[rows, kk] * (x2 - x1) + (c1[rows, kk] * (x2 * x2 - x1 * x1)) / 2.0) + (
        c2[rows, kk] * ((x2 * x2) * x2 - (x1 * x1) * x1)) / 3.0
    massn = masso[rows, kk] + integral * dx[rows, kk + OFF]
    out = np.empty((N, L))
    out[:, 0] = massn[:, 0]
    out[:, 1:] = massn[:, 1:] - massn[:, :-1]
    return out


def remap_np(dpo, dpn, fields, defect=None):
    """remap_column on N columns at once: dpo, dpn (N, L), fields a list of (N, L) arrays -> list of (N, L) arrays."""
    assert defect in (None,) + DEFECTS, defect
    dpo, dpn = np.asarray(dpo, np.float64), np.asarray(dpn, np.float64)
    g = grid_np(dpo, dpn, defect)
    return [remap_field_np(g, dpo, np.asarray(f, np.float64), defect) for f in fields]


# ---- the target thicknesses and the call on handle-shaped arrays ----------------------------------------------------

def target_dp(dpo, hyai, hybi, ps0):
    """dp (N, L) of columns with source thicknesses dpo (N, L): ps = hyai[0]*ps0 + S, S the sequential sum of dpo."""
    N, L = dpo.shape
    S = np.zeros(N)
    for k in range(L):
        S = S + dpo[:, k]
    ps = hyai[0] * ps0 + S
    return (np.diff(hyai)[None, :] * ps0) + (np.diff(hybi)[None, :] * ps[:, None])


def vertical_remap(A, hyai, hybi, ps0, nets, nete, tl, qtl, qsize, defect=None):
    """caar_vertical_remap in place on a dict of handle-shaped arrays (elem_state_dp3d, elem_state_v, elem_state_T,
    elem_state_Qdp) -> None."""
    if nete <= nets:
        return
    dp3d, v, T, Q = A["elem_state_dp3d"], A["elem_state_v"], A["elem_state_T"], A["elem_state_Qdp"]
    E, L = nete - nets, dp3d.shape[2]
    cols = lambda x: np.ascontiguousarray(np.moveaxis(x.reshape(E, L, 16), 1, 2)).reshape(E * 16, L)
    back = lambda y: np.moveaxis(y.reshape(E, 16, L), 2, 1).reshape(E, L, 4, 4)
    dpo = cols(dp3d[nets:nete, tl])
    dpn = target_dp(dpo, np.asarray(hyai, np.float64), np.asarray(hybi, np.float64), ps0)
    fields = [cols(T[nets:nete, tl]) * dpo, cols(v[nets:nete, tl, ..., 0]) * dpo, cols(v[nets:nete, tl, ..., 1]) * dpo]
    fields += [cols(Q[nets:nete, iq, qtl]) for iq in range(qsize)]
    out = remap_np(dpo, dpn, fields, defect)
    T[nets:nete, tl] = back(out[0] / dpn)
    v[nets:nete, tl, ..., 0] = back(out[1] / dpn)
    v[nets:nete, tl, ..., 1] = back(out[2] / dpn)
    for iq in range(qsize):
        Q[nets:nete, iq, qtl] = back(out[3 + iq])
    dp3d[nets:nete, tl] = back(dpn)


# ---- inputs ---------------------------------------------------------------------------------------------------------

PS0 = 1.0e5


def coordinate(L):
    """(hyai, hybi) [L+1] of a hybrid coordinate with positive layers: hyai[L] = 0, hybi[0] = 0, hybi[L] = 1, a model
    top at 2 hPa and layers that thicken downwards."""
    s = np.linspace(0.0, 1.0, L + 1)
    s = 0.6 * s + 0.4 * s * s                       # stretched, strictly increasing from 0 to 1
    eta = 0.002 + 0.998 * s
    hybi = s ** 3
    hybi[0], hybi[-1] = 0.0, 1.0
    hyai = eta - hybi
    hyai[-1] = 0.0
    return hyai, hybi


def columns(N, L, regime, seed):
    """dp_star (N, L) for the regime: "identity" the target of a surface pressure near PS0 (so dp_star == dp to
    rounding), "under" interfaces moved by under half of the thinner adjacent layer (a deformation under one cell),
    "over" interfaces moved by a smooth warp of up to a quarter of the column (many cells; the kid = k-1 path)."""
    rng = np.random.default_rng(seed)
    hyai, hybi = coordinate(L)
    ps = PS0 * rng.uniform(0.95, 1.03, N)
    dp = np.diff(hyai)[None, :] * PS0 + np.diff(hybi)[None, :] * ps[:, None]
    if regime == "identity":
        return dp
    pint = np.zeros((N, L + 1))
    for k in range(L):
        pint[:, k + 1] = pint[:, k] + dp[:, k]
    if regime == "under":
        thin = np.minimum(dp[:, :-1], dp[:, 1:])
        moved = pint.copy()
        moved[:, 1:L] += rng.uniform(-0.45, 0.45, (N, L - 1)) * thin
    else:
        P = pint[:, L:]
        s = pint / P
        alpha = rng.uniform(0.5, 0.9, (N, 1)) * np.where(np.arange(N) % 2 == 0, 1.0, -1.0)[:, None]   # w(s) = s + alpha sin(pi s)/pi
        moved = P * (s + alpha * np.sin(np.pi * s) / np.pi)                     # is increasing for |alpha| < 1
        moved[:, 0], moved[:, L] = 0.0, pint[:, L]
    return np.diff(moved, axis=1)


def mixing_ratios(N, L, seed):
    """Smooth profiles with noise, extrema and a flat stretch: a test for the limiter branches of the PPM edges."""
    rng = np.random.default_rng(seed)
    z = np.linspace(0.0, 1.0, L)[None, :]
    q = 1e-3 * (1.0 + np.sin(rng.uniform(2, 12, (N, 1)) * z + rng.uniform(0, 6, (N, 1))))
    q *= 10.0 ** rng.uniform(-3, 0, (N, 1))
    q += rng.uniform(0, 1e-4, (N, L)) * q.max(1, keepdims=True) * (rng.uniform(size=(N, 1)) < 0.5)
    q[:, L // 3:L // 3 + max(1, L // 8)] = q[:, L // 3:L // 3 + 1]
    return q
