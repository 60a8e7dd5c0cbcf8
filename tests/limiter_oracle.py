"""tests/limiter_oracle.py — TEST INFRASTRUCTURE ONLY.

HOMME's quasi-monotone tracer limiter (euler_step with ``limiter_option == 8``): the element-local bounds and
``limiter_optim_iter_full``, as specified in include/caar_b200.h (``caar_tracer_bounds``, ``caar_limit_tracers``).
The header's text is the contract; this file transcribes it twice:

  * ``bounds_problem`` / ``limit_problem``: literal scalar transcriptions, loop for loop, on Python floats (IEEE
    double, every operation rounded separately);
  * ``bounds_np`` / ``limit_np``: numpy, vectorised over problems but sequential over the points and the iterations,
    with a per-problem active mask. No ``np.sum``: its pairwise summation would change the bits.

Points are given in the C order of the pointers_only layout (offset 4*igp + jgp); both transcriptions visit them in
Fortran sequence-association order (``FORTRAN``: i = igp fastest). ``tracer_bounds`` and ``limit_tracers`` apply the
numpy transcription to whole handle-shaped arrays, as the two C-API calls do.

``limit_np`` also takes ``defect``: one of ``DEFECTS``, each a deliberately wrong limiter that the CPU tests must
catch (redistributing onto saturated points, no relaxation, the exit test before the clip, sums in C order).
"""
from __future__ import annotations

import numpy as np

TOL = 5e-14
MAXITER = 15
FORTRAN = [4 * (m % 4) + m // 4 for m in range(16)]   # C offset of the m-th point in Fortran order
C_ORDER = list(range(16))
DEFECTS = ("saturated", "no_relax", "exit_first", "c_order")
EXIT_NONE, EXIT_TOL, EXIT_WS0, EXIT_MAXITER = 0, 1, 2, 3   # EXIT_NONE: sumc <= 0, not limited


# ---- scalar transcriptions ------------------------------------------------------------------------------------------

def bounds_problem(p, d):
    """(qmin, qmax) of one problem: p, d are 16 floats in C order."""
    x = [p[o] / d[o] for o in FORTRAN]
    qmin = qmax = x[0]
    for n in range(1, 16):
        if x[n] < qmin:
            qmin = x[n]
        if x[n] > qmax:
            qmax = x[n]
    if qmin < 0.0:
        qmin = 0.0
    return qmin, qmax


def limit_problem(p, d, w, minp, maxp):
    """limiter_optim_iter_full on one problem -> (p_new, minp, maxp, x, iterations, exit kind); p, d, w are 16 floats
    in C order, p_new and x are returned in C order."""
    p = [float(v) for v in p]
    c = [0.0] * 16
    x = [0.0] * 16
    for n, o in enumerate(FORTRAN):
        c[n] = w[o] * d[o]
        x[n] = p[o] / d[o]
    sumc = 0.0
    for n in range(16):
        sumc = sumc + c[n]
    if sumc <= 0.0:
        return p, minp, maxp, [p[o] / d[o] for o in C_ORDER], 0, EXIT_NONE
    mass = 0.0
    for n in range(16):
        mass = mass + c[n] * x[n]
    if mass < minp * sumc:
        minp = mass / sumc
    if mass > maxp * sumc:
        maxp = mass / sumc
    iters, kind = 0, EXIT_MAXITER
    for _ in range(MAXITER):
        iters += 1
        addmass = 0.0
        for n in range(16):
            if x[n] > maxp:
                addmass = addmass + (x[n] - maxp) * c[n]
                x[n] = maxp
            if x[n] < minp:
                addmass = addmass - (minp - x[n]) * c[n]
                x[n] = minp
        if abs(addmass) <= TOL * abs(mass):
            kind = EXIT_TOL
            break
        ws = 0.0
        if addmass > 0.0:
            for n in range(16):
                if x[n] < maxp:
                    ws = ws + c[n]
            if ws == 0.0:
                kind = EXIT_WS0
                break
            for n in range(16):
                if x[n] < maxp:
                    x[n] = x[n] + addmass / ws
        else:
            for n in range(16):
                if x[n] > minp:
                    ws = ws + c[n]
            if ws == 0.0:
                kind = EXIT_WS0
                break
            for n in range(16):
                if x[n] > minp:
                    x[n] = x[n] + addmass / ws
    out = list(p)
    xc = [0.0] * 16
    for n, o in enumerate(FORTRAN):
        out[o] = x[n] * d[o]
        xc[o] = x[n]
    return out, minp, maxp, xc, iters, kind


# ---- numpy transcriptions -------------------------------------------------------------------------------------------

def bounds_np(p, d):
    """(qmin, qmax) arrays of N problems: p, d are (N, 16) in C order."""
    p, d = np.asarray(p, np.float64), np.asarray(d, np.float64)
    with np.errstate(all="ignore"):
        x = p[:, FORTRAN] / d[:, FORTRAN]
    qmin, qmax = x[:, 0].copy(), x[:, 0].copy()
    for n in range(1, 16):
        qmin = np.where(x[:, n] < qmin, x[:, n], qmin)
        qmax = np.where(x[:, n] > qmax, x[:, n], qmax)
    qmin = np.where(qmin < 0.0, 0.0, qmin)
    return qmin, qmax


def limit_np(p, d, w, minp, maxp, defect=None):
    """limiter_optim_iter_full on N problems -> dict(p, minp, maxp, x, iters, exit): p, d, w are (N, 16) in C order,
    minp, maxp (N,); the outputs p and x are (N, 16) in C order, iters the loop passes and exit the EXIT_* kind."""
    assert defect in (None,) + DEFECTS, defect
    p, d, w = (np.asarray(a, np.float64) for a in (p, d, w))
    order = C_ORDER if defect == "c_order" else FORTRAN
    N = p.shape[0]
    with np.errstate(all="ignore"):
        c = w[:, order] * d[:, order]
        x = p[:, order] / d[:, order]
        sumc = np.zeros(N)
        for n in range(16):
            sumc = sumc + c[:, n]
        act = ~(sumc <= 0.0)
        mass = np.zeros(N)
        for n in range(16):
            mass = mass + c[:, n] * x[:, n]
        minp = np.asarray(minp, np.float64).copy()
        maxp = np.asarray(maxp, np.float64).copy()
        if defect != "no_relax":
            minp = np.where(act & (mass < minp * sumc), mass / sumc, minp)
            maxp = np.where(act & (mass > maxp * sumc), mass / sumc, maxp)
        tol = TOL * np.abs(mass)
        iters = np.zeros(N, np.int64)
        kind = np.where(act, EXIT_MAXITER, EXIT_NONE)
        run = act.copy()
        addmass = np.zeros(N)
        for _ in range(MAXITER):
            if not run.any():
                break
            iters += run
            if defect == "exit_first":   # tests the previous pass's addmass (0 on the first) before clipping
                done = run & (np.abs(addmass) <= tol)
                kind = np.where(done, EXIT_TOL, kind)
                run = run & ~done
            addmass = np.zeros(N)
            for n in range(16):
                xn = x[:, n]
                over = run & (xn > maxp)
                addmass = np.where(over, addmass + (xn - maxp) * c[:, n], addmass)
                xn = np.where(over, maxp, xn)
                under = run & (xn < minp)
                addmass = np.where(under, addmass - (minp - xn) * c[:, n], addmass)
                x[:, n] = np.where(under, minp, xn)
            if defect != "exit_first":
                done = run & (np.abs(addmass) <= tol)
                kind = np.where(done, EXIT_TOL, kind)
                run = run & ~done
            up = addmass > 0.0
            ws = np.zeros(N)
            sel = np.zeros((N, 16), bool)
            for n in range(16):
                sel[:, n] = run & (np.where(up, x[:, n] < maxp, x[:, n] > minp) | (defect == "saturated"))
                ws = np.where(sel[:, n], ws + c[:, n], ws)
            zero = run & (ws == 0.0)
            kind = np.where(zero, EXIT_WS0, kind)
            run = run & ~zero
            inc = addmass / ws
            for n in range(16):
                x[:, n] = np.where(run & sel[:, n], x[:, n] + inc, x[:, n])
        pn = p.copy()
        xc = p / d
        newp = x * d[:, order]
        pn[:, order] = np.where(act[:, None], newp, p[:, order])
        xc[:, order] = np.where(act[:, None], x, xc[:, order])
    return dict(p=pn, minp=minp, maxp=maxp, x=xc, iters=iters, exit=kind)


# ---- the two calls on handle-shaped arrays --------------------------------------------------------------------------

def _problems(Qdp, dp3d, nets, nete, qtl, qsize, dp_tl):
    """(p, d) as (N, 16) over problems (e, iq, k) of [nets,nete) x [0,qsize) x [0,L), in that order."""
    ne, L = nete - nets, Qdp.shape[3]
    p = Qdp[nets:nete, :qsize, qtl].reshape(ne * qsize * L, 16)
    d = np.broadcast_to(dp3d[nets:nete, dp_tl].reshape(ne, 1, L, 16), (ne, qsize, L, 16)).reshape(-1, 16)
    return p, d


def tracer_bounds(Qdp, dp3d, bounds, nets, nete, qtl, qsize, dp_tl):
    """caar_tracer_bounds in place on bounds [E][qsize_d][L][2]."""
    if nete <= nets or qsize <= 0:
        return
    p, d = _problems(Qdp, dp3d, nets, nete, qtl, qsize, dp_tl)
    qmin, qmax = bounds_np(p, d)
    shape = bounds[nets:nete, :qsize].shape[:-1]
    bounds[nets:nete, :qsize, :, 0] = qmin.reshape(shape)
    bounds[nets:nete, :qsize, :, 1] = qmax.reshape(shape)


def limit_tracers(Qdp, dp3d, spheremp, bounds, nets, nete, qtl, qsize, dp_tl, defect=None):
    """caar_limit_tracers in place on Qdp [E][qsize_d][2][L][4][4] and bounds -> limit_np's dict (iters, exit)."""
    if nete <= nets or qsize <= 0:
        return None
    ne, L = nete - nets, Qdp.shape[3]
    p, d = _problems(Qdp, dp3d, nets, nete, qtl, qsize, dp_tl)
    w = np.broadcast_to(spheremp[nets:nete].reshape(ne, 1, 1, 16), (ne, qsize, L, 16)).reshape(-1, 16)
    b = bounds[nets:nete, :qsize].reshape(-1, 2)
    r = limit_np(p, d, w, b[:, 0], b[:, 1], defect=defect)
    Qdp[nets:nete, :qsize, qtl] = r["p"].reshape(ne, qsize, L, 4, 4)
    shape = bounds[nets:nete, :qsize].shape[:-1]
    bounds[nets:nete, :qsize, :, 0] = r["minp"].reshape(shape)
    bounds[nets:nete, :qsize, :, 1] = r["maxp"].reshape(shape)
    return r
