"""tests/tracer_ssp_oracle.py — TEST INFRASTRUCTURE ONLY.

HOMME's three-stage tracer step (Eulerian advection with ``rkstage = 3`` in prim_advection_mod: three euler_step
calls and qdp_time_avg), composed from the single-call tracer oracles of oracle/: the FP64 restatement
(``ssp_step``, PortOracle.euler_step) and the extended-precision reference with its error yardstick (``ssp_step_hp``,
hp_reference.euler_step). Both transcribe the schedule of ``caar_advect_tracers`` in include/caar_b200.h literally.
With n0 = qn0 on entry and np1 = 1 - n0, for tracers iq < qsize of elements [nets,nete):

    1  Qdp(np1) = Qdp(n0)  - dt/2 div(vstar Qdp(n0))
    2  Qdp(np1) = Qdp(np1) - dt/2 div(vstar Qdp(np1))
    3  Qdp(np1) = Qdp(np1) - dt/2 div(vstar Qdp(np1))
    a  Qdp(np1) = (Qdp(n0) + 2 Qdp(np1)) / 3

after which qn0 becomes np1. dt/2 is exact in double, so the stage scalar is the same on every side.

The yardstick of a step, k_ssp
------------------------------
``K_EULER = 16`` bounds the longest chain of dependent roundings of one tracer step (oracle/hp_reference.py), and
first order, a step whose input is within k u M of exact returns values within (k + K_EULER) u M: each stage adds at
most K_EULER to the chain of its input. With D the chain of Qdp on entry:
  stage 1, 2, 3:                   D + 16, D + 32, D + 48
  average (a + 2 b) / 3:           2 b is exact; the add and the division round once each: D + 48 + 2
After the swap the next step starts from the average, so nsteps steps stay within
``k_ssp(nsteps) = nsteps * (3 * K_EULER + 2) = 50 * nsteps``.
"""
from __future__ import annotations

import numpy as np

from oracle import hp_reference as hp

K_STEP = 3 * hp.K_EULER + 2


def k_ssp(nsteps=1):
    return nsteps * K_STEP


def schedule(n0, np1):
    """The step as a list: the Qdp level each stage reads (it writes np1), then "average"."""
    return [n0, np1, np1, "average"]


def average(a, b):
    """qdp_time_avg: (Qdp(n0) + 2 Qdp(np1)) / 3, rounded as the Fortran expression (numpy float64: no contraction)."""
    return (a + 2.0 * b) / 3.0


def ssp_step(orc, state, vstar, qn0, qsize, dt):
    """One step on a harness.State with PortOracle.euler_step, in place on state.arrays["elem_state_Qdp"] over
    [ctl[0], ctl[1]) -> the new qn0."""
    n0, np1 = int(qn0), 1 - int(qn0)
    r = slice(int(state.ctl[0]), int(state.ctl[1]))
    Q = state.arrays["elem_state_Qdp"]
    if r.stop <= r.start or qsize <= 0:
        return np1
    out = np.zeros((state.nelem, state.qsize_d, state.nlev, 4, 4))
    for st in schedule(n0, np1):
        if st == "average":
            Q[r, :qsize, np1] = average(Q[r, :qsize, n0], Q[r, :qsize, np1])
            continue
        orc.euler_step(state, vstar, out, st, qsize, dt / 2)
        Q[r, :qsize, np1] = out[r, :qsize]
    return np1


def ssp_step_hp(hs, vstar, qn0, qsize, dt):
    """The same step on an hp_reference.HPState, in place on hs.arrays["elem_state_Qdp"] (an HP) -> the new qn0."""
    n0, np1 = int(qn0), 1 - int(qn0)
    r = slice(hs.nets, hs.nete)
    Q = hs.arrays["elem_state_Qdp"]
    if hs.nete <= hs.nets or qsize <= 0:
        return np1
    for st in schedule(n0, np1):
        if st == "average":
            Q[r, :qsize, np1] = (Q[r, :qsize, n0] + 2.0 * Q[r, :qsize, np1]) / 3.0
            continue
        out = hp.euler_step(hs, vstar, st, qsize, dt / 2)
        Q[r, :qsize, np1] = out[r, :qsize]
    return np1
