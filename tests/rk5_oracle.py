"""tests/rk5_oracle.py — TEST INFRASTRUCTURE ONLY.

HOMME's five-stage Runge-Kutta dynamics step (``tstep_type == 5`` of ``prim_advance_exp``, preqx
prim_advance_mod.F90), composed from the single-call oracles of oracle/: the FP64 restatement or the reference
(``rk5_step``) and the extended-precision reference with its error yardstick (``rk5_step_hp``). Both transcribe the
schedule of ``caar_run_rk5`` in include/caar_b200.h literally. With (n0, np1, nm1) the levels on entry, dt the step
and w the handle's eta_ave_w:

    stage  ctl n0  np1  nm1   dt2        eta_ave_w
    1          n0  nm1  n0    dt/5       w/4
    2          nm1 np1  n0    dt/5       0
    3          np1 np1  n0    dt/3       0
    4          np1 np1  n0    (2*dt)/3   0
    c          v, T, dp3d at nm1 = (5*X(nm1) - X(n0))/4 on [nets,nete)
    5          np1 np1  nm1   (3*dt)/4   (3*w)/4

after which the levels rotate as in caar_update_time_levels (np1 <- nm1, nm1 <- n0, n0 <- old np1). The stage
scalars are computed in double precision with exactly these expressions, so that the strict kernel can equal the
FP64 composition bit for bit.

The yardstick of a step, k_rk5
------------------------------
``K = k_rhs(L) = 3L + 24`` bounds the longest chain of dependent roundings of one compute_and_apply_rhs call
(oracle/hp_reference.py), and first order, a call whose inputs are within k u M of exact returns values within
(k + K) u M: each stage adds at most K to the chain of its inputs. With D the chain of the state on entry:
  u1 = stage 1 (u0):                 D + K
  u2, u3, u4 = stages 2-4:           D + 2K, D + 3K, D + 4K
  combination (5 u1 - u0)/4:         D + K + 2   (5*a and the subtraction round; the division by 4 is exact)
  u5 = stage 5 (u4 and the comb.):   D + max(4K, K + 2) + K <= D + 5K + 2
The accumulators (vn0, omega_p, eta_dot_dpdn) take stage 1's and stage 5's contributions, each within K of the
stage's inputs, so they stay inside the same bound. The stage scalars (dt/5, (3*w)/4, ...) are HP inputs combined
as in the table: a product's chain is the longer of its factors' plus one, so their one or two roundings lengthen
no chain. After the rotation the next step starts from u5, so nsteps steps stay within
``k_rk5(L, nsteps) = nsteps * (5 * (3L + 24) + 2)``; max(4K, K + 2) = 4K for every L >= 2, and the 2 are kept so
that the bound does not rest on that comparison.
"""
from __future__ import annotations

import numpy as np

from oracle import hp_reference as hp

COMBINED = ("elem_state_v", "elem_state_T", "elem_state_dp3d")


def k_rk5(nlev, nsteps=1):
    return nsteps * (5 * (3 * nlev + 24) + 2)


def schedule(n0, np1, nm1, dt, w):
    """The step as a list: (n0, np1, nm1, dt2, eta_ave_w) per stage, and "combine" between stages 4 and 5."""
    return [(n0, nm1, n0, dt / 5, w / 4),
            (nm1, np1, n0, dt / 5, 0.0),
            (np1, np1, n0, dt / 3, 0.0),
            (np1, np1, n0, (2 * dt) / 3, 0.0),
            "combine",
            (np1, np1, nm1, (3 * dt) / 4, (3 * w) / 4)]


def rotate(n0, np1, nm1):
    """caar_update_time_levels: -> (n0, np1, nm1) of the next step."""
    return np1, nm1, n0


def rk5_step(orc, state, dt, hybi=None):
    """One step on a harness.State with a single-call oracle (orc.run, or orc.run_eulerian when hybi is given), in
    place. state.ctl's levels come back rotated; state.dt2 and state.consts[1] (eta_ave_w) are restored."""
    n0, np1, nm1 = (int(x) for x in state.ctl[2:5])
    assert len({n0, np1, nm1}) == 3, "caar_run_rk5 needs pairwise distinct time levels"
    dt2, w = state.dt2, float(state.consts[1])
    r = slice(int(state.ctl[0]), int(state.ctl[1]))
    for st in schedule(n0, np1, nm1, float(dt), w):
        if st == "combine":
            for name in COMBINED:
                X = state.arrays[name]
                X[r, nm1] = (5 * X[r, nm1] - X[r, n0]) / 4
            continue
        state.ctl[2:5] = st[:3]
        state.dt2, state.consts[1] = st[3], st[4]
        if hybi is None:
            orc.run(state)
        else:
            orc.run_eulerian(state, hybi)
    state.ctl[2:5] = rotate(n0, np1, nm1)
    state.dt2, state.consts[1] = dt2, w
    return state


def rk5_step_hp(hs, dt, hybi=None):
    """The same step on an hp_reference.HPState, in place; the stage scalars are HP inputs combined as in the
    table. hs's levels come back rotated, its dt2 and eta_ave_w restored."""
    n0, np1, nm1 = hs.n0, hs.np1, hs.nm1
    assert len({n0, np1, nm1}) == 3
    dt2, w = hs.dt2, hs.eta_ave_w
    d = hp.HP.input(dt, hs.dtype)
    zero = hp.HP.input(0.0, hs.dtype)
    r = slice(hs.nets, hs.nete)
    stages = [(n0, nm1, n0, d / 5, w / 4), (nm1, np1, n0, d / 5, zero), (np1, np1, n0, d / 3, zero),
              (np1, np1, n0, (2 * d) / 3, zero), "combine", (np1, np1, nm1, (3 * d) / 4, (3 * w) / 4)]
    for st in stages:
        if st == "combine":
            if hs.nete > hs.nets:
                for name in COMBINED:
                    X = hs.arrays[name]
                    X[r, nm1] = (5.0 * X[r, nm1] - X[r, n0]) / 4.0
            continue
        hs.n0, hs.np1, hs.nm1 = st[:3]
        hs.dt2, hs.eta_ave_w = st[3], st[4]
        hp.rhs(hs, hybi)
    hs.n0, hs.np1, hs.nm1 = rotate(n0, np1, nm1)
    hs.dt2, hs.eta_ave_w = dt2, w
    return hs
