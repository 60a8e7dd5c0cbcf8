"""HOMME's five-stage RK step (caar_run_rk5) on the CPU: the composition of tests/rk5_oracle.py is a third-order
integrator, the convergence test has teeth, and the FP64 composition passes the pointwise gate with k_rk5.

The GPU tests compare the kernels against these compositions (tests/test_rk5_gpu.py), so what is checked here is the
schedule itself: stage levels, dt2, eta_ave_w and the combination between stages 4 and 5."""
import numpy as np
import pytest

from oracle import harness
from oracle import hp_reference as hp
import rk5_oracle as ro
from test_pointwise_cpu import make_state

T_END = 5.0          # s; the random state stays smooth well past this (it blows up beyond about 100 s)
STEPS = (2, 4, 8, 16, 32)
N_REF = 512


def integrate(orc, nsteps, t_end, eulerian, E=4, L=16):
    """harness.randomize(seed=3) with spheremp = 1 (the update multiplies by spheremp: with 1 the stages are a
    consistent integrator), levels (0, 1, 2); -> v, T, dp3d at the final n0 (u5 of the last step)."""
    s = harness.randomize(orc.init(E, L), seed=3)
    s.arrays["elem_spheremp"][...] = 1.0
    s.ctl[2:5] = (0, 1, 2)
    hybi = np.linspace(0.0, 1.0, L + 1) if eulerian else None
    for _ in range(nsteps):
        ro.rk5_step(orc, s, t_end / nsteps, hybi)
    n0 = int(s.ctl[2])
    return np.concatenate([s.arrays[n][:, n0].ravel() for n in ro.COMBINED])


def observed_orders(t_end, eulerian):
    orc = harness.PortOracle()
    ref = integrate(orc, N_REF, t_end, eulerian)
    err = [np.max(np.abs(integrate(orc, n, t_end, eulerian) - ref)) for n in STEPS]
    return [float(np.log2(a / b)) for a, b in zip(err, err[1:])]


@pytest.mark.parametrize("eulerian", [False, True], ids=["lagrangian", "eulerian"])
def test_rk5_step_is_third_order(eulerian):
    """N = 2 ... 32 steps to T = 5 s against N = 512: the order between successive halvings is 3 (measured 3.00
    on both branches). A stage 2 that reads u0 instead of u1 keeps third order on this problem: only the bit-exact
    comparison with the strict kernel (tests/test_rk5_gpu.py) catches that one."""
    orders = observed_orders(T_END, eulerian)
    assert all(2.8 <= p <= 3.2 for p in orders), orders


def _defect_stage4_half_dt(n0, np1, nm1, dt, w):
    st = schedule_ok(n0, np1, nm1, dt, w)
    st[3] = st[3][:3] + (dt / 2, st[3][4])
    return st


def _defect_no_combination(n0, np1, nm1, dt, w):
    return [x for x in schedule_ok(n0, np1, nm1, dt, w) if x != "combine"]


schedule_ok = ro.schedule


@pytest.mark.parametrize("defect", [_defect_stage4_half_dt, _defect_no_combination],
                         ids=["stage4_dt_half", "combination_skipped"])
def test_convergence_test_catches_schedule_defects(defect, monkeypatch):
    """At T = 20 s the correct schedule shows order 2.97-3.00 (max-norm error of v, T, dp3d); stage 4 with dt/2 and a
    skipped combination both drop it to about 1."""
    assert all(2.8 <= p <= 3.2 for p in observed_orders(20.0, False))
    monkeypatch.setattr(ro, "schedule", defect)
    orders = observed_orders(20.0, False)
    assert not all(2.8 <= p <= 3.2 for p in orders), orders
    assert max(orders) < 1.5, orders


GATE_CASES = [dict(nlev=L, gen=g, eulerian=e, qn0=q, seed=7000 + i)
              for i, (L, g, e, q) in enumerate((L, g, e, q) for L in (16, 72, 128) for g in ("randomize", "stratified")
                                               for e in (False, True) for q in (-1, 0))]
GATE_DT = 1.0        # s; at 10 s the stratified Eulerian columns and the randomize ones at nlev 128 overflow M
GATE_E = 3


def gate_state(c):
    s = make_state(c["gen"], GATE_E, c["nlev"], c["seed"])
    s.ctl[0:2] = (0, GATE_E)
    s.ctl[2:5] = (0, 1, 2)
    s.ctl[5] = c["qn0"]
    hybi = np.linspace(0.0, 1.0, c["nlev"] + 1) ** 1.5 if c["eulerian"] else None
    return s, hybi


WORST = {}


@pytest.mark.parametrize("c", GATE_CASES, ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items() if k != "seed"))
def test_fp64_rk5_passes_the_pointwise_gate(c):
    """Two steps of the FP64 composition against the same composition in long double: |g - v| <= k_rk5 u M at every
    point of the seven mutated arrays (k_rk5(72, 2) = 2404; the worst ratio is about 3), and the rotated levels
    agree."""
    s, hybi = gate_state(c)
    hs = hp.from_state(s)
    got = s.copy()
    orc = harness.PortOracle()
    for _ in range(2):
        ro.rk5_step(orc, got, GATE_DT, hybi)
        ro.rk5_step_hp(hs, GATE_DT, hybi)
    assert (hs.n0, hs.np1, hs.nm1) == tuple(int(x) for x in got.ctl[2:5]) == (2, 0, 1)
    assert got.dt2 == s.dt2 and got.consts[1] == s.consts[1]
    K = ro.k_rk5(c["nlev"], 2)
    for n in harness.MUTATED:
        g = got.arrays[n]
        assert np.all(np.isfinite(g)), n
        r, at, _ = hp.worst(g, hs.arrays[n])
        WORST[n] = max(WORST.get(n, 0.0), r)
        assert r <= K, (n, r, at, K)


def test_k_rk5():
    assert ro.k_rk5(72, 2) == 2404 and ro.k_rk5(16, 2) == 724
    assert ro.k_rk5(30, 3) == 3 * (5 * hp.k_rhs(30) + 2)
