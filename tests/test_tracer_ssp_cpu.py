"""HOMME's three-stage tracer step (caar_advect_tracers) on the CPU: the composition of tests/tracer_ssp_oracle.py is a
second-order integrator, the convergence test has teeth, and the FP64 composition passes the pointwise gate with k_ssp.

The GPU tests compare the kernels against these compositions (tests/test_tracer_ssp_gpu.py), so what is checked here
is the schedule itself: the level each stage reads, dt/2 and the time average."""
import numpy as np
import pytest
import scipy.linalg

from oracle import harness
from oracle import hp_reference as hp
import tracer_ssp_oracle as so
from test_pointwise_cpu import EULER_CASES, case_id, level_local_inputs

E, L, Q = 3, 4, 16
STEPS = (16, 32, 64)


def problem(seed=11):
    """harness.randomize geometry, vstar uniform in +-40 m/s, 16 tracers of random Qdp at level 0."""
    s = harness.randomize(harness.PortOracle().init(E, L, Q), seed=seed)
    rng = np.random.default_rng(seed)
    vstar = rng.uniform(-40.0, 40.0, size=(E, L, 4, 4, 2))
    s.ctl[0:2] = (0, E)
    return s, vstar


def stage_matrices(s, vstar):
    """Per element and level, the 16x16 matrix A of div(vstar q) (q on the 16 GLL points): the tracer step with dt = 1
    on the 16 unit vectors is I - A column by column."""
    b = s.copy()
    Qdp = b.arrays["elem_state_Qdp"]
    Qdp[:, :, 0] = np.eye(16).reshape(16, 1, 4, 4)[None]          # tracer k = unit vector k at every level
    out = np.zeros((E, Q, L, 4, 4))
    harness.PortOracle().euler_step(b, vstar, out, 0, Q, 1.0)
    cols = out.reshape(E, Q, L, 16)                                  # [e][k][l][point]
    return np.eye(16)[None, None] - np.transpose(cols, (0, 2, 3, 1))  # [e][l][point][k]


def exact(s, vstar, t_end):
    A = stage_matrices(s, vstar)
    q0 = s.arrays["elem_state_Qdp"][:, :, 0].reshape(E, Q, L, 16)
    out = np.empty_like(q0)
    for e in range(E):
        for lev in range(L):
            out[e, :, lev] = (scipy.linalg.expm(-t_end * A[e, lev]) @ q0[e, :, lev].T).T
    return out, A


def integrate(s, vstar, nsteps, t_end):
    st = s.copy()
    qn0 = 0
    orc = harness.PortOracle()
    for _ in range(nsteps):
        qn0 = so.ssp_step(orc, st, vstar, qn0, Q, t_end / nsteps)
    return st.arrays["elem_state_Qdp"][:, :, qn0].reshape(E, Q, L, 16)


def observed_orders():
    s, vstar = problem()
    A = stage_matrices(s, vstar)
    t_end = 2.0 / max(np.max(np.abs(np.linalg.eigvals(A[e, lev]))) for e in range(E) for lev in range(L))
    ref, _ = exact(s, vstar, t_end)
    err = [np.max(np.abs(integrate(s, vstar, n, t_end) - ref)) for n in STEPS]
    return [float(np.log2(a / b)) for a, b in zip(err, err[1:])]


def test_stage_matrix_reproduces_the_tracer_step():
    """The matrix the exact solution is built from is the operator the step applies: I - dt A on random Qdp."""
    s, vstar = problem()
    A = stage_matrices(s, vstar)
    out = np.zeros((E, Q, L, 4, 4))
    harness.PortOracle().euler_step(s, vstar, out, 0, Q, 37.0)
    q = s.arrays["elem_state_Qdp"][:, :, 0].reshape(E, Q, L, 16)
    want = q - 37.0 * np.einsum("elpk,eqlk->eqlp", A, q)
    assert hp.rel_err(out.reshape(E, Q, L, 16), want) <= 1e-12


def test_ssp_step_is_second_order():
    """N = 16, 32, 64 steps to T = 2 / (largest |eigenvalue| of the stage operators) against the matrix exponential:
    the order between successive halvings is 2 (stability polynomial 1 + z + z^2/2 + z^3/12)."""
    orders = observed_orders()
    assert all(1.9 <= p <= 2.1 for p in orders), orders


def _defect_half_average(a, b):
    return (a + b) / 2.0


def _defect_stage2_reads_n0(n0, np1):
    return [n0, n0, np1, "average"]


@pytest.mark.parametrize("attr,defect", [("average", _defect_half_average), ("schedule", _defect_stage2_reads_n0)],
                         ids=["average_a_plus_b_over_2", "stage2_reads_n0"])
def test_convergence_test_catches_schedule_defects(attr, defect, monkeypatch):
    """Both defects make the step inconsistent (the z coefficient of its polynomial is 3/4 or 2/3, not 1): the error
    stops shrinking with the step."""
    monkeypatch.setattr(so, attr, defect)
    orders = observed_orders()
    assert not all(1.9 <= p <= 2.1 for p in orders), orders
    assert max(orders) < 0.5, orders


GATE_DT = 150.0
WORST = {}


@pytest.mark.parametrize("c", EULER_CASES, ids=case_id)
def test_fp64_ssp_passes_the_pointwise_gate(c):
    """Two steps of the FP64 composition against the same composition in long double, on the tracer-step inputs of
    tests/test_pointwise_cpu.py (qsize_d 35, elements [1, E-1)): |g - v| <= k_ssp(2) u M at every point of the level
    the second step wrote, and the tracers iq >= qsize and the elements outside the range are untouched."""
    E_, Q_ = 9, 35
    s, vstar, _, _ = level_local_inputs(c["gen"], E_, c["nlev"], c["seed"], qsize_d=Q_)
    s.ctl[0:2] = (1, E_ - 1)
    hs = hp.from_state(s)
    got = s.copy()
    orc = harness.PortOracle()
    q, qh = c["qn0"], c["qn0"]
    for _ in range(2):
        q = so.ssp_step(orc, got, vstar, q, c["qsize"], GATE_DT)
        qh = so.ssp_step_hp(hs, vstar, qh, c["qsize"], GATE_DT)
    assert q == qh == c["qn0"]
    g = got.arrays["elem_state_Qdp"]
    ref = hs.arrays["elem_state_Qdp"]
    r = slice(1, E_ - 1)
    assert np.all(np.isfinite(g[r, :c["qsize"], q]))
    ratio, at, _ = hp.worst(g[r, :c["qsize"], q], ref[r, :c["qsize"], q])
    WORST[c["gen"]] = max(WORST.get(c["gen"], 0.0), ratio)
    assert ratio <= so.k_ssp(2), (ratio, at)
    untouched = np.ones(g.shape, dtype=bool)
    untouched[r, :c["qsize"]] = False
    assert np.array_equal(g[untouched], s.arrays["elem_state_Qdp"][untouched])


def test_k_ssp():
    assert so.k_ssp(1) == 50 and so.k_ssp(3) == 150
    assert so.k_ssp(2) == 2 * (3 * hp.K_EULER + 2)
