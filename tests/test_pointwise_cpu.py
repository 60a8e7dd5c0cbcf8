"""The pointwise yardstick on the CPU: the extended-precision reference (oracle/hp_reference.py) against the FP64
restatement, and proof that its per-point gate |g - v| <= K u M catches what the field-normalised gate cannot.

The inputs come from two generators: harness.randomize (every field within about one order of magnitude of its
maximum) and ``stratified`` below (realistic columns: pressure from 10 Pa to about 1e5 Pa, dp3d over three orders of
magnitude, tracer mass over seven), on which a field-normalised 1e-12 accepts a 1e-5 relative error at the top of the
column. The case matrices here are also the ones tests/test_pointwise_gpu.py runs on the GPU."""
import numpy as np
import pytest

from oracle import harness
from oracle import hp_reference as hp

TOL = 1e-12          # the field-normalised gate of the parity tests


# ---- inputs ---------------------------------------------------------------------------------------------------------

def stratified(s, seed):
    """Realistic columns on the geometry of harness.randomize (|det D| >= 1/64, physical rrearth): ps0 = 1e5 with
    hyai[0]*ps0 = 10 Pa; dp3d geometric from 1 Pa to 2000 Pa down the upper half of the column and about 2000 Pa
    below, +-10 % horizontal noise; T from a lapse-rate profile between 180 and 300 K; v about +-50 m/s with sign
    changes inside each element; Qdp = q*dp with q log-spaced from 1e-7 to 2e-2 down the column; eta_dot_dpdn zero at
    the top and bottom interfaces."""
    harness.randomize(s, seed=seed)
    rng = np.random.default_rng(seed + 7919)
    E, L, ntl, Q = s.nelem, s.nlev, s.ntl, s.qsize_d
    A = s.arrays
    s.ps0 = 1.0e5
    s.hyai[...] = np.linspace(1.0e-4, 0.0, L + 1)
    top = max(L // 2, 2)
    prof = np.full(L, 2000.0)
    prof[:top] = np.geomspace(1.0, 2000.0, top)
    noise = lambda *shape: 1.0 + 0.1 * rng.uniform(-1.0, 1.0, size=shape)
    dp = prof[None, None, :, None, None] * noise(E, ntl, L, 4, 4)
    A["elem_state_dp3d"][...] = dp
    p = s.hyai[0] * s.ps0 + np.cumsum(dp, axis=2) - 0.5 * dp
    A["elem_state_T"][...] = 180.0 + 120.0 * (p / p[:, :, -1:]) ** 0.3 + rng.uniform(-1.0, 1.0, size=dp.shape)
    ph = rng.uniform(0.0, 2.0 * np.pi, size=(E, ntl, L, 1, 1, 2))
    ij = np.arange(4)
    wave = ij[:, None, None] * 1.3 + ij[None, :, None] * 0.9 * np.array([1.0, -1.0])
    A["elem_state_v"][...] = 50.0 * np.sin(ph + wave)
    q = np.geomspace(1.0e-7, 2.0e-2, L)
    A["elem_state_Qdp"][...] = q[:, None, None] * dp[:, None, None, 0] * noise(E, Q, 2, L, 4, 4)
    eta = A["elem_derived_eta_dot_dpdn"]
    eta[:, 0] = 0.0
    eta[:, L] = 0.0
    s.consts[0] = 1.0 / 6.376e6
    return s


def make_state(gen, E, L, seed, qsize_d=1):
    s = harness.PortOracle().init(E, L, qsize_d)
    return stratified(s, seed) if gen == "stratified" else harness.randomize(s, seed=seed)


def level_scaled(rng, field, lo=1e-8):
    """field scaled per element and per level by factors log-uniform in [lo, 1]: a row computed with the wrong
    element's geometry, or a padded or clipped row leaking into a real one, shows at the small rows."""
    E, L = field.shape[:2]
    f = 10.0 ** rng.uniform(np.log10(lo), 0.0, size=(E, L))
    return field * f.reshape((E, L) + (1,) * (field.ndim - 2))


def level_local_inputs(gen, E, L, seed, qsize_d=1):
    """state, vstar / vector field (E,L,4,4,2), scalar field (E,L,4,4) and tensorVisc for the level-local operators"""
    s = make_state(gen, E, L, seed, qsize_d)
    rng = np.random.default_rng(seed)
    if gen == "stratified":
        vin = level_scaled(rng, s.arrays["elem_state_v"][:, 0])
        sin = level_scaled(rng, s.arrays["elem_state_T"][:, 0])
        A = s.arrays["elem_state_Qdp"]
        A[...] = level_scaled(rng, A.reshape(E, qsize_d * 2 * L, 4, 4)).reshape(A.shape)
    else:
        vin = rng.uniform(-40.0, 40.0, size=(E, L, 4, 4, 2))
        sin = rng.uniform(200.0, 300.0, size=(E, L, 4, 4))
    tv = rng.uniform(-1.0, 1.0, size=(E, 4, 4, 2, 2))
    return s, np.ascontiguousarray(vin), np.ascontiguousarray(sin), tv


# ---- the case matrices (shared with the GPU tests) ------------------------------------------------------------------

TLS = [(0, 1, 2), (0, 0, 0), (1, 0, 0)]
GENS = ("stratified", "randomize")


def _rhs_cases():
    """compute_and_apply_rhs, 2 calls: every level count with both generators on the Lagrangian branch, the Eulerian
    branch at 26, 72, 127, 128; time levels and qn0 rotate; every fourth case runs a sub-range with nets > 0."""
    cases = []
    n = 0
    for eulerian, nlevs in ((False, (8, 16, 24, 26, 30, 64, 72, 96, 104, 127, 128)), (True, (26, 72, 127, 128))):
        for L in nlevs:
            for gen in GENS:
                E = 7 + (n * 5) % 10
                rng = (2, E - 1) if n % 4 == 3 else (0, E)
                cases.append(dict(nlev=L, eulerian=eulerian, gen=gen, tls=TLS[n % 3], qn0=(n % 3) - 1, E=E, range=rng,
                                  seed=1000 + n))
                n += 1
    return cases


RHS_CASES = _rhs_cases()
EULER_CASES = [dict(nlev=L, gen=GENS[i % 2], qn0=i % 2, qsize=35 - 1 - 3 * (i % 3), seed=2000 + i)
               for i, L in enumerate((5, 8, 9, 30, 72, 127, 128))]
DIVWK_CASES = [dict(nlev=L, gen=GENS[i % 2], seed=3000 + i) for i, L in enumerate((5, 8, 9, 30, 72, 127, 128))]
# laplacians: 5 and 13 run on the groups-of-8 kernel, 16 and up on the 32-row flat tiles; E is chosen so that
# E * nlev is not a multiple of 32 and tiles straddle elements
LAP_CASES = [dict(nlev=L, E=E, gen=GENS[i % 2], seed=4000 + i)
             for i, (L, E) in enumerate(((5, 11), (13, 9), (16, 11), (17, 13), (24, 9), (40, 11), (72, 13), (127, 9),
                                         (128, 11)))]


def case_id(c):
    return "-".join(f"{k}{v}" for k, v in c.items() if k != "seed").replace(" ", "")


def rhs_case_state(c):
    s = make_state(c["gen"], c["E"], c["nlev"], c["seed"])
    s.ctl[0:2] = c["range"]
    s.ctl[2:5] = c["tls"]
    s.ctl[5] = c["qn0"]
    hybi = np.linspace(0.0, 1.0, c["nlev"] + 1) ** 1.5 if c["eulerian"] else None
    return s, hybi


def rhs_reference(s, ncalls, hybi):
    return hp.compute_and_apply_rhs(hp.from_state(s), ncalls, hybi)


def port_run(s, ncalls, hybi):
    orc = harness.PortOracle()
    if hybi is None:
        orc.run(s, ncalls)
    else:
        orc.run_eulerian(s, hybi, ncalls)


WORST = {}           # (operator, field) -> worst ratio over this session's soundness checks


def note(op, field, g, ref):
    r, at, vm = hp.worst(g, ref)
    if r >= WORST.get((op, field), (-1.0,))[0]:
        WORST[(op, field)] = (r, at, vm)
    return r


# ---- double entry: the longdouble reference against the FP64 restatement --------------------------------------------

@pytest.mark.parametrize("c", RHS_CASES, ids=case_id)
def test_rhs_double_entry_and_soundness(c):
    """The longdouble stages agree with PortOracle.run / run_eulerian to 1e-13 field-normalised (a transliteration slip
    shows far above that), and the FP64 restatement passes the pointwise gate at every point."""
    s, hybi = rhs_case_state(c)
    ref = rhs_reference(s, 2, hybi)
    got = s.copy()
    port_run(got, 2, hybi)
    K = hp.k_rhs(c["nlev"], 2)
    op = "rhs_eulerian" if hybi is not None else "rhs"
    for n in harness.FIELD_NAMES:
        R = ref.arrays[n]
        assert hp.rel_err(got.arrays[n], R.v) <= 1e-13, (n, hp.rel_err(got.arrays[n], R.v))
        if n in harness.MUTATED:
            assert note(op, n, got.arrays[n], R) <= K, (n, hp.worst(got.arrays[n], R), K)
        else:
            assert np.array_equal(got.arrays[n], R.v.astype(np.float64)), n


@pytest.mark.parametrize("c", EULER_CASES, ids=case_id)
def test_euler_step_double_entry_and_soundness(c):
    E, L, Q = 9, c["nlev"], 35
    s, vstar, _, _ = level_local_inputs(c["gen"], E, L, c["seed"], qsize_d=Q)
    s.ctl[0:2] = (1, E - 1)
    dt = 150.0
    got = np.zeros((E, Q, L, 4, 4))
    harness.PortOracle().euler_step(s, vstar, got, c["qn0"], c["qsize"], dt)
    ref = hp.euler_step(hp.from_state(s), vstar, c["qn0"], c["qsize"], dt)
    assert hp.rel_err(got, ref.v) <= 1e-13
    assert note("euler_step", "qtens", got, ref) <= hp.K_EULER


@pytest.mark.parametrize("c", DIVWK_CASES + LAP_CASES, ids=case_id)
@pytest.mark.parametrize("name", ["divergence_sphere_wk", "laplace_simple", "laplace_tensor"])
def test_sphere_wk_double_entry_and_soundness(c, name):
    E, L = c.get("E", 9), c["nlev"]
    s, vin, sin, tv = level_local_inputs(c["gen"], E, L, c["seed"])
    nets, nete = 1, E - 1
    field = vin if name == "divergence_sphere_wk" else sin
    got = harness.PortOracle().sphere_wk(name, s, field, tv if name == "laplace_tensor" else None, nets, nete)
    ref = hp.sphere_wk(name, hp.from_state(s), field, tv, nets, nete)
    assert hp.rel_err(got, ref.v) <= 1e-13
    assert note(name, "out", got, ref) <= hp.K_SPHERE_WK[name]


def test_fp64_stages_pass_their_own_gate():
    """The reference's own stages evaluated in FP64 (einsum order, not the restatement's) are a legitimate evaluation
    order: they pass the gate too. The defect (a) below differs from this run in one stage only."""
    c = RHS_CASES[1]
    s, hybi = rhs_case_state(c)
    ref = rhs_reference(s, 2, hybi)
    f64 = hp.compute_and_apply_rhs(hp.from_state(s, np.float64), 2, hybi)
    for n in harness.MUTATED:
        assert hp.gate(f64.arrays[n].v, ref.arrays[n], hp.k_rhs(c["nlev"], 2)), n


# ---- teeth: plausible fast-path defects that pass the field-normalised gate and fail the pointwise one ------------------

def old_gate(got, want):
    return hp.rel_err(got, want) <= TOL


def test_teeth_pressure_as_total_minus_suffix(monkeypatch):
    """(a) p[k] = (column total) - (suffix sum below k): the same sum, but its error at the top is u * p_surface."""
    def pressure_from_total(hyai0, ps0, dp):
        d = hp._levels(dp)
        total = hyai0 * ps0
        for x in d:
            total = total + x
        p, below = [None] * len(d), None
        for k in range(len(d) - 1, -1, -1):
            half = 0.5 * d[k]
            p[k] = total - (half if below is None else below + half)
            below = d[k] if below is None else below + d[k]
        return hp.HP.stack(p, 1)

    s = make_state("stratified", 8, 72, seed=5)
    ref = rhs_reference(s, 1, None)
    want = s.copy()
    port_run(want, 1, None)
    monkeypatch.setattr(hp, "pressure", pressure_from_total)
    bad = hp.compute_and_apply_rhs(hp.from_state(s, np.float64), 1, None)
    failed = []
    for n in harness.MUTATED:
        g = bad.arrays[n].v
        assert old_gate(g, want.arrays[n]), (n, hp.rel_err(g, want.arrays[n]))
        if not hp.gate(g, ref.arrays[n], hp.k_rhs(72)):
            failed.append(n)
    print(f"\n[teeth a] pointwise gate fails on {failed}")
    assert "elem_derived_omega_p" in failed


def test_teeth_tracer_top_group_off():
    """(b) qtens of the top 8-level group off by 1e-6 relative (about what an FP32 intermediate does), realistic Qdp."""
    E, L = 9, 72
    s, vstar, _, _ = level_local_inputs("stratified", E, L, 77, qsize_d=2)
    stratified(s, 77)                                       # unscaled columns: Qdp from 1e-7 to 40 kg/m^2-ish
    s.ctl[0:2] = (0, E)
    want = np.zeros((E, 2, L, 4, 4))
    harness.PortOracle().euler_step(s, vstar, want, 0, 2, 150.0)
    ref = hp.euler_step(hp.from_state(s), vstar, 0, 2, 150.0)
    bad = want.copy()
    bad[:, :, :8] *= 1.0 + 1e-6
    assert old_gate(bad, want), hp.rel_err(bad, want)
    assert hp.gate(want, ref, hp.K_EULER)
    assert not hp.gate(bad, ref, hp.K_EULER)


def test_teeth_laplacian_with_the_neighbours_geometry():
    """(c) one element of laplace_tensor computed with its neighbour's spheremp and Dinv (what a wrong slot of the flat
    kernel's geometry cache does). The element's field is scaled down 1e-14, below what the field-normalised gate can
    see: at 1e-8 a whole wrong element still fails that gate."""
    E, L, e = 9, 40, 4
    s, _, sin, tv = level_local_inputs("stratified", E, L, 91)
    sin[e] *= 1e-14
    orc = harness.PortOracle()
    want = orc.sphere_wk("laplace_tensor", s, sin, tv, 0, E)
    ref = hp.sphere_wk("laplace_tensor", hp.from_state(s), sin, tv, 0, E)
    wrong = s.copy()
    wrong.arrays["elem_spheremp"][e] = s.arrays["elem_spheremp"][e + 1]
    wrong.arrays["elem_Dinv"][e] = s.arrays["elem_Dinv"][e + 1]
    bad = want.copy()
    bad[e] = orc.sphere_wk("laplace_tensor", wrong, sin, tv, e, e + 1)[e]
    assert old_gate(bad, want), hp.rel_err(bad, want)
    assert hp.gate(want, ref, hp.K_LAPLACE_TENSOR)
    assert not hp.gate(bad, ref, hp.K_LAPLACE_TENSOR)


def test_teeth_padded_last_level():
    """(d) nlev = 30 (run on the 32-level instance): the last real level of every mutated field off by 1e-13 of the
    field's maximum, as a padding level leaking into it would leave it."""
    L = 30
    s = make_state("stratified", 8, L, seed=30)
    ref = rhs_reference(s, 1, None)
    want = s.copy()
    port_run(want, 1, None)
    failed = []
    for n in harness.MUTATED:
        a = want.arrays[n]
        bad = a.copy()
        lev = bad[:, int(s.ctl[3])] if n in ("elem_state_dp3d", "elem_state_v", "elem_state_T") else bad
        k = L if n == "elem_derived_eta_dot_dpdn" else L - 1
        lev[:, k] += 1e-13 * np.max(np.abs(a))
        assert old_gate(bad, a), n
        assert hp.gate(a, ref.arrays[n], hp.k_rhs(L)), n
        if not hp.gate(bad, ref.arrays[n], hp.k_rhs(L)):
            failed.append(n)
    print(f"\n[teeth d] pointwise gate fails on {failed}")
    for n in ("elem_state_dp3d", "elem_state_T", "elem_state_v", "elem_derived_phi"):
        assert n in failed, n


def test_zz_report_worst_ratios(capsys):
    """Not a gate: the worst |g - v| / (u M) of the FP64 restatement per operator and field (K is the gate)."""
    with capsys.disabled():
        for (op, n), (r, at, vm) in sorted(WORST.items()):
            print(f"\n[pointwise cpu] {op:22s} {n:28s} worst ratio {r:7.3f} at {at}, |v|/M {vm:.2e}", end="")
        print()
