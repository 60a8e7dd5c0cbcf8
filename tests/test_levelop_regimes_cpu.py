"""The steady-state case matrix of the level-local kernels (tests/test_levelop_regimes_gpu.py) on the CPU: the cases
reach the work-distribution regime they are named for, and the pointwise gate catches the defects a slip in those
regimes would leave.

The level-local kernels are persistent and keep state from one unit of work to the next: ``levelop_kernel<OP>`` a ring
of NS = 4 input stages, a two-slot vstar item buffer refilled two items ahead and a per-warp geometry cache refilled on
every element change; ``laplace_flat_kernel<TENSOR>`` an 8-slot cache of point-local matrices and geometry staged two
tiles ahead, with tiles drawn in chunks from a counter; the strict tracer step a grid-stride loop. A case that gives a
warp one or two units checks none of that, so each case here is sized for a regime on a 148-SM B200, and ``regime``
restates the launch arithmetic that decides it.

The inputs are lean: only the geometry the operators read and the streamed field, so that 21600 x 72 and 76000 x 16
cases fit in a few hundred MB of host memory instead of the whole state."""
import numpy as np
import pytest

from oracle import harness
from oracle import hp_reference as hp
from test_pointwise_cpu import level_scaled

TOL = 1e-12          # the field-normalised gate of the parity tests

# ---- launch arithmetic ----------------------------------------------------------------------------------------------

SMS_B200 = 148
# CTAs per SM, from `ptxas -v` of the sm_100a build (tinman_sandbox_b200/csrc/caar_levelops.ptxas.log) and the dynamic
# shared memory of launch_op / launch_lapflat:
LEVELOP_PER_SM = 4   # levelop_kernel<OP>: 128 registers x 128 threads, 4 stages of 1-2 KB per warp
LAPFLAT_PER_SM = 2   # laplace_flat_kernel<TENSOR>: 194 (simple) / 212 (tensor) registers x 128 threads, ~100 KB smem
WPC = 4              # warps per CTA of both kernels (WPC and FW in caar_levelops.cu)
GL = 8               # levels per unit of levelop_kernel
FT = 32              # rows (element x level) per tile of laplace_flat_kernel


def regime(op, E, L, Q=1, sms=SMS_B200, per_sm=None):
    """The work distribution a launch on E elements gets: mirrors launch_op, launch_lapflat (csrc/caar_levelops.cu)
    and launch_euler_step (csrc/caar_euler.cu) and must follow them when they change. op: "euler" (fast tracer step),
    "divwk", "lap_rows" (the row-decomposed laplacians, nlev < 16), "lap_flat", "euler_strict"."""
    if op == "lap_flat":
        per_sm = LAPFLAT_PER_SM if per_sm is None else per_sm
        tiles = -(-E * L // FT)
        resident = sms * per_sm * WPC
        c = 2 if tiles < resident * 16 else 4
        warps = min(sms * per_sm, -(-tiles // WPC)) * WPC
        return dict(tiles=tiles, chunk=c, warps=warps, per_warp=tiles / warps, chunks=-(-tiles // c),
                    elems_per_tile=max((FT * t % L + FT - 1) // L + 1 for t in range(L)))
    if op == "euler_strict":
        groups = -(-E * L // 64)
        blocks = min(groups, sms * 3 * 2)
        return dict(groups=groups, blocks=blocks, iters=groups / blocks)
    per_sm = LEVELOP_PER_SM if per_sm is None else per_sm
    ng = -(-L // GL)
    units = E * ng * Q
    per_wave = sms * per_sm * WPC * (48 if op == "euler" else 12)
    wv = (units + per_wave // 2) // per_wave
    wv = 1 if (wv < 1 or op == "lap_rows") else min(wv, 16)
    warps = min(sms * per_sm * wv, -(-units // WPC)) * WPC
    upw = units / warps
    return dict(units=units, waves=wv, warps=warps, per_warp=upw, items_per_warp=upw / Q,
                elems_per_warp=upw / (Q * ng), groups=ng)


def levelop_unit_warp(units, warps, unit):
    """The warp whose contiguous range [units*w/warps, units*(w+1)/warps) holds `unit` (levelop_kernel's cut)."""
    w = unit * warps // units
    while units * w // warps > unit:
        w -= 1
    while units * (w + 1) // warps <= unit:
        w += 1
    return w


# ---- the case matrix ------------------------------------------------------------------------------------------------
# op, nlev, E (handle), element range, Q = qsize_d, qsize, qn0, generator, and the regime each case must reach on a
# 148-SM B200 at any occupancy from the ptxas value up to twice it (`need`: lower bounds on fields of regime()).

def _c(cid, op, L, E, rng=None, Q=1, qsize=1, qn0=0, gen="stratified", need=None):
    return dict(id=cid, op=op, nlev=L, E=E, range=rng or (0, E), Q=Q, qsize=qsize, qn0=qn0, gen=gen, need=need or {},
                seed=7000 + sum(map(ord, cid)))


CASES = [
    _c("T1", "euler", 72, 1024, (3, 1024 - 5), Q=35, qsize=34, need=dict(items_per_warp=1.2, per_warp=40, strict_iters=1.2)),
    _c("T2", "euler", 72, 4096, Q=4, qsize=4, qn0=1, gen="randomize", need=dict(items_per_warp=7, strict_iters=4)),
    _c("T3", "euler", 30, 21600, need=dict(items_per_warp=18, elems_per_warp=4.5, strict_iters=11)),
    _c("D1", "divwk", 72, 8192, gen="randomize", need=dict(per_warp=8.0)),
    _c("D2", "divwk", 30, 21600, (1, 21600), need=dict(per_warp=8.0, elems_per_warp=2.0)),
    _c("D3", "divwk", 128, 4096, gen="randomize", need=dict(per_warp=6.0)),
    _c("R1", "lap_rows", 13, 20000, need=dict(per_warp=8.0)),
    _c("R2", "lap_rows", 5, 60000, gen="randomize", need=dict(per_warp=12.0)),
    _c("F1", "lap_flat", 72, 21600, need=dict(chunk=4, per_warp=20)),
    _c("F2", "lap_flat", 30, 43200, (1, 43200), gen="randomize", need=dict(chunk=4, per_warp=12)),
    _c("F3", "lap_flat", 17, 72000, need=dict(chunk=4, per_warp=12, elems_per_tile=3)),
    _c("F4", "lap_flat", 16, 76000, gen="randomize", need=dict(chunk=4, per_warp=12)),
    _c("F5", "lap_flat", 128, 9600, need=dict(chunk=4, per_warp=12)),
]


def case_regime(c, sms=SMS_B200, per_sm=None):
    n = c["range"][1] - c["range"][0]
    r = regime(c["op"], n, c["nlev"], c["qsize"] if c["op"] == "euler" else 1, sms, per_sm)
    if c["op"] == "euler":
        r["strict_iters"] = regime("euler_strict", n, c["nlev"], sms=sms)["iters"]
    return r


def missed(c, r):
    """The `need` entries regime r does not meet (empty: the case reaches its regime)."""
    return {k: (r[k], v) for k, v in c["need"].items() if not r[k] >= v}


def reference_points(c):
    n = c["range"][1] - c["range"][0]
    return n * c["nlev"] * 16 * (c["qsize"] if c["op"] == "euler" else 1)


# ---- lean inputs ----------------------------------------------------------------------------------------------------

GEOMETRY = ("elem_Dinv", "elem_metdet", "elem_rmetdet", "elem_spheremp")


def lean_inputs(gen, E, L, seed, Q=0, qn0=0, qsize=0, vector=True, scalar=True):
    """A harness.State with only what the level-local operators read: the geometry of harness.randomize (distinct per
    element, |det D| >= 1/64) and, for the tracer step, Qdp (time level qn0 and tracers < qsize; the rest NaN, which
    no kernel may read). The other state arrays are one-value placeholders. Returns (state, vector field (E,L,4,4,2)
    = vstar, scalar field (E,L,4,4), tensorVisc (E,4,4,2,2)); fields not asked for are None. ``stratified``: the
    columns of tests/test_pointwise_cpu.stratified (log-spaced tracer mass from 1e-7 to 2e-2 on dp from 1 to 2000 Pa,
    winds of +-50 m/s changing sign inside an element, a lapse-rate temperature), then scaled per element and level
    by factors from 1e-8 to 1; ``randomize``: uniform fields as harness.randomize draws them."""
    base = harness.PortOracle().init(1, L)
    s = harness.State(E, L, qsize_d=max(Q, 1), ctl=base.ctl.copy(), dt2=base.dt2, consts=base.consts.copy(),
                      dvv=base.dvv.copy(), ps0=base.ps0, hyai=base.hyai.copy())
    s.consts[0] = 1.0 / 6.376e6
    s.ctl[0:2] = (0, E)
    rng = np.random.default_rng(seed)
    D = rng.uniform(-1.0, 1.0, size=(E, 4, 4, 2, 2))
    det = D[..., 0, 0] * D[..., 1, 1] - D[..., 0, 1] * D[..., 1, 0]
    D[np.abs(det) < 1.0 / 64] = np.array([[1.0, 0.25], [-0.25, 0.75]])
    det = D[..., 0, 0] * D[..., 1, 1] - D[..., 0, 1] * D[..., 1, 0]
    Dinv = np.stack([np.stack([D[..., 1, 1], -D[..., 0, 1]], -1), np.stack([-D[..., 1, 0], D[..., 0, 0]], -1)], -2)
    A = s.arrays
    A["elem_Dinv"] = Dinv / det[..., None, None]
    A["elem_metdet"] = np.abs(det)
    A["elem_rmetdet"] = 1.0 / np.abs(det)
    A["elem_spheremp"] = rng.uniform(1.0 / 64, 1.0, size=(E, 4, 4))
    for n in harness.FIELD_NAMES:
        A.setdefault(n, np.zeros(1))
    tv = rng.uniform(-1.0, 1.0, size=(E, 4, 4, 2, 2))
    strat = gen == "stratified"
    top = max(L // 2, 2)
    prof = np.full(L, 2000.0)
    prof[:top] = np.geomspace(1.0, 2000.0, top)
    vin = sin = None
    if vector:
        if strat:
            ph = rng.uniform(0.0, 2.0 * np.pi, size=(E, L, 1, 1, 2))
            ij = np.arange(4)
            wave = ij[:, None, None] * 1.3 + ij[None, :, None] * 0.9 * np.array([1.0, -1.0])
            vin = level_scaled(rng, 50.0 * np.sin(ph + wave))
        else:
            vin = rng.uniform(-40.0, 40.0, size=(E, L, 4, 4, 2))
    if scalar:
        if strat:
            p = 10.0 + np.cumsum(prof) - 0.5 * prof
            T = 180.0 + 120.0 * (p / p[-1]) ** 0.3
            sin = level_scaled(rng, T[None, :, None, None] + rng.uniform(-1.0, 1.0, size=(E, L, 4, 4)))
        else:
            sin = rng.uniform(200.0, 300.0, size=(E, L, 4, 4))
    if Q:
        qdp = np.full((E, Q, 2, L, 4, 4), np.nan)
        if strat:
            q = np.geomspace(1.0e-7, 2.0e-2, L) * prof
            x = q[None, None, :, None, None] * (1.0 + 0.1 * rng.uniform(-1.0, 1.0, size=(E, qsize, L, 4, 4)))
            qdp[:, :qsize, qn0] = level_scaled(rng, x.reshape(E, qsize * L, 4, 4)).reshape(x.shape)
        else:
            qdp[:, :qsize, qn0] = rng.uniform(0.0, 0.2, size=(E, qsize, L, 4, 4))
        A["elem_state_Qdp"] = qdp
    return s, vin, sin, tv


def sub_state(s, lo, hi):
    """Elements [lo,hi) of a lean state (geometry and Qdp), range [0, hi-lo): the reference in slices."""
    sub = harness.State(hi - lo, s.nlev, qsize_d=s.qsize_d, ctl=s.ctl.copy(), dt2=s.dt2, consts=s.consts, dvv=s.dvv,
                        ps0=s.ps0, hyai=s.hyai)
    sub.arrays = {n: (a[lo:hi] if a.shape[0] == s.nelem and a.ndim > 1 else a) for n, a in s.arrays.items()}
    sub.ctl[0:2] = (0, hi - lo)
    return sub


def hp_slice(name, s, lo, hi, field, tv=None, qn0=0, qsize=0, dt=150.0):
    """The extended-precision reference on elements [lo,hi) -> HP over those elements only."""
    sub = sub_state(s, lo, hi)
    hs = hp.from_state(sub)
    if name == "euler_step":
        return hp.euler_step(hs, field[lo:hi], qn0, qsize, dt)
    return hp.sphere_wk(name, hs, field[lo:hi], None if tv is None else tv[lo:hi], 0, hi - lo)


# ---- the case table reaches its regimes -----------------------------------------------------------------------------

@pytest.mark.parametrize("c", CASES, ids=lambda c: c["id"])
@pytest.mark.parametrize("scale", [1.0, 1.5, 2.0])
def test_case_reaches_its_regime(c, scale):
    """On 148 SMs at the ptxas occupancy and up to twice it; the reference stays between 2 and 40 M points."""
    per = LAPFLAT_PER_SM if c["op"] == "lap_flat" else LEVELOP_PER_SM
    r = case_regime(c, SMS_B200, int(round(per * scale)))
    assert not missed(c, r), (c["id"], missed(c, r), r)
    assert 2e6 <= reference_points(c) <= 4.1e7, reference_points(c)


def test_regime_mirrors_the_launch_arithmetic():
    """Spot values worked by hand from launch_op / launch_lapflat at 148 SMs."""
    r = regime("euler", 21600, 72, 4)                          # 777600 units, per wave 113664 -> 7 waves
    assert r["waves"] == 7 and r["warps"] == 148 * 4 * 7 * 4
    assert regime("divwk", 9, 72)["warps"] == 84               # 81 units: 21 CTAs
    f = regime("lap_flat", 21600, 72)                          # 48600 tiles >= 1184 * 16
    assert f["tiles"] == 48600 and f["chunk"] == 4 and f["warps"] == 1184
    assert regime("lap_flat", 8192, 72)["chunk"] == 2          # the two-stream test: 18432 < 18944
    assert regime("euler_strict", 9, 72)["iters"] == 1
    assert levelop_unit_warp(100, 7, 0) == 0 and levelop_unit_warp(100, 7, 99) == 6
    for u in range(100):
        w = levelop_unit_warp(100, 7, u)
        assert 100 * w // 7 <= u < 100 * (w + 1) // 7


def test_lean_inputs_match_the_full_state_layout():
    s, vin, sin, tv = lean_inputs("stratified", 5, 9, seed=1, Q=3, qn0=1, qsize=2)
    assert s.arrays["elem_Dinv"].shape == harness.field_shape("elem_Dinv", 5, 9)
    assert s.arrays["elem_state_Qdp"].shape == harness.field_shape("elem_state_Qdp", 5, 9, 3)
    D = s.arrays["elem_Dinv"]
    det = D[..., 0, 0] * D[..., 1, 1] - D[..., 0, 1] * D[..., 1, 0]
    assert np.allclose(np.abs(det) * s.arrays["elem_metdet"], 1.0)
    q = s.arrays["elem_state_Qdp"]
    assert np.all(np.isfinite(q[:, :2, 1])) and np.all(np.isnan(q[:, 2])) and np.all(np.isnan(q[:, :, 0]))
    assert vin.shape == (5, 9, 4, 4, 2) and sin.shape == (5, 9, 4, 4) and tv.shape == (5, 4, 4, 2, 2)
    # the FP64 restatement on the lean state passes the gate, slice by slice
    want = np.zeros((5, 3, 9, 4, 4))
    harness.PortOracle().euler_step(s, vin, want, 1, 2, 150.0)
    for lo, hi in ((0, 2), (2, 5)):
        assert hp.gate(want[lo:hi, :2], hp_slice("euler_step", s, lo, hi, vin, qn0=1, qsize=2)[:, :2], hp.K_EULER)
    got = harness.PortOracle().sphere_wk("laplace_tensor", s, sin, tv, 0, 5)
    assert hp.gate(got[1:4], hp_slice("laplace_tensor", s, 1, 4, sin, tv), hp.K_LAPLACE_TENSOR)


# ---- teeth: the defects a slip in the steady state leaves -----------------------------------------------------------

def old_gate(got, want):
    return hp.rel_err(got, want) <= TOL


def test_teeth_first_unit_after_an_element_change_uses_the_previous_geometry():
    """(1) A stale geometry cache: the first unit (tracer 0 of level group 0) of element e computed with element
    e - 1's Dinv, metdet and rmetdet. With geometry distinct per element the error is of the size of the rows it
    hits: the old gate sees it too unless those rows are small."""
    E, L, Q, e = 6, 16, 3, 3
    s, vstar, _, _ = lean_inputs("stratified", E, L, seed=11, Q=Q, qsize=Q, vector=True, scalar=False)
    want = np.zeros((E, Q, L, 4, 4))
    orc = harness.PortOracle()
    orc.euler_step(s, vstar, want, 0, Q, 150.0)
    ref = hp_slice("euler_step", s, 0, E, vstar, qsize=Q)
    wrong = s.copy()
    for n in ("elem_Dinv", "elem_metdet", "elem_rmetdet"):
        wrong.arrays[n][e] = s.arrays[n][e - 1]
    bad = want.copy()
    stale = np.zeros_like(want)
    orc.euler_step(wrong, vstar, stale, 0, Q, 150.0)
    bad[e, 0, :GL] = stale[e, 0, :GL]
    assert hp.gate(want, ref, hp.K_EULER)
    assert not hp.gate(bad, ref, hp.K_EULER)
    print(f"\n[teeth 1] old gate {'catches' if not old_gate(bad, want) else 'misses'} it "
          f"(field-normalised {hp.rel_err(bad, want):.1e})")


def test_teeth_tracers_with_the_previous_items_vstar():
    """(2) An item-buffer parity slip: the tracers of one (element, group) read the vstar tile of the item before
    it. Realistic winds of +-50 m/s differ between neighbouring groups by much more than the gate allows. On a group
    whose tracer mass is 1e-14 of the field's maximum the error is below 1e-12 of the field: the old gate misses it."""
    E, L, Q, e, g = 4, 24, 2, 2, 1
    s, vstar, _, _ = lean_inputs("stratified", E, L, seed=12, Q=Q, qsize=Q, vector=True, scalar=False)
    qdp = s.arrays["elem_state_Qdp"]
    grp = qdp[e, :, 0, g * GL:(g + 1) * GL]
    grp *= 1e-14 * np.max(np.abs(qdp[:, :, 0])) / np.max(np.abs(grp))
    orc = harness.PortOracle()
    want = np.zeros((E, Q, L, 4, 4))
    orc.euler_step(s, vstar, want, 0, Q, 150.0)
    ref = hp_slice("euler_step", s, 0, E, vstar, qsize=Q)
    slipped = vstar.copy()
    slipped[e, g * GL:(g + 1) * GL] = vstar[e, (g - 1) * GL:g * GL]
    stale = np.zeros_like(want)
    orc.euler_step(s, slipped, stale, 0, Q, 150.0)
    bad = want.copy()
    bad[e, :, g * GL:(g + 1) * GL] = stale[e, :, g * GL:(g + 1) * GL]
    assert hp.gate(want, ref, hp.K_EULER)
    assert not hp.gate(bad, ref, hp.K_EULER)
    assert old_gate(bad, want), hp.rel_err(bad, want)


def test_teeth_flat_laplacian_row_with_the_n_of_element_e_minus_8():
    """(3) Slot aliasing in the 8-slot cache of point-local matrices (slot = e & 7): one row of element e computed
    with the N of element e - 8. On a row 1e-14 of the field's maximum the old gate misses it."""
    E, L, e = 12, 20, 10
    s, _, sin, tv = lean_inputs("stratified", E, L, seed=13, vector=False)
    k = 7
    sin[e, k] *= 1e-14 * np.max(np.abs(sin)) / np.max(np.abs(sin[e, k]))
    orc = harness.PortOracle()
    want = orc.sphere_wk("laplace_tensor", s, sin, tv, 0, E)
    ref = hp_slice("laplace_tensor", s, 0, E, sin, tv)
    wrong = s.copy()
    wtv = tv.copy()
    for n in ("elem_Dinv", "elem_spheremp"):
        wrong.arrays[n][e] = s.arrays[n][e - 8]
    wtv[e] = tv[e - 8]
    bad = want.copy()
    bad[e, k] = orc.sphere_wk("laplace_tensor", wrong, sin, wtv, e, e + 1)[e, k]
    assert hp.gate(want, ref, hp.K_LAPLACE_TENSOR)
    assert not hp.gate(bad, ref, hp.K_LAPLACE_TENSOR)
    assert old_gate(bad, want), hp.rel_err(bad, want)


def test_teeth_skipped_tile_keeps_laplace_simple_output():
    """(4) A tile the scheduler skips in a buffer reused from a laplace_simple launch: 32 rows of the laplace_tensor
    output hold laplace_simple values. tensorVisc in [-1, 1] changes every value by O(1): the old gate sees it too,
    unless the tile lies in rows scaled far below the field's maximum, which the pointwise gate does not need."""
    E, L, tile = 6, 16, 1
    s, _, sin, tv = lean_inputs("stratified", E, L, seed=14, vector=False)
    orc = harness.PortOracle()
    want = orc.sphere_wk("laplace_tensor", s, sin, tv, 0, E)
    simple = orc.sphere_wk("laplace_simple", s, sin, None, 0, E)
    ref = hp_slice("laplace_tensor", s, 0, E, sin, tv)
    bad = want.copy().reshape(E * L, 16)
    bad[tile * FT:(tile + 1) * FT] = simple.reshape(E * L, 16)[tile * FT:(tile + 1) * FT]
    bad = bad.reshape(want.shape)
    assert hp.gate(want, ref, hp.K_LAPLACE_TENSOR)
    assert not hp.gate(bad, ref, hp.K_LAPLACE_TENSOR)
    print(f"\n[teeth 4] old gate {'catches' if not old_gate(bad, want) else 'misses'} it "
          f"(field-normalised {hp.rel_err(bad, want):.1e})")
