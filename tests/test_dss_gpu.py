"""caar_set_connectivity, caar_dss, caar_neighbor_minmax and caar_run_rk5_dss on the GPU, bit for bit against
tests/dss_oracle.py: cubed spheres (permuted, with rotated element blocks) and random meshes with up to 8 copies per
point, at nlev 72, 30 and 128 and at 2, 3, 5, 7, 26, 80, 127 and 131 (every residue of the level batches' tails), every
field alone and all together, both weightings, every tl, both qtl, qsize < qsize_d,
with every value outside the selection compared by bits; a size where the walk over the groups wraps; the full ne = 120
mesh; the five-call limited tracer step; the RK5 step with a DSS after every stage; argument errors, launch counts,
connectivity input and run-to-run bits."""
import ctypes as C

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
import dss_oracle as do
import limiter_oracle as lo
import rk5_oracle as ro
import tracer_ssp_oracle as so
from oracle import harness
from test_pointwise_cpu import level_local_inputs

pytestmark = pytest.mark.gpu
INVALID, STATE_ERR = 1, 5
F = {n: tb.capi.FIELD_BIT[n] for n in tb.DSS_FIELDS}
ALL4 = tuple(tb.DSS_FIELDS)
SEL_NAMES = ("elem_spheremp",) + ALL4
TOL = 1e-12
STATE_NAMES = ("elem_state_dp3d", "elem_state_v", "elem_state_T")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def random_fields(E, L, Qd, ntl, seed):
    """spheremp in [0.5, 2) and every state value a random double in [2, 2^17) of full mantissa (so that every bit of
    every slice is distinct from its neighbours')"""
    rng = np.random.default_rng(seed)
    out = {"elem_spheremp": rng.uniform(0.5, 2.0, (E, 4, 4))}
    for n in ALL4:
        shape = tb.field_shape(n, E, L, Qd, ntl)
        out[n] = rng.integers(0x4000000000000000, 0x4100000000000000, size=shape, dtype=np.uint64).view(np.float64)
    return out


def handle_with(E, L, Qd, ntl, arrays, gid):
    h = tb.Caar(E, L, Qd, ntl)
    h.upload({n: np.ascontiguousarray(arrays[n]) for n in SEL_NAMES}, names=SEL_NAMES)
    if gid is not None:
        h.set_connectivity(gid)
    return h


def download(h, E, L, Qd, ntl, names=SEL_NAMES):
    out = {n: np.empty(tb.field_shape(n, E, L, Qd, ntl)) for n in names}
    h.download(out, names=names)
    return out


MESHES = {
    "cube2": lambda rng: do.cubed_sphere_gid(2, rng),
    "cube3": lambda rng: do.cubed_sphere_gid(3, rng),
    "cube5": lambda rng: do.cubed_sphere_gid(5, rng),
    "random8": lambda rng: do.random_gid(40, rng, 8),
}
# nlev 72, 30, 128, then the tails of dss_slice's level batches (2 levels of v, 4 of a scalar): L % 4 = 0, 1, 2, 3 and a
# single partial batch, on groups of up to 4 copies (cube*) and of up to 8 (random8)
CASES = [("cube2", 72), ("cube3", 30), ("cube5", 128), ("random8", 72), ("random8", 30), ("cube3", 72),
         ("cube2", 2), ("random8", 3), ("cube3", 5), ("random8", 7), ("cube2", 26), ("cube3", 80), ("random8", 80),
         ("cube5", 127), ("random8", 131), ("cube2", 131)]
SELECTIONS = [(n,) for n in ALL4] + [ALL4]


@pytest.mark.parametrize("mesh,L", CASES, ids=[f"{m}-L{L}" for m, L in CASES])
def test_dss_equals_oracle(mesh, L):
    """Every selection (each field alone, all four) with both weightings; tl and qtl cycle through every value. The whole
    of every field is compared by bits: the selection against the oracle, everything else against its input."""
    rng = np.random.default_rng(CASES.index((mesh, L)))
    gid = MESHES[mesh](rng)
    E, Qd, ntl = gid.shape[0], 4, 3
    conn = do.Connectivity(gid)
    inp = random_fields(E, L, Qd, ntl, 11 * L)
    h = handle_with(E, L, Qd, ntl, inp, gid)
    i = 0
    for names in SELECTIONS:
        for w in (do.ASSEMBLE, do.PROJECT):
            tl, qtl, qs = i % ntl, (i // 3) % 2, 3 if i % 2 else 1
            i += 1
            h.upload({n: np.ascontiguousarray(inp[n]) for n in ALL4}, names=ALL4)
            n0 = h.launch_count()
            h.dss(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
            assert h.launch_count() - n0 == 1
            got = download(h, E, L, Qd, ntl)
            want = {n: inp[n].copy() for n in SEL_NAMES}
            do.dss_arrays(want, conn, names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
            for n in SEL_NAMES:
                assert np.array_equal(bits(got[n]), bits(want[n])), (names, w, tl, qtl, n)
            assert not np.array_equal(bits(got[names[0]]), bits(inp[names[0]]))
    h.close()


def test_walk_wraps_ne60():
    """ne = 60 (21600 elements, 194402 groups) x 72: more groups than the threads of one launch (two CTAs of 256 per SM),
    so every thread walks more than one group. All four fields, ASSEMBLE; Qdp alone with PROJECT. Run twice: same bits."""
    import torch
    rng = np.random.default_rng(60)
    gid = do.cubed_sphere_gid(60, rng)
    E, L, Qd, ntl = gid.shape[0], 72, 2, 2
    conn = do.Connectivity(gid)
    assert conn.G > 2 * 256 * torch.cuda.get_device_properties(0).multi_processor_count
    inp = random_fields(E, L, Qd, ntl, 60)
    h = handle_with(E, L, Qd, ntl, inp, gid)
    for names, w, tl, qtl, qs in ((ALL4, do.ASSEMBLE, 1, 0, 2), (("elem_state_Qdp",), do.PROJECT, 0, 1, 1)):
        runs = []
        for _ in range(2):
            h.upload({n: np.ascontiguousarray(inp[n]) for n in ALL4}, names=ALL4)
            h.dss(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
            runs.append(download(h, E, L, Qd, ntl, ALL4))
        want = {n: inp[n].copy() for n in SEL_NAMES}
        do.dss_arrays(want, conn, names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
        for n in ALL4:
            assert np.array_equal(bits(runs[0][n]), bits(want[n])), (names, n)
            assert np.array_equal(bits(runs[1][n]), bits(runs[0][n])), (names, n)
    h.close()


def test_full_size_ne120():
    """86400 x 72, dp3d, v and T (four scalar fields) assembled at once in panel order. A sample of 2000 groups equals
    the oracle bit for bit; over the whole output every copy of a point holds the same bits and sum(spheremp * out) equals
    sum(in) to 1e-12 per level."""
    gid = do.cubed_sphere_gid(120)
    E, L, Qd, ntl = gid.shape[0], 72, 1, 1
    conn = do.Connectivity(gid)
    assert (E, conn.G, int(conn.mult.sum())) == (86400, 777602, 1382400)
    rng = np.random.default_rng(120)
    sph = rng.uniform(0.5, 2.0, (E, 4, 4))
    inp = {"elem_spheremp": sph}
    for n in STATE_NAMES:
        inp[n] = rng.uniform(-1.0, 1.0, tb.field_shape(n, E, L, Qd, ntl)) + (2.0 if n != "elem_state_v" else 0.0)
    h = tb.Caar(E, L, Qd, ntl)
    h.upload(inp, names=("elem_spheremp",) + STATE_NAMES)
    h.set_connectivity(gid)
    n0 = h.launch_count()
    h.dss(STATE_NAMES, tl=0)
    assert h.launch_count() - n0 == 1
    got = download(h, E, L, Qd, ntl, STATE_NAMES)
    h.close()
    s = sph.reshape(-1)
    sample = np.sort(rng.choice(conn.G, 2000, replace=False))
    for n in STATE_NAMES:
        comp = (2,) if n == "elem_state_v" else ()
        x = np.moveaxis(inp[n][:, 0].reshape((E, L, 16) + comp), 2, 1).reshape((E * 16, L) + comp)
        y = np.moveaxis(got[n][:, 0].reshape((E, L, 16) + comp), 2, 1).reshape((E * 16, L) + comp)
        tail = (slice(None),) + (None,) * (x.ndim - 1)
        for g in sample:      # the header's text on the sampled groups
            grp = conn.groups[g]
            m = s[grp[0]]
            for c in grp[1:]:
                m = m + s[c]
            S = x[grp[0]].copy()
            for c in grp[1:]:
                S = S + x[c]
            for c in grp:
                assert np.array_equal(bits(y[c]), bits(S * (1.0 / m))), (n, g)
        for c in range(1, conn.M):
            has = conn.mult > c
            assert np.array_equal(bits(y[conn.idx[has, c]]), bits(y[conn.idx[has, 0]])), (n, c)
        mass_in = x.sum(0)
        mass_out = (s[tail] * y).sum(0)
        assert np.all(np.abs(mass_out - mass_in) <= 1e-12 * np.abs(x).sum(0)), n


# ---- neighbor_minmax ------------------------------------------------------------------------------------------------

MINMAX_CASES = [("cube3", 30), ("random8", 30), ("cube3", 3), ("random8", 5), ("cube2", 80), ("random8", 127),
                ("cube3", 131)]


@pytest.mark.parametrize("mesh,L", MINMAX_CASES, ids=[m if L == 30 else f"{m}-L{L}" for m, L in MINMAX_CASES])
def test_neighbor_minmax_equals_oracle(mesh, L):
    """Random bounds [E][4][L][2], qsize 3: bit for bit with the numpy transcription, tracer 3 untouched; a second call
    widens again from the first call's output."""
    rng = np.random.default_rng(7)
    gid = MESHES[mesh](rng)
    E, Qd = gid.shape[0], 4
    conn = do.Connectivity(gid)
    b = np.ascontiguousarray(np.sort(rng.standard_normal((E, Qd, L, 2)), -1))
    h = tb.Caar(E, L, Qd)
    h.set_connectivity(gid)
    h.upload_bounds(b)
    want = b
    for qs in (3, 1):
        n0 = h.launch_count()
        h.neighbor_minmax(qs)
        assert h.launch_count() - n0 == 1
        want = do.neighbor_minmax_np(want, conn, qs)
        got = h.download_bounds()
        assert np.array_equal(bits(got), bits(want)), qs
    assert np.array_equal(bits(got[:, 3]), bits(b[:, 3]))
    assert not np.array_equal(bits(got), bits(b))
    h.close()


# ---- the five-call limited tracer step ------------------------------------------------------------------------------

QNAMES = ("elem_Dinv", "elem_metdet", "elem_rmetdet", "elem_spheremp", "elem_state_dp3d", "elem_state_Qdp")


def test_limited_tracer_step_strict():
    """bounds -> neighbor_minmax -> strict caar_advect_tracers -> limiter -> caar_dss(Qdp, PROJECT) on a permuted ne = 2
    sphere, qsize 2 of 3: equal in every bit to the FP64 composition of the oracles."""
    gid = do.cubed_sphere_gid(2, np.random.default_rng(2))
    E, L, Qd, qs, dtl, DT = gid.shape[0], 30, 3, 2, 1, 150.0
    conn = do.Connectivity(gid)
    s, vstar, _, _ = level_local_inputs("randomize", E, L, 6400, qsize_d=Qd)
    want = s.copy()
    h = tb.Caar(E, L, Qd, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays, names=QNAMES)
    h.upload_vstar(vstar)
    h.set_connectivity(gid)
    h.tracer_bounds(0, qs, dtl)
    h.neighbor_minmax(qs)
    q = h.advect_tracers(0, qs, DT, 1, tb.MODE_STRICT)
    h.limit_tracers(q, qs, dtl)
    h.dss(("elem_state_Qdp",), qtl=q, qsize=qs, weighting=tb.DSS_PROJECT)
    got = {"elem_state_Qdp": np.empty_like(s.arrays["elem_state_Qdp"])}
    h.download(got, names=("elem_state_Qdp",))
    gb = h.download_bounds()
    h.close()
    A = want.arrays
    wb = np.zeros((E, Qd, L, 2))
    lo.tracer_bounds(A["elem_state_Qdp"], A["elem_state_dp3d"], wb, 0, E, 0, qs, dtl)
    wb = do.neighbor_minmax_np(wb, conn, qs)
    want.ctl[0:2] = (0, E)
    qw = so.ssp_step(harness.PortOracle(), want, vstar, 0, qs, DT)
    assert qw == q
    r = lo.limit_tracers(A["elem_state_Qdp"], A["elem_state_dp3d"], A["elem_spheremp"], wb, 0, E, q, qs, dtl)
    do.dss_arrays(A, conn, ("elem_state_Qdp",), qtl=q, qsize=qs, weighting=do.PROJECT)
    assert np.array_equal(bits(gb), bits(wb))
    assert np.array_equal(bits(got["elem_state_Qdp"]), bits(A["elem_state_Qdp"]))
    assert (r["iters"] > 1).any()


# ---- caar_run_rk5_dss -----------------------------------------------------------------------------------------------

DT = 2.0


def rk5_handle(s, gid, hybi):
    h = tb.Caar(s.nelem, s.nlev, s.qsize_d, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    if hybi is not None:
        h.set_vertical_coordinate(0, hybi)
    h.set_control(*[int(x) for x in s.ctl], dt2=s.dt2)
    h.upload(s.arrays)
    h.set_connectivity(gid)
    return h


def rk5_state(L, seed):
    gid = do.cubed_sphere_gid(3, np.random.default_rng(seed))
    s = harness.randomize(harness.PortOracle().init(gid.shape[0], L), seed=seed)
    s.ctl[0:2] = (0, s.nelem)
    s.ctl[2:5] = (0, 1, 2)
    return s, gid


RK5_DSS_CASES = [(False, 72), (True, 72), (False, 5), (True, 5), (False, 127), (True, 127)]


@pytest.mark.parametrize("eulerian,L", RK5_DSS_CASES,
                         ids=[("eulerian" if e else "lagrangian") + ("" if L == 72 else f"-L{L}") for e, L in RK5_DSS_CASES])
def test_rk5_dss_strict_bit_identical(eulerian, L):
    """Strict mode, 2 steps on a permuted ne = 3 sphere at nlev 72, 5 and 127: every array equal to rk5_dss_step in every
    bit, 11 launches per step, levels rotated twice."""
    s, gid = rk5_state(L, 31 + eulerian + (L != 72) * L)
    hybi = np.linspace(0.0, 1.0, L + 1) ** 1.5 if eulerian else None
    want = s.copy()
    conn = do.Connectivity(gid)
    for _ in range(2):
        do.rk5_dss_step(harness.PortOracle(), want, DT, conn, hybi)
    got = s.copy()
    h = rk5_handle(got, gid, hybi)
    n0 = h.launch_count()
    h.run_rk5_dss(2, DT, tb.MODE_STRICT)
    assert h.launch_count() - n0 == 22
    h.download(got.arrays, names=None)
    assert (h.control.n0, h.control.np1, h.control.nm1) == tuple(want.ctl[2:5]) == (2, 0, 1)
    h.close()
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(got.arrays[n]), bits(want.arrays[n])), n
    assert all(np.isfinite(want.arrays[n]).all() for n in harness.MUTATED)


def test_rk5_dss_fast_equals_public_calls_and_strict():
    """Fast mode: one step equals five caar_run calls each followed by caar_dss, with the combination on the host, bit
    for bit; and it is within 1e-12 per field of the strict step."""
    s, gid = rk5_state(72, 41)
    dt, w = DT, float(s.consts[1])
    a = rk5_handle(s.copy(), gid, None)
    a.run_rk5_dss(1, dt, tb.MODE_FAST)
    man = s.copy()
    b = rk5_handle(man, gid, None)
    for st in ro.schedule(0, 1, 2, dt, w):
        if st == "combine":
            b.download(man.arrays, names=ro.COMBINED)
            for n in ro.COMBINED:
                X = man.arrays[n]
                X[:, 2] = (5 * X[:, 2] - X[:, 0]) / 4
            b.upload(man.arrays, names=ro.COMBINED)
            continue
        consts = s.consts.copy()
        consts[1] = st[4]
        b.set_params(consts, s.dvv, s.ps0, s.hyai)
        b.set_control(n0=st[0], np1=st[1], nm1=st[2], dt2=st[3])
        b.compute_and_apply_rhs(1, tb.MODE_FAST)
        b.dss(STATE_NAMES, tl=st[1])
    strict = rk5_handle(s.copy(), gid, None)
    strict.run_rk5_dss(1, dt, tb.MODE_STRICT)
    ga, gb, gs = s.copy(), s.copy(), s.copy()
    for h, g in ((a, ga), (b, gb), (strict, gs)):
        h.download(g.arrays, names=None)
        h.close()
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(ga.arrays[n]), bits(gb.arrays[n])), n
        ref = gs.arrays[n]
        err = float(np.max(np.abs(ga.arrays[n] - ref)) / max(np.max(np.abs(ref)), 1e-300))
        assert err <= TOL, (n, err)


def test_rk5_alone_unchanged_with_connectivity():
    """caar_run_rk5 on a handle that holds a connectivity runs no DSS: 6 launches per step and the bits of
    rk5_oracle.rk5_step (strict)."""
    s, gid = rk5_state(30, 51)
    want = s.copy()
    ro.rk5_step(harness.PortOracle(), want, DT)
    got = s.copy()
    h = rk5_handle(got, gid, None)
    n0 = h.launch_count()
    h.run_rk5(1, DT, tb.MODE_STRICT)
    assert h.launch_count() - n0 == 6
    h.download(got.arrays, names=None)
    h.close()
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(got.arrays[n]), bits(want.arrays[n])), n


# ---- connectivity input ---------------------------------------------------------------------------------------------

def test_connectivity_replaced_and_f90_layout():
    """A second caar_set_connectivity replaces the first (the result changes, and equals the oracle of the new map); the
    F90 layout ([ie][j][i]) of the transposed blocks gives the same bits as the C++ layout."""
    rng = np.random.default_rng(9)
    g1, g2 = do.cubed_sphere_gid(2, rng), do.random_gid(24, rng, 4)
    E, L, Qd, ntl = 24, 16, 1, 1
    inp = random_fields(E, L, Qd, ntl, 9)
    outs = []
    for gid, layout in ((g1, tb.capi.LAYOUT_CXX), (g2, tb.capi.LAYOUT_CXX), (np.swapaxes(g1, 1, 2), tb.capi.LAYOUT_F90)):
        h = handle_with(E, L, Qd, ntl, inp, g2 if layout == tb.capi.LAYOUT_F90 else g1)
        h.set_connectivity(gid, layout)
        h.dss(("elem_state_T",), tl=0)
        outs.append(download(h, E, L, Qd, ntl, ("elem_state_T",))["elem_state_T"])
        h.close()
    want2 = {n: inp[n].copy() for n in SEL_NAMES}
    do.dss_arrays(want2, do.Connectivity(g2), ("elem_state_T",), tl=0)
    assert np.array_equal(bits(outs[1]), bits(want2["elem_state_T"]))
    assert not np.array_equal(bits(outs[0]), bits(outs[1]))
    assert np.array_equal(bits(outs[2]), bits(outs[0]))


# ---- argument errors and launch counts ------------------------------------------------------------------------------

E_, L_, Q_, NTL_ = 24, 16, 2, 3
GOOD_DSS = dict(mask=F["elem_state_T"] | F["elem_state_Qdp"], tl=0, qtl=0, qsize=2, weighting=0)
DSS_BAD = ([dict(mask=tb.capi.FIELD_BIT["elem_spheremp"]), dict(mask=1 << 16), dict(tl=-1), dict(tl=NTL_),
            dict(qtl=-1), dict(qtl=2), dict(qsize=-1), dict(qsize=Q_ + 1), dict(weighting=2), dict(weighting=-1)])
# entry point, case, handle kind (None, "bare": no connectivity, "noparams": connectivity without caar_set_params,
# "ready"), arguments, code
ERR_CASES = (
    [("caar_dss", "null handle", None, {}, INVALID), ("caar_dss", "no connectivity", "bare", {}, STATE_ERR)]
    + [("caar_dss", f"{k}={v}", "ready", {k: v}, INVALID) for o in DSS_BAD for k, v in o.items()]
    + [("caar_neighbor_minmax", "null handle", None, {}, INVALID),
       ("caar_neighbor_minmax", "no connectivity", "bare", {}, STATE_ERR),
       ("caar_neighbor_minmax", "qsize=-1", "ready", dict(qsize=-1), INVALID),
       ("caar_neighbor_minmax", "qsize=3", "ready", dict(qsize=Q_ + 1), INVALID)]
    + [("caar_run_rk5_dss", "null handle", None, {}, INVALID),
       ("caar_run_rk5_dss", "no connectivity", "bare", {}, STATE_ERR),
       ("caar_run_rk5_dss", "before set_params", "noparams", {}, STATE_ERR),
       ("caar_run_rk5_dss", "null control", "ready", dict(ctl=None), INVALID),
       ("caar_run_rk5_dss", "range 1:24", "ready", dict(nets=1), INVALID),
       ("caar_run_rk5_dss", "range 0:23", "ready", dict(nete=E_ - 1), INVALID),
       ("caar_run_rk5_dss", "range 0:25", "ready", dict(nete=E_ + 1), INVALID),
       ("caar_run_rk5_dss", "levels 0,0,1", "ready", dict(tls=(0, 0, 1)), INVALID),
       ("caar_run_rk5_dss", "level 3", "ready", dict(tls=(0, 1, 3)), INVALID),
       ("caar_run_rk5_dss", "qn0 2", "ready", dict(qn0=2), INVALID),
       ("caar_run_rk5_dss", "nsteps -1", "ready", dict(nsteps=-1), INVALID),
       ("caar_run_rk5_dss", "mode 7", "ready", dict(mode=7), INVALID)]
    + [("caar_set_connectivity", "null handle", None, {}, INVALID),
       ("caar_set_connectivity", "null gid", "ready", dict(gid=None), INVALID),
       ("caar_set_connectivity", "layout 2", "ready", dict(layout=2), INVALID)]
)


@pytest.fixture(scope="module")
def env():
    gid = do.cubed_sphere_gid(2, np.random.default_rng(4))
    s = harness.randomize(harness.PortOracle().init(E_, L_, Q_, NTL_), seed=4)
    hs = {k: tb.Caar(E_, L_, Q_, NTL_) for k in ("bare", "noparams", "ready")}
    for k, h in hs.items():
        if k != "noparams":
            h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
        h.upload(s.arrays)
        if k != "bare":
            h.set_connectivity(gid)
        h.upload_bounds(np.sort(np.random.default_rng(5).standard_normal((E_, Q_, L_, 2)), -1))
    yield dict(gid=gid, handles=hs, state=s)
    for h in hs.values():
        h.close()


def call(env, ep, kind, over):
    lib = tb.load_library()
    h = env["handles"][kind].h if kind else None
    if ep == "caar_dss":
        a = {**GOOD_DSS, **over}
        return lib.caar_dss(h, a["mask"], a["tl"], a["qtl"], a["qsize"], a["weighting"]), None
    if ep == "caar_neighbor_minmax":
        return lib.caar_neighbor_minmax(h, over.get("qsize", 2)), None
    if ep == "caar_set_connectivity":
        gid = np.ascontiguousarray(env["gid"])
        p = None if "gid" in over else gid.ctypes.data_as(C.POINTER(C.c_longlong))
        return lib.caar_set_connectivity(h, p, over.get("layout", 0)), None
    tls = over.get("tls", (0, 1, 2))
    ctl = tb.capi.Control(over.get("nets", 0), over.get("nete", E_), *tls, over.get("qn0", 0), 0.5)
    arg = None if "ctl" in over else C.byref(ctl)
    rc = lib.caar_run_rk5_dss(h, arg, 1.0, over.get("nsteps", 1), over.get("mode", tb.MODE_FAST))
    return rc, (ctl.nets, ctl.nete, ctl.n0, ctl.np1, ctl.nm1, ctl.qn0, ctl.dt2)


def snapshot(h):
    return {**download(h, E_, L_, Q_, NTL_, ALL4), "bounds": h.download_bounds()}


@pytest.mark.parametrize("ep,case,kind,over,want", ERR_CASES, ids=[f"{c[0]}-{c[1]}" for c in ERR_CASES])
def test_rejected_call_changes_nothing(env, ep, case, kind, over, want):
    before = {k: snapshot(h) for k, h in env["handles"].items()}
    launches = {k: h.launch_count() for k, h in env["handles"].items()}
    rc, ctl = call(env, ep, kind, over)
    assert rc == want, tb.load_library().caar_last_error().decode()
    for k, h in env["handles"].items():
        h.sync()
        assert h.launch_count() == launches[k]
        after = snapshot(h)
        for n in after:
            assert np.array_equal(bits(after[n]), bits(before[k][n])), (k, n)
    if ctl is not None:
        tls = over.get("tls", (0, 1, 2))
        assert ctl == (over.get("nets", 0), over.get("nete", E_), *tls, over.get("qn0", 0), 0.5)


def test_launch_counts(env):
    """1 per caar_dss and caar_neighbor_minmax call with work, 0 for an empty selection, 11 per caar_run_rk5_dss step;
    set_connectivity launches nothing."""
    lib = tb.load_library()
    h = env["handles"]["ready"]
    for args, n in (((0, 0, 0, 0, 0), 0), ((F["elem_state_Qdp"], 0, 0, 0, 0), 0), ((F["elem_state_Qdp"], 0, 1, 1, 1), 1),
                    ((F["elem_state_v"], 2, 0, 0, 0), 1), ((sum(F.values()), 1, 1, 2, 1), 1)):
        k = h.launch_count()
        assert lib.caar_dss(h.h, *args) == 0
        h.sync()
        assert h.launch_count() - k == n, args
    for qs, n in ((0, 0), (1, 1), (2, 1)):
        k = h.launch_count()
        assert lib.caar_neighbor_minmax(h.h, qs) == 0
        assert h.launch_count() - k == n, qs
    k = h.launch_count()
    h.set_connectivity(env["gid"])
    ctl = tb.capi.Control(0, E_, 0, 1, 2, 0, 0.5)
    assert lib.caar_run_rk5_dss(h.h, C.byref(ctl), 1.0, 2, tb.MODE_FAST) == 0
    h.sync()
    assert h.launch_count() - k == 22 and (ctl.n0, ctl.np1, ctl.nm1) == (2, 0, 1)
