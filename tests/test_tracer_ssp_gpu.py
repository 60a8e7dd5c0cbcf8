"""caar_advect_tracers (HOMME's three-stage tracer step on the resident Qdp) on the GPU, against the compositions of
tests/tracer_ssp_oracle.py and against the public calls it replaces: the strict kernel bit for bit with the FP64
composition; fast mode bit for bit with three public caar_euler_step(dt/2) calls composed on the host, within 1e-12
per field and within k_ssp u M of the long-double composition. Also the in-place stages at the sizes where the
per-warp pipelines wrap, the average kernel where its grid-stride loop wraps, launch counts, qn0 toggling, error
paths, run-to-run bits, and a dynamics step followed by a tracer step followed by CAAR."""
import ctypes as C
import time

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
from oracle import harness
from oracle import hp_reference as hp
import rk5_oracle as ro
import tracer_ssp_oracle as so
from test_levelop_regimes_cpu import CASES as REGIME_CASES, lean_inputs
from test_pointwise_cpu import level_local_inputs

pytestmark = pytest.mark.gpu
T0 = time.time()
TOL = 1e-12
DT = 150.0
MODES = [tb.MODE_STRICT, tb.MODE_FAST]
MODE_NAME = {tb.MODE_STRICT: "strict", tb.MODE_FAST: "fast"}
QNAMES = ("elem_Dinv", "elem_metdet", "elem_rmetdet", "elem_state_Qdp")
WORST = {}


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def sentinel(rng, shape):
    return rng.integers(0x4000000000000000, 0x4100000000000000, size=shape, dtype=np.uint64).view(np.float64)


def with_sentinels(s, lo, hi, qsize, seed):
    """Sentinel bit patterns in Qdp outside [lo,hi) and at tracers iq >= qsize (both levels)."""
    rng = np.random.default_rng(seed)
    Q = s.arrays["elem_state_Qdp"]
    for part in (Q[:lo], Q[hi:], Q[lo:hi, qsize:]):
        part[...] = sentinel(rng, part.shape)
    return s


def handle(s, names=QNAMES):
    h = tb.Caar(s.nelem, s.nlev, s.qsize_d, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays, names=names)
    return h


def gpu_advect(s, vstar, qn0, qsize, dt, nsteps, mode, lo, hi, names=QNAMES):
    """advect_tracers on a handle holding s -> (Qdp, new qn0); checks the launch count and that vstar and a sentinel
    qtens are untouched."""
    h = handle(s, names)
    h.upload_vstar(vstar)
    E, L, Q = s.nelem, s.nlev, s.qsize_d
    qt = np.full((E, Q, L, 4, 4), -7.0)
    h.upload_extra(tb.X_QTENS, qt)
    n = h.launch_count()
    q = h.advect_tracers(qn0, qsize, dt, nsteps, mode, nets=lo, nete=hi)
    assert q == (qn0 + nsteps) % 2
    assert h.launch_count() - n == (4 * nsteps if hi > lo and qsize > 0 else 0)
    out = {"elem_state_Qdp": np.empty_like(s.arrays["elem_state_Qdp"])}
    h.download(out, names=("elem_state_Qdp",))
    assert np.array_equal(h.download_qtens(), qt)
    assert np.array_equal(h.download_extra(tb.X_VSTAR, vstar.shape), vstar)
    h.close()
    return out["elem_state_Qdp"], q


def cpu_ssp(s, vstar, qn0, qsize, dt, nsteps, lo, hi):
    want = s.copy()
    want.ctl[0:2] = (lo, hi)
    orc = harness.PortOracle()
    q = qn0
    for _ in range(nsteps):
        q = so.ssp_step(orc, want, vstar, q, qsize, dt)
    return want.arrays["elem_state_Qdp"], q


def public_ssp(s, vstar, qn0, qsize, dt, nsteps, mode, lo, hi, names=QNAMES):
    """The same steps through the public calls: three caar_euler_step(dt/2), each qtens downloaded and uploaded into
    Qdp(np1), then the average on the host."""
    h = handle(s, names)
    h.upload_vstar(vstar)
    Qh = s.arrays["elem_state_Qdp"].copy()
    r = slice(lo, hi)
    q = qn0
    for _ in range(nsteps):
        n0, np1 = q, 1 - q
        for src in so.schedule(n0, np1):
            if src == "average":
                Qh[r, :qsize, np1] = so.average(Qh[r, :qsize, n0], Qh[r, :qsize, np1])
            else:
                h.euler_step(src, qsize, dt / 2, mode, nets=lo, nete=hi)
                Qh[r, :qsize, np1] = h.download_qtens()[r, :qsize]
            h.upload({"elem_state_Qdp": Qh}, names=("elem_state_Qdp",))
        q = np1
    h.close()
    return Qh, q


# ---- strict: bit for bit with the FP64 composition ------------------------------------------------------------------

def _strict_cases():
    cases, i = [], 0
    for L in (72, 128, 30, 5):
        for k in range(3):
            E = 6 + (i * 3) % 5
            cases.append(dict(nlev=L, qsize=(1, 4, 34)[(i + k) % 3], qn0=i % 2, nsteps=(1, 3)[k % 2],
                              gen=("randomize", "stratified")[i % 2], E=E, range=(2, E - 1) if k == 2 else (0, E),
                              seed=5000 + i))
            i += 1
    return cases


def case_id(c):
    return "-".join(f"{k}{v}" for k, v in c.items() if k != "seed").replace(" ", "")


def case_inputs(c, qsize_d=35):
    s, vstar, _, _ = level_local_inputs(c["gen"], c["E"], c["nlev"], c["seed"], qsize_d=qsize_d)
    lo, hi = c["range"]
    return with_sentinels(s, lo, hi, c["qsize"], c["seed"]), vstar


STRICT_CASES = _strict_cases()


@pytest.mark.parametrize("c", STRICT_CASES, ids=case_id)
def test_strict_step_bit_identical(c):
    """qsize 1, 4 and 34 of qsize_d 35, qn0 0 and 1, 1 and 3 steps, sub-ranges: Qdp equal to the FP64 composition in
    every bit (sentinels outside the range and at iq >= qsize included); after one step Qdp(n0) is untouched."""
    s, vstar = case_inputs(c)
    lo, hi = c["range"]
    want, qw = cpu_ssp(s, vstar, c["qn0"], c["qsize"], DT, c["nsteps"], lo, hi)
    got, q = gpu_advect(s, vstar, c["qn0"], c["qsize"], DT, c["nsteps"], tb.MODE_STRICT, lo, hi)
    assert q == qw
    assert np.array_equal(bits(got), bits(want))
    Q0 = s.arrays["elem_state_Qdp"]
    if c["nsteps"] == 1:
        assert np.array_equal(bits(got[:, :, c["qn0"]]), bits(Q0[:, :, c["qn0"]]))
    for part in (np.s_[:lo], np.s_[hi:], np.s_[lo:hi, c["qsize"]:]):
        assert np.array_equal(bits(got[part]), bits(Q0[part]))


# ---- fast: the public calls bit for bit, 1e-12 and the pointwise gate -----------------------------------------------

FAST_CASES = [{k: v for k, v in c.items() if k != "gen"} for c in STRICT_CASES[::2]]


@pytest.mark.parametrize("gen", ["randomize", "stratified"])
@pytest.mark.parametrize("c", FAST_CASES, ids=case_id)
def test_fast_step(c, gen):
    """Bit for bit with the public calls; within 1e-12 per field of the FP64 composition on the randomize inputs and
    within k_ssp u M of the long-double composition at every point on both (on the stratified columns, scaled per
    level down to 1e-8, a field-normalised 1e-12 is no yardstick)."""
    c = dict(c, gen=gen)
    s, vstar = case_inputs(c)
    lo, hi = c["range"]
    qs, n = c["qsize"], c["nsteps"]
    got, q = gpu_advect(s, vstar, c["qn0"], qs, DT, n, tb.MODE_FAST, lo, hi)
    pub, qp = public_ssp(s, vstar, c["qn0"], qs, DT, n, tb.MODE_FAST, lo, hi)
    assert q == qp
    assert np.array_equal(bits(got), bits(pub))
    want, _ = cpu_ssp(s, vstar, c["qn0"], qs, DT, n, lo, hi)
    hs = hp.from_state(s)
    hs.nets, hs.nete = lo, hi
    qh = c["qn0"]
    for _ in range(n):
        qh = so.ssp_step_hp(hs, vstar, qh, qs, DT)
    ref = hs.arrays["elem_state_Qdp"]
    for lvl in (0, 1):
        g = got[lo:hi, :qs, lvl]
        if c["gen"] == "randomize":
            assert hp.rel_err(g, want[lo:hi, :qs, lvl]) <= TOL, lvl
        r, at, _ = hp.worst(g, ref[lo:hi, :qs, lvl])
        WORST[c["gen"]] = max(WORST.get(c["gen"], 0.0), r / so.k_ssp(n))
        assert r <= so.k_ssp(n), (lvl, r, at)


# ---- in place where the per-warp pipelines wrap ---------------------------------------------------------------------

REGIME_T = [c for c in REGIME_CASES if c["op"] == "euler"]


def regime_inputs(c):
    s, vin, _, _ = lean_inputs(c["gen"], c["E"], c["nlev"], c["seed"], Q=c["Q"], qn0=c["qn0"], qsize=c["qsize"],
                               scalar=False)
    return s, vin


@pytest.mark.parametrize("mode", MODES, ids=MODE_NAME.get)
@pytest.mark.parametrize("c", REGIME_T, ids=lambda c: c["id"])
def test_in_place_at_regime_sizes(c, mode):
    """Cases T1-T3 (tests/test_levelop_regimes_cpu.py): 10 to 60 units per warp, the input ring wrapping many times
    while stages 2 and 3 overwrite the tiles they read. One step equals the public calls bit for bit; the NaN the
    lean inputs put at iq >= qsize and outside the range keep their bits."""
    s, vin = regime_inputs(c)
    lo, hi = c["range"]
    got, q = gpu_advect(s, vin, c["qn0"], c["qsize"], DT, 1, mode, lo, hi)
    pub, _ = public_ssp(s, vin, c["qn0"], c["qsize"], DT, 1, mode, lo, hi)
    assert np.array_equal(bits(got), bits(pub))
    assert np.isfinite(got[lo:hi, :c["qsize"]]).all()


# ---- the average kernel where its grid-stride loop wraps -----------------------------------------------------------

def test_average_kernel_at_scale():
    """20000 x 30, qsize 2 of qsize_d 3, on [3, E - 5): launch_qdp_avg runs min(ceil(rows / 2048), 2 * SMs) CTAs of 512
    over rows = elements * qsize * 8 L of 16 B, so every thread runs its unrolled loop of 2 rows many times. Both modes
    equal their public calls bit for bit, with sentinels outside the range and at iq >= qsize."""
    import torch
    E, L, Qd, qs, lo, hi = 20000, 30, 3, 2, 3, 20000 - 5
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rows = (hi - lo) * qs * 8 * L
    threads = min(-(-rows // 2048), 2 * sms) * 512
    assert rows // (2 * threads) >= 4, (rows, threads)
    s, vin, _, _ = lean_inputs("randomize", E, L, 5200, Q=Qd, qn0=0, qsize=qs, scalar=False)
    with_sentinels(s, lo, hi, qs, 5200)
    for mode in MODES:
        got, _ = gpu_advect(s, vin, 0, qs, DT, 1, mode, lo, hi)
        pub, _ = public_ssp(s, vin, 0, qs, DT, 1, mode, lo, hi)
        assert np.array_equal(bits(got), bits(pub)), MODE_NAME[mode]
        Q0 = s.arrays["elem_state_Qdp"]
        for part in (np.s_[:lo], np.s_[hi:], np.s_[lo:hi, qs:]):
            assert np.array_equal(bits(got[part]), bits(Q0[part]))


# ---- launch counts, toggling, errors, reproducibility ---------------------------------------------------------------

def test_launch_counts_toggling_and_error_paths():
    lib = tb.load_library()
    s, vstar = case_inputs(dict(gen="randomize", E=5, nlev=16, seed=5300, range=(0, 5), qsize=2), qsize_d=3)
    h = tb.Caar(5, 16, 3)
    q = C.c_int(0)
    rc = lambda nets=0, nete=5, qp=C.byref(q), qsize=2, n=1, mode=tb.MODE_FAST: lib.caar_advect_tracers(
        h.h, nets, nete, qp, qsize, 1.0, n, mode)
    assert rc() == 5 and q.value == 0                          # CAAR_ERR_STATE before set_params
    assert lib.caar_advect_tracers(None, 0, 5, C.byref(q), 2, 1.0, 1, tb.MODE_FAST) == 1
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays, names=QNAMES)
    h.upload_vstar(vstar)
    assert rc(qp=None) == 1
    for bad in (dict(nets=-1), dict(nete=6), dict(nets=3, nete=2), dict(qsize=-1), dict(qsize=4), dict(n=-1),
                dict(mode=7)):
        assert rc(**bad) == 1, bad
        assert q.value == 0, bad
    for bad_q in (-1, 2):
        qq = C.c_int(bad_q)
        assert rc(qp=C.byref(qq)) == 1 and qq.value == bad_q
    assert h.launch_count() == 0
    assert rc(n=0) == 0 and q.value == 0
    assert rc(n=3) == 0 and q.value == 1
    h.sync()
    assert h.launch_count() == 12
    assert rc(nets=2, nete=2, n=3) == 0 and q.value == 0          # empty range: no launch, still toggles
    assert rc(qsize=0, n=1) == 0 and q.value == 1                 # qsize 0: the same
    assert h.launch_count() == 12
    assert rc(n=1, mode=tb.MODE_STRICT) == 0 and q.value == 0
    h.sync()
    assert h.launch_count() == 16
    h.close()


def test_two_runs_reproduce_bits():
    """21600 x 72, qsize 4, 5 fast steps, twice: Qdp identical in every bit."""
    E, L, Qd = 21600, 72, 4
    s, vin, _, _ = lean_inputs("stratified", E, L, 5400, Q=Qd, qn0=0, qsize=Qd, scalar=False)
    runs = [gpu_advect(s, vin, 0, Qd, DT, 5, tb.MODE_FAST, 0, E)[0] for _ in range(2)]
    assert np.isfinite(runs[0]).all()
    assert np.array_equal(bits(runs[0]), bits(runs[1]))


# ---- a dynamics step, a tracer step, then CAAR with the advanced water vapour ---------------------------------------

@pytest.mark.parametrize("L", [72, 30])
def test_rk5_then_tracers_then_caar(L):
    """Strict caar_run_rk5 (one step), strict caar_advect_tracers (one step from qn0 = 0), then a strict caar_run with
    ctl.qn0 = the new level: every array equal to the FP64 composition in every bit, so CAAR reads the advanced Qdp."""
    E, Qd = 7, 2
    s = harness.randomize(harness.PortOracle().init(E, L, Qd), seed=5500 + L)
    s.ctl[0:2] = (0, E)
    s.ctl[2:5] = (0, 1, 2)
    s.ctl[5] = 0
    vstar = np.random.default_rng(L).uniform(-40.0, 40.0, size=(E, L, 4, 4, 2))
    want = s.copy()
    orc = harness.PortOracle()
    ro.rk5_step(orc, want, 2.0)
    qn = so.ssp_step(orc, want, vstar, 0, Qd, DT)
    want.ctl[5] = qn
    orc.run(want)
    got = s.copy()
    h = tb.Caar(E, L, Qd, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.set_control(*[int(x) for x in s.ctl], dt2=s.dt2)
    h.upload(s.arrays)
    h.upload_vstar(vstar)
    h.run_rk5(1, 2.0, tb.MODE_STRICT)
    q = h.advect_tracers(0, Qd, DT, 1, tb.MODE_STRICT)
    assert q == qn == 1
    h.control.qn0 = q
    h.compute_and_apply_rhs(1, tb.MODE_STRICT)
    h.download(got.arrays, names=None)
    h.close()
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(got.arrays[n]), bits(want.arrays[n])), n


def test_zz_report(capsys):
    with capsys.disabled():
        worst = ", ".join(f"{k} {v:.2e}" for k, v in sorted(WORST.items()))
        print(f"\n[tracer ssp] worst pointwise ratio / k_ssp (fast): {worst or 'n/a'}; "
              f"tests/test_tracer_ssp_gpu.py wall time {time.time() - T0:.1f} s")
