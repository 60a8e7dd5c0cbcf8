"""caar_run_rk5 (HOMME's tstep_type 5 step on the resident state) and its combination kernel on the GPU, against the
compositions of tests/rk5_oracle.py: the strict kernels bit for bit, the fast ones within 1e-12 per field and the
pointwise gate with k_rk5. Also the n0 == np1 != nm1 pattern of stages 3 to 5 on its own, the equivalence with five
public caar_run calls, the combination kernel at a size where its grid-stride loop wraps, a full-size step, the rank
split, run-to-run reproducibility and the error paths."""
import ctypes as C
import time

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
from oracle import harness
from oracle import hp_reference as hp
import rk5_oracle as ro
from test_pointwise_cpu import make_state

pytestmark = pytest.mark.gpu
T0 = time.time()
TOL = 1e-12
MODES = [tb.MODE_STRICT, tb.MODE_FAST]
MODE_NAME = {tb.MODE_STRICT: "strict", tb.MODE_FAST: "fast"}
DT = 2.0             # s: the randomize inputs stay finite over 3 steps (they blow up within about 100 s)
PERMS = [(0, 1, 2), (2, 0, 1), (1, 2, 0)]
WORST = {}           # kernel -> worst pointwise ratio against K


def rel_err(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def hybi_for(L, eulerian):
    return np.linspace(0.0, 1.0, L + 1) ** 1.5 if eulerian else None


def handle_for(s, hybi):
    h = tb.Caar(s.nelem, s.nlev, s.qsize_d, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    if hybi is not None:
        h.set_vertical_coordinate(0, hybi)
    h.set_control(*[int(x) for x in s.ctl], dt2=s.dt2)
    h.upload(s.arrays)
    return h


def gpu_rk5(s, hybi, dt, nsteps, mode):
    """run_rk5 on a copy of s -> the copy, with its ctl taken from the handle; checks the launch count and dt2."""
    got = s.copy()
    h = handle_for(got, hybi)
    n = h.launch_count()
    h.run_rk5(nsteps, dt, mode)
    h.download(got.arrays, names=None)
    c = h.control
    assert c.dt2 == s.dt2
    assert h.launch_count() - n == (6 * nsteps if s.ctl[1] > s.ctl[0] else 0)
    got.ctl[:] = (c.nets, c.nete, c.n0, c.np1, c.nm1, c.qn0)
    h.close()
    return got


def cpu_rk5(s, hybi, dt, nsteps):
    want = s.copy()
    orc = harness.PortOracle()
    for _ in range(nsteps):
        ro.rk5_step(orc, want, dt, hybi)
    return want


def rotated(tls, nsteps):
    for _ in range(nsteps):
        tls = ro.rotate(*tls)
    return tls


# ---- the n0 == np1 != nm1 pattern of stages 3 to 5, alone -----------------------------------------------------------

ALIAS_CASES = [(L, e, tls) for L, e in ((72, False), (128, False), (30, False), (72, True), (128, True))
               for tls in ((1, 1, 0), (2, 2, 0))]


@pytest.mark.parametrize("mode", MODES, ids=MODE_NAME.get)
@pytest.mark.parametrize("L,eulerian,tls", ALIAS_CASES)
def test_aliased_stage_pattern(L, eulerian, tls, mode):
    """One caar_run with (n0, np1, nm1) = (1, 1, 0) or (2, 2, 0): np1 overwrites the level being read while nm1 is
    another one. The Eulerian instances split over CTAs take the cluster-barrier path for np1 == n0."""
    s = harness.randomize(harness.PortOracle().init(9, L), seed=L + tls[0])
    s.ctl[2:5] = tls
    hybi = hybi_for(L, eulerian)
    want = s.copy()
    orc = harness.PortOracle()
    orc.run(want) if hybi is None else orc.run_eulerian(want, hybi)
    got = s.copy()
    h = handle_for(got, hybi)
    h.compute_and_apply_rhs(1, mode)
    h.download(got.arrays, names=None)
    h.close()
    if mode == tb.MODE_STRICT:
        for n in harness.FIELD_NAMES:
            assert np.array_equal(got.arrays[n], want.arrays[n]), n
        return
    ref = hp.compute_and_apply_rhs(hp.from_state(s), 1, hybi)
    for n in harness.MUTATED:
        assert rel_err(got.arrays[n], want.arrays[n]) <= TOL, n
        r, at, _ = hp.worst(got.arrays[n], ref.arrays[n])
        assert r <= hp.k_rhs(L), (n, r, at)


# ---- the strict step, bit for bit -----------------------------------------------------------------------------------

def _strict_cases():
    cases, i = [], 0
    for eulerian, nlevs in ((False, (72, 128, 30, 5, 130)), (True, (72, 128, 30, 5, 130))):
        for L in nlevs:
            for k in range(3):
                E = 6 + (i * 3) % 7
                cases.append(dict(nlev=L, eulerian=eulerian, tls=PERMS[(i + k) % 3], qn0=(i + k) % 3 - 1,
                                  nsteps=(1, 3)[(i + k) % 2], E=E, range=(2, E - 1) if k == 2 else (0, E), seed=9000 + i))
                i += 1
    return cases


def case_id(c):
    return "-".join(f"{k}{v}" for k, v in c.items() if k != "seed").replace(" ", "")


def case_state(c, gen="randomize"):
    s = make_state(gen, c["E"], c["nlev"], c["seed"])
    s.ctl[0:2] = c["range"]
    s.ctl[2:5] = c["tls"]
    s.ctl[5] = c["qn0"]
    return s, hybi_for(c["nlev"], c["eulerian"])


STRICT_CASES = _strict_cases()


@pytest.mark.parametrize("c", STRICT_CASES, ids=case_id)
def test_strict_step_bit_identical(c):
    """Every array, every time level, equal to the FP64 composition; elements outside [nets,nete) untouched; ctl
    rotated once per step. At nlev 130 fast mode announces its fallback to the strict kernel, and must match too."""
    s, hybi = case_state(c)
    want = cpu_rk5(s, hybi, DT, c["nsteps"])
    modes = [tb.MODE_STRICT] + ([tb.MODE_FAST] if c["nlev"] > 128 else [])
    for mode in modes:
        got = gpu_rk5(s, hybi, DT, c["nsteps"], mode)
        assert tuple(got.ctl[2:5]) == rotated(c["tls"], c["nsteps"]) == tuple(want.ctl[2:5])
        lo, hi = c["range"]
        for n in harness.FIELD_NAMES:
            assert np.array_equal(bits(got.arrays[n]), bits(want.arrays[n])), (MODE_NAME[mode], n)
            assert np.array_equal(got.arrays[n][:lo], s.arrays[n][:lo]) and np.array_equal(got.arrays[n][hi:], s.arrays[n][hi:])
        assert all(np.isfinite(want.arrays[n]).all() for n in harness.MUTATED)


def test_fast_mode_announces_the_fallback_above_128_levels():
    h = tb.Caar(2, 130)
    text, fused = h.describe(tb.MODE_FAST)
    h.close()
    assert not fused and "FALLBACK" in text


# ---- the fast step: 1e-12 per field and the pointwise gate ---------------------------------------------------------

FAST_DT = 1.0        # s: the stratified columns stay finite over two steps (CPU gate tests: k_rk5 holds at this dt)
FAST_CASES = [dict(c, nsteps=min(c["nsteps"], 2)) for c in STRICT_CASES if c["nlev"] <= 128][::2]


@pytest.mark.parametrize("gen", ["randomize", "stratified"])
@pytest.mark.parametrize("c", FAST_CASES, ids=case_id)
def test_fast_step(c, gen):
    """Within 1e-12 per field of the FP64 composition on the randomize inputs, and within k_rk5 u M of the
    long-double composition at every point on both. On the stratified columns the field-normalised 1e-12 is no
    yardstick: there the FP64 composition itself is up to 7e-11 of the field maximum away from the exact value
    (nlev 30), while its pointwise ratio stays below 2 % of k_rk5."""
    s, hybi = case_state(c, gen)
    want = cpu_rk5(s, hybi, FAST_DT, c["nsteps"])
    hs = hp.from_state(s)
    for _ in range(c["nsteps"]):
        ro.rk5_step_hp(hs, FAST_DT, hybi)
    got = gpu_rk5(s, hybi, FAST_DT, c["nsteps"], tb.MODE_FAST)
    assert tuple(got.ctl[2:5]) == tuple(want.ctl[2:5])
    K = ro.k_rk5(c["nlev"], c["nsteps"])
    lo, hi = c["range"]
    kernel = f"rk5_{'eulerian' if hybi is not None else 'lagrangian'}_{gen}"
    for n in harness.FIELD_NAMES:
        g = got.arrays[n]
        assert np.array_equal(g[:lo], s.arrays[n][:lo]) and np.array_equal(g[hi:], s.arrays[n][hi:]), n
        if n not in harness.MUTATED:
            assert np.array_equal(g, s.arrays[n]), n
            continue
        assert np.isfinite(want.arrays[n]).all(), n
        if gen == "randomize":
            assert rel_err(g, want.arrays[n]) <= TOL, (n, rel_err(g, want.arrays[n]))
        r, at, _ = hp.worst(g[lo:hi], hs.arrays[n][lo:hi])
        WORST[kernel] = max(WORST.get(kernel, 0.0), r / K)
        assert r <= K, (n, r, at, K)


# ---- the step equals the public calls ------------------------------------------------------------------------------

@pytest.mark.parametrize("L,eulerian", [(72, False), (30, True)])
def test_step_equals_five_public_calls(L, eulerian):
    """Fast mode: one run_rk5 step == five caar_run calls, set_params carrying each stage's eta_ave_w, plus the
    combination on the host, bit for bit. A plain caar_run afterwards uses the set_params value again."""
    s = harness.randomize(harness.PortOracle().init(11, L), seed=77)
    s.ctl[2:5] = (0, 1, 2)
    hybi = hybi_for(L, eulerian)
    dt, w = DT, float(s.consts[1])
    a = handle_for(s.copy(), hybi)
    a.run_rk5(1, dt, tb.MODE_FAST)
    man = s.copy()
    b = handle_for(man, hybi)
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
    b.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    assert (a.control.n0, a.control.np1, a.control.nm1) == (1, 2, 0)
    for h in (a, b):   # one more plain call on each, with the set_params eta_ave_w
        h.set_control(n0=1, np1=2, nm1=0, dt2=s.dt2)
        h.compute_and_apply_rhs(1, tb.MODE_FAST)
    ga, gb = s.copy(), s.copy()
    a.download(ga.arrays, names=None)
    b.download(gb.arrays, names=None)
    a.close()
    b.close()
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(ga.arrays[n]), bits(gb.arrays[n])), n


# ---- the combination kernel where its grid-stride loop wraps --------------------------------------------------------

@pytest.mark.parametrize("mode", MODES, ids=MODE_NAME.get)
def test_combination_kernel_at_scale(mode):
    """20000 x 72 on [3, E - 5): the kernel's grid (launch_rk5_combine: min(ceil(rows / 2048), 2 * SMs) CTAs of 512,
    rows = elements * 32 L of 16 B) makes every thread run its unrolled loop of 4 rows at least 4 times. nm1 after the
    step equals numpy's (5*u1 - u0)/4 with u1 from a caar_run of stage 1 alone, bit for bit; n0 is bit-untouched;
    the other elements hold sentinel bit patterns in every field and time level and keep them."""
    import torch
    E, L, lo, hi = 20000, 72, 3, 20000 - 5
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rows = (hi - lo) * 32 * L
    threads = min(-(-rows // 2048), 2 * sms) * 512
    assert rows // (4 * threads) >= 4, (rows, threads)
    s = harness.PortOracle().init(E, L)
    s.arrays["elem_spheremp"][...] = 1.0
    s.ctl[0:2] = (lo, hi)
    s.ctl[2:5] = (0, 1, 2)
    rng = np.random.default_rng(5)
    for n in harness.FIELD_NAMES:
        a = s.arrays[n]
        for part in (a[:lo], a[hi:]):
            part.view(np.uint64)[...] = rng.integers(0x4000000000000000, 0x4100000000000000, size=part.shape,
                                                     dtype=np.uint64)
    dt, w = DT, float(s.consts[1])
    got = s.copy()
    h = handle_for(got, None)
    h.run_rk5(1, dt, mode)
    h.download(got.arrays, names=None)
    h.close()
    u1 = s.copy()
    h = handle_for(u1, None)
    c = s.consts.copy()
    c[1] = w / 4
    h.set_params(c, s.dvv, s.ps0, s.hyai)
    h.set_control(n0=0, np1=2, nm1=0, dt2=dt / 5)
    h.compute_and_apply_rhs(1, mode)
    h.download(u1.arrays, names=ro.COMBINED)
    h.close()
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(got.arrays[n][:lo]), bits(s.arrays[n][:lo])), n
        assert np.array_equal(bits(got.arrays[n][hi:]), bits(s.arrays[n][hi:])), n
    for n in ro.COMBINED:
        a, b = u1.arrays[n][lo:hi, 2], s.arrays[n][lo:hi, 0]
        assert np.array_equal(bits(got.arrays[n][lo:hi, 2]), bits((5 * a - b) / 4)), n
        assert np.array_equal(bits(got.arrays[n][lo:hi, 0]), bits(b)), n


# ---- full size ------------------------------------------------------------------------------------------------------

def test_full_size_step_fast():
    """86400 x 72, one fast step. The handle is filled with 257 distinct randomize elements, tiled (element e holds
    pool element e % 257), so that every sampled element's expected value is rk5_step on its pool element: the first,
    middle and last 64 elements and 256 random ones are compared."""
    E, L, P = 86400, 72, 257
    pool = harness.randomize(harness.PortOracle().init(P, L), seed=86400)
    pool.ctl[0:2] = (0, P)
    pool.ctl[2:5] = (0, 1, 2)
    want = cpu_rk5(pool, None, DT, 1)
    h = tb.Caar(E, L)
    h.set_params(pool.consts, pool.dvv, pool.ps0, pool.hyai)
    h.set_control(0, E, 0, 1, 2, int(pool.ctl[5]), dt2=pool.dt2)
    reps = 32
    tile = {n: np.ascontiguousarray(np.concatenate([a] * reps)) for n, a in pool.arrays.items()}
    for e0 in range(0, E, P * reps):
        e1 = min(E, e0 + P * reps)
        h.upload_range({n: np.ascontiguousarray(a[:e1 - e0]) for n, a in tile.items()}, e0, e1)
    h.run_rk5(1, DT, tb.MODE_FAST)
    rng = np.random.default_rng(1)
    picks = [np.arange(0, 64), np.arange(E // 2 - 32, E // 2 + 32), np.arange(E - 64, E),
             np.sort(rng.choice(E, 256, replace=False))]
    for idx in picks:
        for e in idx:
            got = h.download_range(int(e), int(e) + 1, names=harness.MUTATED)
            for n in harness.MUTATED:
                w_ = want.arrays[n][e % P:e % P + 1]
                assert rel_err(got[n], w_) <= TOL, (int(e), n, rel_err(got[n], w_))
    assert (h.control.n0, h.control.np1, h.control.nm1) == (1, 2, 0)
    h.close()


# ---- rank split, reproducibility ------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", MODES, ids=MODE_NAME.get)
def test_two_handles_on_disjoint_halves_match_one(mode):
    E, L = 600, 72
    s = harness.randomize(harness.PortOracle().init(E, L), seed=600)
    s.ctl[0:2] = (0, E)
    s.ctl[2:5] = (0, 1, 2)
    one = handle_for(s.copy(), None)
    one.run_rk5(2, DT, mode)
    halves = []
    for e0, e1 in ((0, E // 2), (E // 2, E)):
        part = s.copy()
        part.nelem = e1 - e0
        part.arrays = {n: np.ascontiguousarray(a[e0:e1]) for n, a in s.arrays.items()}
        part.ctl[0:2] = (0, e1 - e0)
        h = handle_for(part, None)
        h.run_rk5(2, DT, mode)
        halves.append(h)
    for tl in range(3):
        want = one.checksums(tl, 0, E)["bits"]
        got = halves[0].checksums(tl)["bits"] + halves[1].checksums(tl)["bits"]   # uint64, mod 2^64
        assert np.array_equal(got, want), tl
    for h in [one] + halves:
        h.close()


def test_two_runs_reproduce_checksum_bits():
    """ne = 30 (5400 elements) x 72, closed-form init with spheremp = 1, dt = 1 s, 10 fast steps, twice: identical
    checksum bits at every time level after every step, and the state stays finite (with the closed-form spheremp
    of 2 to 8, every stage scales the state and it overflows within a few steps at any dt)."""
    E, L = 5400, 72
    s = harness.PortOracle().init(E, L)
    s.arrays["elem_spheremp"][...] = 1.0
    s.ctl[0:2] = (0, E)
    s.ctl[2:5] = (0, 1, 2)
    runs = []
    for _ in range(2):
        h = handle_for(s.copy(), None)
        trace = []
        for _ in range(10):
            h.run_rk5(1, 1.0, tb.MODE_FAST)
            cks = [h.checksums(tl, 0, E) for tl in range(3)]
            for ck in cks:
                assert np.isfinite(ck["sum"]).all() and np.isfinite(ck["sumsq"]).all()
            trace.append(np.stack([ck["bits"] for ck in cks]))
        h.close()
        runs.append(trace)
    for k in range(10):
        assert np.array_equal(runs[0][k], runs[1][k]), k


# ---- error paths and launch counts ----------------------------------------------------------------------------------

def test_error_paths_and_launch_counts():
    lib = tb.load_library()
    s = harness.randomize(harness.PortOracle().init(5, 16), seed=1)
    h = tb.Caar(5, 16)
    ctl = tb.capi.Control(0, 5, 0, 1, 2, 0, 0.5)
    rc = lambda c, n=1, mode=tb.MODE_FAST, dt=1.0: lib.caar_run_rk5(h.h, c, dt, n, mode)
    assert rc(C.byref(ctl)) == 5                              # CAAR_ERR_STATE before set_params
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays)
    assert rc(None) == 1
    for bad in (dict(n=-1), dict(mode=7)):
        assert rc(C.byref(ctl), **bad) == 1
    for tls in ((0, 0, 1), (0, 1, 1), (1, 0, 1), (0, 0, 0), (0, 1, 3)):
        c = tb.capi.Control(0, 5, *tls, 0, 0.5)
        assert rc(C.byref(c)) == 1, tls
        assert (c.n0, c.np1, c.nm1, c.dt2) == (*tls, 0.5)       # unchanged on a validation error
    assert h.launch_count() == 0
    assert rc(C.byref(ctl), n=0) == 0 and (ctl.n0, ctl.np1, ctl.nm1) == (0, 1, 2)
    assert rc(C.byref(ctl), n=2) == 0
    h.sync()
    assert h.launch_count() == 12 and (ctl.n0, ctl.np1, ctl.nm1) == (2, 0, 1) and ctl.dt2 == 0.5
    empty = tb.capi.Control(3, 3, 0, 1, 2, 0, 0.5)
    assert rc(C.byref(empty), n=1) == 0
    assert h.launch_count() == 12 and (empty.n0, empty.np1, empty.nm1) == (1, 2, 0)
    h.close()
    h2 = tb.Caar(3, 16, ntl=2)                                 # ntl < 3: never three distinct levels
    h2.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    for tls in ((0, 1, 0), (1, 0, 0), (0, 0, 1)):
        c = tb.capi.Control(0, 3, *tls, 0, 0.5)
        assert lib.caar_run_rk5(h2.h, C.byref(c), 1.0, 1, tb.MODE_STRICT) == 1
    h2.close()


def test_zz_report(capsys):
    with capsys.disabled():
        worst = ", ".join(f"{k} {v:.2e}" for k, v in sorted(WORST.items()))
        print(f"\n[rk5] worst pointwise ratio / k_rk5 (fast): {worst or 'n/a'}; "
              f"tests/test_rk5_gpu.py wall time {time.time() - T0:.1f} s")
