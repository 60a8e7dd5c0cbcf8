"""The CUDA kernels, both modes, against the extended-precision reference (oracle/hp_reference.py) with the pointwise
gate |g - v| <= K u M at every point, on realistic columns (``stratified``) and on harness.randomize inputs; plus two
handles running the thread-per-level laplacians concurrently on two streams. The case matrices and the input
generators are those of tests/test_pointwise_cpu.py, where the same gate is shown to pass the FP64 restatement
everywhere and to fail on plausible fast-path defects that the field-normalised 1e-12 accepts."""
import numpy as np
import pytest

import tinman_sandbox_b200 as tb
from oracle import harness
from oracle import hp_reference as hp
from test_pointwise_cpu import (DIVWK_CASES, EULER_CASES, LAP_CASES, RHS_CASES, case_id, level_local_inputs,
                                make_state, rhs_case_state, rhs_reference)

pytestmark = pytest.mark.gpu
MODES = [tb.MODE_STRICT, tb.MODE_FAST]
MODE_NAME = {tb.MODE_STRICT: "strict", tb.MODE_FAST: "fast"}
WORST = {}   # (kernel, field) -> (ratio, index, |v|/M, case)
WORST_REL = {}   # (kernel, field) -> (|g-v|/|v|, index, |v|/M, ratio, case): where the largest relative error sits


def record(kernel, field, g, ref, K, case):
    r, at, vm = hp.worst(g, ref)
    if r >= WORST.get((kernel, field), (-1.0,))[0]:
        WORST[(kernel, field)] = (r, at, vm, case)
    v = ref.v.astype(np.float64)
    nz = v != 0
    if nz.any():
        rel = np.where(nz, np.abs(g - v) / np.where(nz, np.abs(v), 1.0), -1.0)
        i = np.unravel_index(int(np.argmax(rel)), rel.shape)
        if rel[i] >= WORST_REL.get((kernel, field), (-1.0,))[0]:
            WORST_REL[(kernel, field)] = (float(rel[i]), tuple(int(x) for x in i), float(abs(ref.v[i]) / ref.M[i]),
                                          float(hp.ratio(g[i], ref[i])), case)
    assert r <= K, (kernel, field, case, r, at, vm, K)


# ---- compute_and_apply_rhs ------------------------------------------------------------------------------------------

def run_rhs(s, hybi, ncalls, mode):
    h = tb.Caar(s.nelem, s.nlev, s.qsize_d, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    if hybi is not None:
        h.set_vertical_coordinate(0, hybi)
    h.set_control(*[int(x) for x in s.ctl], dt2=s.dt2)
    h.upload(s.arrays)
    h.compute_and_apply_rhs(ncalls, mode)
    h.download(s.arrays, names=None)
    h.close()


def check_rhs(got, base, ref, nlev, ncalls, kernel, case, lo=None, hi=None):
    lo = int(base.ctl[0]) if lo is None else lo
    hi = int(base.ctl[1]) if hi is None else hi
    for n in harness.FIELD_NAMES:
        g, b = got.arrays[n], base.arrays[n]
        if n not in harness.MUTATED:
            assert np.array_equal(g, b), n
            continue
        assert np.array_equal(g[:lo], b[:lo]) and np.array_equal(g[hi:], b[hi:]), (n, "outside [nets,nete)")
        record(kernel, n, g[lo:hi], ref.arrays[n][lo:hi], hp.k_rhs(nlev, ncalls), case)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("c", RHS_CASES, ids=case_id)
def test_rhs_pointwise(c, mode):
    s, hybi = rhs_case_state(c)
    ref = rhs_reference(s, 2, hybi)
    got = s.copy()
    run_rhs(got, hybi, 2, mode)
    kernel = f"rhs_{'eulerian' if hybi is not None else 'lagrangian'}_{MODE_NAME[mode]}"
    check_rhs(got, s, ref, c["nlev"], 2, kernel, case_id(c))


@pytest.mark.parametrize("mode", MODES)
def test_rhs_tail_of_a_large_handle(mode):
    """20000 elements, only the last 8 run and compared: TMA slice coordinates near the end of the arrays."""
    E, L, n = 20000, 72, 8
    tail = make_state("stratified", n, L, seed=20000)
    ref = rhs_reference(tail, 2, None)
    big = harness.PortOracle().init(E, L)
    for f in harness.FIELD_NAMES:
        big.arrays[f][E - n:] = tail.arrays[f]
    h = tb.Caar(E, L)
    h.set_params(tail.consts, tail.dvv, tail.ps0, tail.hyai)
    h.set_control(E - n, E, 0, 1, 2, 0, dt2=tail.dt2)
    h.upload(big.arrays)
    h.compute_and_apply_rhs(2, mode)
    before = h.download_range(E - 2 * n, E - n, names=harness.MUTATED)
    got = tail.copy()
    got.arrays.update(h.download_range(E - n, E, names=harness.FIELD_NAMES))
    h.close()
    for f in harness.MUTATED:
        assert np.array_equal(before[f], big.arrays[f][E - 2 * n:E - n]), f
    check_rhs(got, tail, ref, L, 2, f"rhs_lagrangian_{MODE_NAME[mode]}", "tail E=20000")


# ---- tracer step ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("c", EULER_CASES, ids=case_id)
def test_euler_step_pointwise(c, mode):
    E, L, Q = 9, c["nlev"], 35
    s, vstar, _, _ = level_local_inputs(c["gen"], E, L, c["seed"], qsize_d=Q)
    s.ctl[0:2] = (1, E - 1)
    dt, qsize = 150.0, c["qsize"]
    ref = hp.euler_step(hp.from_state(s), vstar, c["qn0"], qsize, dt)
    h = tb.Caar(E, L, Q)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.set_control(*[int(x) for x in s.ctl], dt2=s.dt2)
    h.upload(s.arrays)
    h.upload_vstar(vstar)
    h.upload_extra(tb.X_QTENS, np.full((E, Q, L, 4, 4), -7.0))
    h.euler_step(c["qn0"], qsize, dt, mode)
    got = h.download_qtens()
    h.close()
    assert np.all(got[0] == -7.0) and np.all(got[E - 1] == -7.0) and np.all(got[:, qsize:] == -7.0)
    record(f"euler_step_{MODE_NAME[mode]}", "qtens", got[1:E - 1, :qsize], ref[1:E - 1, :qsize], hp.K_EULER, case_id(c))


# ---- weak-form operators --------------------------------------------------------------------------------------------

def _wk_handle(s, vin, sin, tv):
    h = tb.Caar(s.nelem, s.nlev)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays)
    h.upload_extra(tb.X_VSTAR, vin)
    h.upload_extra(tb.X_SCALAR_IN, sin)
    h.upload_extra(tb.X_TENSORVISC, tv)
    return h


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("c", DIVWK_CASES, ids=case_id)
def test_divergence_sphere_wk_pointwise(c, mode):
    E, L = 9, c["nlev"]
    s, vin, sin, tv = level_local_inputs(c["gen"], E, L, c["seed"])
    ref = hp.sphere_wk("divergence_sphere_wk", hp.from_state(s), vin, None, 1, E - 2)
    h = _wk_handle(s, vin, sin, tv)
    h.upload_extra(tb.X_SCALAR_OUT, np.full((E, L, 4, 4), -7.0))
    h.sphere_wk(tb.OP_DIVERGENCE_WK, mode, nets=1, nete=E - 2)
    got = h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4))
    h.close()
    assert np.all(got[0] == -7.0) and np.all(got[E - 2:] == -7.0)
    record(f"divergence_sphere_wk_{MODE_NAME[mode]}", "out", got[1:E - 2], ref[1:E - 2], hp.K_DIVWK, case_id(c))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("c", LAP_CASES, ids=case_id)
def test_laplacians_pointwise(c, mode):
    """laplace_simple / laplace_tensor on a sub-range with nets > 0 (sentinel around it), then laplace_tensor_replace in
    place on another sub-range. nlev 5 and 13 run on the groups-of-8 kernel, 16 and up on the 32-row flat tiles."""
    E, L = c["E"], c["nlev"]
    s, vin, sin, tv = level_local_inputs(c["gen"], E, L, c["seed"])
    hs = hp.from_state(s)
    h = _wk_handle(s, vin, sin, tv)
    kind = ("flat" if L >= 16 else "levelop") if mode == tb.MODE_FAST else "strict"
    for op, name, K in ((tb.OP_LAPLACE_SIMPLE, "laplace_simple", hp.K_LAPLACE_SIMPLE),
                        (tb.OP_LAPLACE_TENSOR, "laplace_tensor", hp.K_LAPLACE_TENSOR)):
        ref = hp.sphere_wk(name, hs, sin, tv, 2, E - 1)
        h.upload_extra(tb.X_SCALAR_OUT, np.full((E, L, 4, 4), -7.0))
        h.sphere_wk(op, mode, nets=2, nete=E - 1)
        got = h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4))
        assert np.all(got[:2] == -7.0) and np.all(got[E - 1:] == -7.0), name
        record(f"{name}_{kind}", "out", got[2:E - 1], ref[2:E - 1], K, case_id(c))
    ref = hp.sphere_wk("laplace_tensor", hs, sin, tv, 1, E - 2)
    h.upload_extra(tb.X_SCALAR_OUT, sin)
    h.sphere_wk(tb.OP_LAPLACE_TENSOR_REPLACE, mode, nets=1, nete=E - 2)
    got = h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4))
    h.close()
    assert np.array_equal(got[:1], sin[:1]) and np.array_equal(got[E - 2:], sin[E - 2:])
    record(f"laplace_tensor_replace_{kind}", "out", got[1:E - 2], ref[1:E - 2], hp.K_LAPLACE_TENSOR,
           case_id(c))


# ---- two handles, two streams ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("E,L", [(48, 40), (8192, 72)])
def test_concurrent_laplacians_on_two_streams(E, L):
    """laplace_simple on one handle and laplace_tensor on another, each on its own torch stream, queued without
    synchronisation so that they overlap, must both give the solo results. The thread-per-level laplacians hand out
    tiles from a counter pair that every launch leaves at zero; two launches that overlap must never share one. Each of
    the 256 rounds adds one more laplace_tensor launch on the first handle (whose output laplace_simple must then
    overwrite completely), so any pairing of counters that depends on launch counts is met. Afterwards 512 launches of
    each op, alternating on one handle and each checked, show that no launch left its counters dirty.
    48 x 40: both grids fit on the device side by side; 8192 x 72: more tiles than the resident warps take in their
    first chunks, so the counter is really drawn from."""
    import torch
    s1, _, f1, _ = level_local_inputs("stratified", E, L, seed=E + 1)
    s2, _, f2, tv = level_local_inputs("randomize", E, L, seed=E + 2)
    h1, h2 = (_wk_handle(s, np.zeros((E, L, 4, 4, 2)), f, tv) for s, f in ((s1, f1), (s2, f2)))
    st1, st2 = torch.cuda.Stream(), torch.cuda.Stream()
    h1.set_stream(st1.cuda_stream)
    h2.set_stream(st2.cuda_stream)
    shape = (E, L, 4, 4)

    def solo(h, op):
        h.sphere_wk(op, tb.MODE_FAST)
        return h.download_extra(tb.X_SCALAR_OUT, shape)

    want = {"s1": solo(h1, tb.OP_LAPLACE_SIMPLE), "t1": solo(h1, tb.OP_LAPLACE_TENSOR),
            "t2": solo(h2, tb.OP_LAPLACE_TENSOR)}
    for name, s, f, key in (("laplace_simple", s1, f1, "s1"), ("laplace_tensor", s1, f1, "t1"),
                            ("laplace_tensor", s2, f2, "t2")):
        for lo in range(0, E, 512):                   # the reference in slices of elements: bounded memory
            hi = min(lo + 512, E)
            sub = harness.State(hi - lo, L, ctl=s.ctl, dt2=s.dt2, consts=s.consts, dvv=s.dvv, ps0=s.ps0, hyai=s.hyai,
                                arrays={n: s.arrays[n][lo:hi] for n in ("elem_Dinv", "elem_spheremp")})
            ref = hp.sphere_wk(name, hp.from_state(sub), f[lo:hi], tv[lo:hi], 0, hi - lo)
            record(f"{name}_flat_fast", "out", want[key][lo:hi], ref, hp.K_SPHERE_WK[name], f"two streams {E}x{L}")
    sentinel = np.full(shape, -7.0)
    bad = []
    for it in range(256):
        h2.upload_extra(tb.X_SCALAR_OUT, sentinel)
        h1.sphere_wk(tb.OP_LAPLACE_TENSOR, tb.MODE_FAST, sync=False)      # the extra launch of this round
        h1.sphere_wk(tb.OP_LAPLACE_SIMPLE, tb.MODE_FAST, sync=False)
        h2.sphere_wk(tb.OP_LAPLACE_TENSOR, tb.MODE_FAST, sync=False)
        h1.sync()
        h2.sync()
        ok1 = np.array_equal(h1.download_extra(tb.X_SCALAR_OUT, shape), want["s1"])
        ok2 = np.array_equal(h2.download_extra(tb.X_SCALAR_OUT, shape), want["t2"])
        if not (ok1 and ok2):
            bad.append((it, ok1, ok2))
    seq_bad = []
    for it in range(1024):
        op, key = (tb.OP_LAPLACE_SIMPLE, "s1") if it % 2 else (tb.OP_LAPLACE_TENSOR, "t1")
        h1.sphere_wk(op, tb.MODE_FAST)
        if not np.array_equal(h1.download_extra(tb.X_SCALAR_OUT, shape), want[key]):
            seq_bad.append(it)
    h1.set_stream(0)
    h2.set_stream(0)
    h1.close()
    h2.close()
    assert not bad and not seq_bad, (f"{len(bad)} of 256 concurrent rounds wrong, first {bad[:4]}; "
                                     f"{len(seq_bad)} of 1024 sequential launches wrong, first {seq_bad[:4]}")


def test_zz_report_pointwise(capsys):
    """Not a gate: per kernel and field, the worst |g - v| / (u M) of this session and where it sits, and the point of
    the largest relative error |g - v| / |v| with |v| / M there (|v| / M << 1: cancellation, M >> |v|). Indices are
    into the compared slice: [element][time level][level][i][j][component] for the state arrays, [element][level]...
    for the others, [element][tracer][level][i][j] for qtens."""
    with capsys.disabled():
        for (k, n), (r, at, vm, case) in sorted(WORST.items()):
            print(f"\n[pointwise] {k:36s} {n:26s} worst ratio {r:8.3f} at {at} |v|/M {vm:.2e} ({case})", end="")
        for (k, n), (rel, at, vm, r, case) in sorted(WORST_REL.items()):
            print(f"\n[relative]  {k:36s} {n:26s} max |g-v|/|v| {rel:.2e} at {at} |v|/M {vm:.2e} ratio {r:.3f} ({case})",
                  end="")
        print()
