"""The level-local kernels in the regimes their persistent warps reach in production, against the extended-precision
reference (oracle/hp_reference.py) with the pointwise gate |g - v| <= K u M.

The steady-state matrix (CASES of tests/test_levelop_regimes_cpu.py): tracer step (T), fast and strict;
divergence_sphere_wk (D); the row-decomposed laplacians (R, nlev < 16); the flat laplacians (F, chunk 4). Each case must
reach its regime on this device (the test fails, not skips, when it does not). Fast mode is checked pointwise; strict mode
must equal the FP64 restatement (PortOracle) bit for bit. Rows outside the element range and tracers past qsize must
keep their -7 sentinel. F2 and F3 then queue 50 flat-laplacian launches over random element ranges into one buffer,
which must equal, bit for bit, the element-wise composition of whole-handle launches.

The report (test_zz_report_regimes) prints, per kernel and case, the regime, the worst ratio against K and where the
worst point sits in the work distribution: (warp, unit) for levelop_kernel, (tile, chunk) for the flat laplacians."""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
from oracle import harness
from oracle import hp_reference as hp
from test_levelop_regimes_cpu import (CASES, FT, GL, case_regime, hp_slice, lean_inputs, levelop_unit_warp, missed,
                                      sub_state)

pytestmark = pytest.mark.gpu
DT = 150.0
REPORT = []          # lines of the final report
LAP_OPS = (("laplace_simple", tb.OP_LAPLACE_SIMPLE, hp.K_LAPLACE_SIMPLE),
           ("laplace_tensor", tb.OP_LAPLACE_TENSOR, hp.K_LAPLACE_TENSOR))
RANDOM_RANGES = ("F2", "F3")  # flat laplacian cases at chunk 4 that also run the random-range composition check


# ---- running a job on the device -------------------------------------------------------------------------------------

def _handle(s, E, L, Q, names):
    h = tb.Caar(E, L, Q)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays, names=names)
    return h


def job_inputs(j):
    """The lean inputs of a job (deterministic in its parameters)."""
    op = j["op"]
    return lean_inputs(j["gen"], j["E"], j["nlev"], j["seed"], Q=j["Q"] if op == "euler" else 0, qn0=j["qn0"],
                       qsize=j["qsize"], vector=op in ("euler", "divwk"), scalar=op not in ("euler", "divwk"))


def run_job(j, inputs=None):
    """-> dict of output arrays. j: a case of CASES plus "mode"."""
    s, vin, sin, tv = inputs or job_inputs(j)
    E, L, (lo, hi), mode = j["E"], j["nlev"], j["range"], j["mode"]
    if j["op"] == "euler":
        Q = j["Q"]
        h = _handle(s, E, L, Q, ("elem_Dinv", "elem_metdet", "elem_rmetdet", "elem_state_Qdp"))
        h.upload_vstar(vin)
        h.upload_extra(tb.X_QTENS, np.full((E, Q, L, 4, 4), -7.0))
        h.euler_step(j["qn0"], j["qsize"], DT, mode, nets=lo, nete=hi)
        out = {"qtens": h.download_qtens()}
        h.close()
        return out
    h = _handle(s, E, L, 1, ("elem_Dinv", "elem_spheremp"))
    shape = (E, L, 4, 4)
    sentinel = np.full(shape, -7.0)
    out = {}
    if j["op"] == "divwk":
        h.upload_extra(tb.X_VSTAR, vin)
        h.upload_extra(tb.X_SCALAR_OUT, sentinel)
        h.sphere_wk(tb.OP_DIVERGENCE_WK, mode, nets=lo, nete=hi)
        out["divergence_sphere_wk"] = h.download_extra(tb.X_SCALAR_OUT, shape)
        h.close()
        return out
    h.upload_extra(tb.X_SCALAR_IN, sin)
    h.upload_extra(tb.X_TENSORVISC, tv)
    for name, op, _ in LAP_OPS:
        h.upload_extra(tb.X_SCALAR_OUT, sentinel)
        h.sphere_wk(op, mode, nets=lo, nete=hi)
        out[name] = h.download_extra(tb.X_SCALAR_OUT, shape)
    h.upload_extra(tb.X_SCALAR_OUT, sin)
    h.sphere_wk(tb.OP_LAPLACE_TENSOR_REPLACE, mode, nets=lo, nete=hi)
    out["laplace_tensor_replace"] = h.download_extra(tb.X_SCALAR_OUT, shape)
    h.close()
    return out


def lap_buffers(c, inputs, runs):
    """One handle on a case's inputs; per run, a sentinel-filled output buffer and the run's fast-mode (op, nets, nete)
    launches queued without synchronisation -> the buffers after each run."""
    s, _, sin, tv = inputs
    E, L = c["E"], c["nlev"]
    h = _handle(s, E, L, 1, ("elem_Dinv", "elem_spheremp"))
    h.upload_extra(tb.X_SCALAR_IN, sin)
    h.upload_extra(tb.X_TENSORVISC, tv)
    out = []
    for launches in runs:
        h.upload_extra(tb.X_SCALAR_OUT, np.full((E, L, 4, 4), -7.0))
        for op, a, b in launches:
            h.sphere_wk(op, tb.MODE_FAST, nets=a, nete=b, sync=False)
        h.sync()
        out.append(h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4)))
    h.close()
    return out


def check_random_ranges(c, inputs, fast):
    """50 launches over seeded random element ranges, alternating laplace_simple and laplace_tensor, queued into one
    sentinel-filled buffer: a tile-scheduler counter left non-zero by one launch would make the next skip tiles. A row
    of the flat laplacians depends only on its own element's data and geometry, so every element must hold, bit for
    bit, the whole-handle [0, E) output of the op of the last launch that covered it, and the sentinel if none did."""
    E = c["E"]
    rng = np.random.default_rng(c["seed"] + 1)
    launches = []
    for n in range(50):
        a = int(rng.integers(0, E - 1))
        launches.append((LAP_OPS[n % 2], a, int(rng.integers(a + 1, E + 1))))
    whole = fast
    if c["range"] != (0, E):  # the tested range (F2: from element 1) is not the whole handle
        whole = dict(zip([name for name, _, _ in LAP_OPS],
                         lap_buffers(c, inputs, [[(op, 0, E)] for _, op, _ in LAP_OPS])))
    got, = lap_buffers(c, inputs, [[(op, a, b) for (_, op, _), a, b in launches]])
    want = np.full(got.shape, -7.0)
    for (name, _, _), a, b in launches:
        want[a:b] = whole[name][a:b]
    same = np.array_equal(got, want)
    REPORT.append(f"{'laplace_flat random ranges':30s} {c['id']:4s} 50 launches "
                  f"{'bit-identical to' if same else 'DIFFER from'} the composition of whole-handle launches")
    assert same, (c["id"], "elements that differ", np.flatnonzero(np.any(got != want, axis=(1, 2, 3)))[:20])


# ---- gating and reporting -------------------------------------------------------------------------------------------

def locate(c, idx, sms):
    """Where a point of a case's output sits in the work distribution (at the ptxas occupancy)."""
    lo, L = c["range"][0], c["nlev"]
    r = case_regime(c, sms)
    if c["op"] == "lap_flat":
        tile = ((idx[0] - lo) * L + idx[1]) // FT
        ch = tile // r["chunk"]
        return f"tile {tile}, chunk {ch}" + (f" (first chunk of warp {ch})" if ch < r["warps"] else " (drawn)")
    ng = -(-L // GL)
    if c["op"] == "euler":
        unit = ((idx[0] - lo) * ng + idx[2] // GL) * c["qsize"] + idx[1]
    else:
        unit = (idx[0] - lo) * ng + idx[1] // GL
    w = levelop_unit_warp(r["units"], r["warps"], unit)
    return f"warp {w}, unit {unit - r['units'] * w // r['warps']} of {r['per_warp']:.0f}"


def _worst_of_slice(task):
    """hp.worst of one slice of elements: (name, lean sub-state, field, tensorVisc, qn0, qsize, result slice)."""
    name, sub, field, tv, qn0, qsize, got = task
    ref = hp_slice(name, sub, 0, sub.nelem, field, tv, qn0=qn0, qsize=qsize)
    return hp.worst(got, ref[:, :qsize] if name == "euler_step" else ref)


_POOL = []


def pool():
    """Worker processes for the reference (numpy only, no device): spawned, shut down when the session ends."""
    if not _POOL:
        _POOL.append(ProcessPoolExecutor(max_workers=max(1, min(16, (os.cpu_count() or 2) - 1)),
                                         mp_context=multiprocessing.get_context("spawn")))
    return _POOL[0]


@pytest.fixture(scope="module", autouse=True)
def _shutdown_pool():
    yield
    while _POOL:
        _POOL.pop().shutdown()


def gate_sliced(kernel, c, got, name, inputs, K, sms, qn0=0, qsize=0):
    """The pointwise gate over [nets,nete) of `got` (elements first); the extended-precision reference of `name` is
    computed in slices of elements, in parallel."""
    lo, hi = c["range"]
    s, field, tv = inputs
    per_elem = int(np.prod(got.shape[1:]))
    step = max(1, 1_000_000 // per_elem)
    tasks = ((name, sub_state(s, a, min(a + step, hi)), field[a:a + step], None if tv is None else tv[a:a + step], qn0,
              qsize, got[a:min(a + step, hi)]) for a in range(lo, hi, step))
    worst = (-1.0, None, None)
    for a, (r, at, vm) in zip(range(lo, hi, step), pool().map(_worst_of_slice, tasks)):
        if r > worst[0]:
            worst = (r, (at[0] + a,) + at[1:], vm)
    r, at, vm = worst
    REPORT.append(f"{kernel:30s} {c['id']:4s} worst ratio {r:7.3f} (K {K}) at {at}, |v|/M {vm:.1e}, "
                  f"{locate(c, at, sms)}")
    assert r <= K, (kernel, c["id"], r, at, vm, locate(c, at, sms))


def check_sentinel(c, got, name="", sin=None):
    """Outside [nets,nete) the output keeps its -7 sentinel (laplace_tensor_replace: its input)."""
    lo, hi = c["range"]
    keep = sin if name == "laplace_tensor_replace" else np.full(got.shape, -7.0)
    assert np.array_equal(got[:lo], keep[:lo]) and np.array_equal(got[hi:], keep[hi:]), (c["id"], name, "outside")
    if c["op"] == "euler":
        assert np.all(got[:, c["qsize"]:] == -7.0), (c["id"], "tracers past qsize")


def port_reference(c, s, vin, sin, tv):
    """The FP64 restatement (PortOracle, C) of a case: what strict mode must equal bit for bit."""
    lo, hi = c["range"]
    orc = harness.PortOracle()
    if c["op"] == "euler":
        s.ctl[0:2] = (lo, hi)
        want = np.zeros((c["E"], c["Q"], c["nlev"], 4, 4))
        orc.euler_step(s, vin, want, c["qn0"], c["qsize"], DT)
        return {"qtens": want}
    if c["op"] == "divwk":
        return {"divergence_sphere_wk": orc.sphere_wk("divergence_sphere_wk", s, vin, None, lo, hi)}
    return {name: orc.sphere_wk(name, s, sin, tv if name == "laplace_tensor" else None, lo, hi)
            for name, _, _ in LAP_OPS}


def gate_fast(c, got, inputs, sms):
    """Every fast-mode output of a case against the reference; laplace_tensor_replace bit-equal to laplace_tensor."""
    s, vin, sin, tv = inputs
    q = c["qsize"]
    kind = {"euler": "euler_step", "divwk": "divergence_sphere_wk", "lap_rows": "levelop", "lap_flat": "flat"}[c["op"]]
    if c["op"] == "euler":
        gate_sliced("euler_step_fast", c, got["qtens"][:, :q], "euler_step", (s, vin, None), hp.K_EULER, sms,
                    qn0=c["qn0"], qsize=q)
    elif c["op"] == "divwk":
        gate_sliced("divergence_sphere_wk_fast", c, got[kind], kind, (s, vin, None), hp.K_DIVWK, sms)
    else:
        for name, _, K in LAP_OPS:
            gate_sliced(f"{name}_{kind}", c, got[name], name, (s, sin, tv), K, sms)
        lo, hi = c["range"]
        assert np.array_equal(got["laplace_tensor_replace"][lo:hi], got["laplace_tensor"][lo:hi]), c["id"]


def device_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- the steady-state matrix -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("c", CASES, ids=lambda c: c["id"])
def test_steady_state_matrix(c):
    sms = device_sms()
    r = case_regime(c, sms)
    assert not missed(c, r), f"{c['id']} misses its regime on {sms} SMs: {missed(c, r)} ({r})"
    inputs = job_inputs(c)
    strict = run_job(dict(c, mode=tb.MODE_STRICT), inputs)
    want = port_reference(c, *inputs)
    for name, g in strict.items():
        check_sentinel(c, g, name, inputs[2])
        w = want.get(name, want.get("laplace_tensor"))
        lo, hi = c["range"]
        assert np.array_equal(g[lo:hi, :c["qsize"]] if c["op"] == "euler" else g[lo:hi],
                              w[lo:hi, :c["qsize"]] if c["op"] == "euler" else w[lo:hi]), (c["id"], name, "strict")
    REPORT.append(f"{c['op'] + '_strict':30s} {c['id']:4s} bit-identical to the FP64 restatement "
                  f"({', '.join(f'{k} {v:.3g}' for k, v in r.items())})")
    fast = run_job(dict(c, mode=tb.MODE_FAST), inputs)
    for name, g in fast.items():
        check_sentinel(c, g, name, inputs[2])
    gate_fast(c, fast, inputs, sms)
    if c["id"] in RANDOM_RANGES:
        check_random_ranges(c, inputs, fast)


def test_zz_report_regimes(capsys):
    """Not a gate: what the tests above measured, per kernel and case."""
    with capsys.disabled():
        for line in REPORT:
            print(f"\n[regimes] {line}", end="")
        print()

