"""The level-local kernels in the regimes their persistent warps reach in production, against the extended-precision
reference (oracle/hp_reference.py) with the pointwise gate |g - v| <= K u M, and under every launch knob of DESIGN §7b.

1. The steady-state matrix (CASES of tests/test_levelop_regimes_cpu.py) at default knobs: tracer step (T), fast and
   strict; divergence_sphere_wk (D); the row-decomposed laplacians (R, nlev < 16); the flat laplacians (F, chunk 4).
   Each case must reach its regime on this device (the test fails, not skips, when it does not). Fast mode is gated
   pointwise; strict mode must equal the FP64 restatement (PortOracle) bit for bit. Rows outside the element range and
   tracers past qsize must keep their -7 sentinel.
2. Knob legs. Every knob is read once per process into a `static`, so each setting runs in a child process
   (`python tests/test_levelop_regimes_gpu.py --knob-worker SPEC`) that loads the library fresh, runs its jobs and
   writes .npz files; the parent computes the same jobs in process at default knobs and gates the child's results.
   Knobs that only change the schedule must leave the results bit-identical; the two that select other arithmetic
   (CAAR_LAPLACE_V1, CAAR_EULER_V1) are gated pointwise.

The report (test_zz_report_regimes) prints, per kernel, case and knob, the regime, the worst ratio against K and
where the worst point sits in the work distribution: (warp, unit) for levelop_kernel, (tile, chunk) for the flat
laplacians."""
import json
import multiprocessing
import os
import subprocess
import sys
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

if __name__ == "__main__":                          # knob worker: the repository and tests/ on the path
    _HERE = os.path.dirname(os.path.abspath(__file__))
    sys.path[:0] = [os.path.dirname(_HERE), _HERE]

import tinman_sandbox_b200 as tb  # noqa: E402
from oracle import harness  # noqa: E402
from oracle import hp_reference as hp  # noqa: E402
from test_levelop_regimes_cpu import (CASES, FT, GL, case_regime, hp_slice, lean_inputs, levelop_unit_warp,  # noqa: E402
                                      missed, regime, sub_state)
from test_pointwise_cpu import TLS, rhs_case_state  # noqa: E402

pytestmark = pytest.mark.gpu
DT = 150.0
KNOBS = ("CAAR_LEVELOP_WAVES", "CAAR_LAPLACE_CHUNK", "CAAR_LAPLACE_V1", "CAAR_EULER_V1", "CAAR_EULER_WAVES",
         "CAAR_CLUSTER_POLICY", "CAAR_PF_DIST")
REPORT = []          # lines of the final report
LAP_OPS = (("laplace_simple", tb.OP_LAPLACE_SIMPLE, hp.K_LAPLACE_SIMPLE),
           ("laplace_tensor", tb.OP_LAPLACE_TENSOR, hp.K_LAPLACE_TENSOR))


# ---- running a job on the device (in process, or in a knob worker) -------------------------------------------------

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
    """-> dict of output arrays. j: a case of CASES (plus "mode"), or a "rhs" job (fused kernel on an RHS_CASES-style
    state). "ranges": after the first run, that many more launches of the laplacians over random element ranges,
    queued without synchronisation; the output is the buffer after the last."""
    if j["op"] == "rhs":
        s, hybi = rhs_case_state(j)
        h = tb.Caar(s.nelem, s.nlev, s.qsize_d, s.ntl)
        h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
        if hybi is not None:
            h.set_vertical_coordinate(0, hybi)
        h.set_control(*[int(x) for x in s.ctl], dt2=s.dt2)
        h.upload(s.arrays)
        h.compute_and_apply_rhs(2, j["mode"])
        h.download(s.arrays, names=harness.MUTATED)
        h.close()
        return {n: s.arrays[n] for n in harness.MUTATED}
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
    if j.get("ranges"):
        rng = np.random.default_rng(j["seed"] + 1)
        h.upload_extra(tb.X_SCALAR_OUT, sentinel)
        for n in range(j["ranges"]):
            a = int(rng.integers(0, E - 1))
            b = int(rng.integers(a + 1, E + 1))
            h.sphere_wk(LAP_OPS[n % 2][1], mode, nets=a, nete=b, sync=False)
        h.sync()
        out["random_ranges"] = h.download_extra(tb.X_SCALAR_OUT, shape)
    h.close()
    return out


# ---- gating and reporting -------------------------------------------------------------------------------------------

def locate(c, idx, sms):
    """Where a point of a case's output sits in the work distribution (at the ptxas occupancy)."""
    lo, L = c["range"][0], c["nlev"]
    if c.get("v1"):                                     # euler_step_kernel: groups of 64 rows, grid-stride
        return f"row group {((idx[0] - lo) * L + idx[2]) // 64}"
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


def gate_sliced(kernel, c, got, name, inputs, K, knob, sms, qn0=0, qsize=0):
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
    REPORT.append(f"{kernel:30s} {c['id']:4s} {knob:34s} worst ratio {r:7.3f} (K {K}) at {at}, |v|/M {vm:.1e}, "
                  f"{locate(c, at, sms)}")
    assert r <= K, (kernel, c["id"], knob, r, at, vm, locate(c, at, sms))


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


def gate_fast(c, got, inputs, knob, sms, tag=""):
    """Every fast-mode output of a case against the reference; laplace_tensor_replace bit-equal to laplace_tensor."""
    s, vin, sin, tv = inputs
    q = c["qsize"]
    kind = {"euler": "euler_step", "divwk": "divergence_sphere_wk", "lap_rows": "levelop", "lap_flat": "flat"}[c["op"]]
    if c["op"] == "euler":
        gate_sliced(f"euler_step_fast{tag}", c, got["qtens"][:, :q], "euler_step", (s, vin, None), hp.K_EULER, knob,
                    sms, qn0=c["qn0"], qsize=q)
    elif c["op"] == "divwk":
        gate_sliced("divergence_sphere_wk_fast", c, got[kind], kind, (s, vin, None), hp.K_DIVWK, knob, sms)
    else:
        for name, _, K in LAP_OPS:
            gate_sliced(f"{name}_{kind}", c, got[name], name, (s, sin, tv), K, knob, sms)
        lo, hi = c["range"]
        assert np.array_equal(got["laplace_tensor_replace"][lo:hi], got["laplace_tensor"][lo:hi]), (c["id"], knob)


def device_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def default_knobs():
    """The in-process runs are the default-knob runs: none of the knobs may be set for this process."""
    set_ = [k for k in KNOBS if k in os.environ]
    assert not set_, f"run without {set_}: the in-process results stand for the default knobs"


# ---- 1. the steady-state matrix at default knobs --------------------------------------------------------------------

@pytest.mark.parametrize("c", CASES, ids=lambda c: c["id"])
def test_steady_state_matrix(c, default_knobs):
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
    REPORT.append(f"{c['op'] + '_strict':30s} {c['id']:4s} {'default':34s} bit-identical to the FP64 restatement "
                  f"({', '.join(f'{k} {v:.3g}' for k, v in r.items())})")
    fast = run_job(dict(c, mode=tb.MODE_FAST), inputs)
    for name, g in fast.items():
        check_sentinel(c, g, name, inputs[2])
    gate_fast(c, fast, inputs, "default", sms)


# ---- 2. knob legs in child processes --------------------------------------------------------------------------------

def _by_id(cid):
    return next(c for c in CASES if c["id"] == cid)


def _shrunk(cid, E, **kw):
    c = dict(_by_id(cid), E=E, range=(0, E))
    c.update(kw, id=f"{cid}@{E}")
    return c


def _rhs_jobs():
    jobs = []
    for i, (L, eul) in enumerate(((30, False), (72, False), (96, False), (128, False), (72, True))):
        for mode in (tb.MODE_STRICT, tb.MODE_FAST):
            E = 600
            jobs.append(dict(id=f"rhs{'_eul' if eul else ''}{L}_{'strict' if mode else 'fast'}", op="rhs", nlev=L,
                             eulerian=eul, gen=("stratified", "randomize")[i % 2], tls=TLS[i % 3], qn0=(i % 3) - 1,
                             E=E, range=(2, E - 1) if i % 2 else (0, E), seed=9000 + i, mode=mode))
    return jobs


T2, D1 = _by_id("T2"), _by_id("D1")
LAP_CHUNK_JOBS = [dict(_shrunk("F2", 4096, range=(1, 4096)), ranges=50), dict(_shrunk("F3", 4096), ranges=50)]
SCHEDULE_JOBS = ([dict(T2, mode=tb.MODE_FAST, id="T2_fast"), dict(T2, mode=tb.MODE_STRICT, id="T2_strict"),
                  dict(D1, mode=tb.MODE_FAST, id="D1_fast")]
                 + [dict(j, mode=tb.MODE_FAST, id=j["id"] + "_fast") for j in LAP_CHUNK_JOBS] + _rhs_jobs())
# the row decomposition for every nlev: about 24000 units, 10 per warp
LAP_V1_JOBS = [dict(_shrunk("F1", E, nlev=L), mode=tb.MODE_FAST) for L, E in ((16, 12000), (30, 6000), (72, 2700),
                                                                             (128, 1500))]
EULER_V1_JOB = dict(_by_id("T2"), id="V1", E=1200, range=(0, 1200), Q=5, qsize=5, qn0=0, gen="stratified",
                    mode=tb.MODE_FAST, v1=True)
for _j in LAP_V1_JOBS:
    _j["id"] = f"V1_L{_j['nlev']}"

# Schedule-only knob values are combined into three children: each knob is read by one kernel only.
SCHEDULE_LEGS = [
    {"CAAR_LEVELOP_WAVES": "1", "CAAR_LAPLACE_CHUNK": "1", "CAAR_EULER_WAVES": "1", "CAAR_CLUSTER_POLICY": "1",
     "CAAR_PF_DIST": "0"},
    {"CAAR_LEVELOP_WAVES": "16", "CAAR_LAPLACE_CHUNK": "3", "CAAR_EULER_WAVES": "0", "CAAR_CLUSTER_POLICY": "2",
     "CAAR_PF_DIST": "1"},
    {"CAAR_LEVELOP_WAVES": "200", "CAAR_LAPLACE_CHUNK": "64", "CAAR_PF_DIST": str(600 + 5)},
]
ARITHMETIC_LEGS = [
    ({"CAAR_LAPLACE_V1": "1", "CAAR_EULER_V1": "1", "CAAR_EULER_WAVES": "1"}, LAP_V1_JOBS + [EULER_V1_JOB]),
    ({"CAAR_EULER_V1": "1", "CAAR_EULER_WAVES": "2"}, [EULER_V1_JOB]),
    ({"CAAR_EULER_V1": "1", "CAAR_EULER_WAVES": "0"}, [EULER_V1_JOB]),
]


def run_worker(env_knobs, jobs, tmp_path, tag):
    """One child process with the knobs set: -> {job id: {name: array}}."""
    out = tmp_path / tag
    out.mkdir()
    spec = tmp_path / f"{tag}.json"
    spec.write_text(json.dumps({"out": str(out), "jobs": jobs}))
    env = {k: v for k, v in os.environ.items() if k not in KNOBS}
    env.update(env_knobs)
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--knob-worker", str(spec)], env=env,
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, f"knob worker {env_knobs} failed:\n{p.stdout[-3000:]}\n{p.stderr[-3000:]}"
    res = {}
    for j in jobs:
        with np.load(out / f"{j['id']}.npz") as z:
            res[j["id"]] = {k: z[k] for k in z.files}
    return res


def knob_str(env_knobs, kernel_knobs):
    return ",".join(f"{k[5:]}={v}" for k, v in env_knobs.items() if k in kernel_knobs) or "default"


KNOBS_OF = {"euler_fast": ("CAAR_LEVELOP_WAVES",), "euler_strict": ("CAAR_EULER_WAVES",),
            "divwk": ("CAAR_LEVELOP_WAVES",), "lap_flat": ("CAAR_LAPLACE_CHUNK",),
            "rhs": ("CAAR_CLUSTER_POLICY", "CAAR_PF_DIST")}


def test_schedule_knobs_are_bit_identical(tmp_path, default_knobs):
    """CAAR_LEVELOP_WAVES 1 / 16 / 200 (tracer step T2, divergence_sphere_wk D1: about 124 units per warp down to
    one), CAAR_LAPLACE_CHUNK 1 / 3 / 64 (F2 and F3 shapes at 4096 elements, then 50 launches over random ranges
    queued without synchronisation: a scheduler counter left non-zero skips tiles of the next launch),
    CAAR_EULER_WAVES 1 / 0 (strict tracer step T2, which must also still equal the FP64 restatement),
    CAAR_CLUSTER_POLICY 1 / 2 and CAAR_PF_DIST 0 / 1 / E + 5 (the fused kernel, both modes, nlev 30, 72, 96, 128 and
    Eulerian 72 at 600 elements) change who computes what, never a result."""
    want = {j["id"]: run_job(j) for j in SCHEDULE_JOBS}
    s, vin, _, _ = job_inputs(T2)
    port = port_reference(T2, s, vin, None, None)["qtens"]
    assert np.array_equal(want["T2_strict"]["qtens"][:, :T2["qsize"]], port[:, :T2["qsize"]])
    bad = []
    for n, env_knobs in enumerate(SCHEDULE_LEGS):
        got = run_worker(env_knobs, SCHEDULE_JOBS, tmp_path, f"schedule{n}")
        for j in SCHEDULE_JOBS:
            key = "rhs" if j["op"] == "rhs" else ("euler_strict" if j["id"] == "T2_strict" else
                                                 "euler_fast" if j["op"] == "euler" else j["op"])
            same = all(np.array_equal(got[j["id"]][k], v) for k, v in want[j["id"]].items())
            REPORT.append(f"{j['id']:30s} {'':4s} {knob_str(env_knobs, KNOBS_OF[key]):34s} "
                          f"{'bit-identical to the default knobs' if same else 'DIFFERS from the default knobs'}")
            if not same:
                bad.append((j["id"], env_knobs))
        assert np.array_equal(got["T2_strict"]["qtens"][:, :T2["qsize"]], port[:, :T2["qsize"]]), env_knobs
    assert not bad, bad


def test_arithmetic_knobs_pass_the_pointwise_gate(tmp_path, default_knobs):
    """CAAR_LAPLACE_V1=1 runs the row-decomposed laplacians at nlev 16, 30, 72 and 128 (about 10 units per warp);
    CAAR_EULER_V1=1 the first-generation tracer step at nlev 72, qsize_d = qsize = 5 (odd: the remainder of its
    unroll by two), with CAAR_EULER_WAVES 1, 2 and 0. Each is gated pointwise; the three V1 tracer runs, which differ
    in their grid only, must also agree bit for bit."""
    sms = device_sms()
    v1_runs = []
    for n, (env_knobs, jobs) in enumerate(ARITHMETIC_LEGS):
        got = run_worker(env_knobs, jobs, tmp_path, f"arith{n}")
        for j in jobs:
            g = got[j["id"]]
            if j["op"] == "euler":
                check_sentinel(j, g["qtens"])
                v1_runs.append(g["qtens"])
                knob = knob_str(env_knobs, ("CAAR_EULER_V1", "CAAR_EULER_WAVES"))
                gate_fast(j, g, job_inputs(j), knob, sms, tag="_v1")
            else:
                inputs = job_inputs(j)
                for name, v in g.items():
                    check_sentinel(j, v, name, inputs[2])
                c = dict(j, op="lap_rows")
                gate_fast(c, g, inputs, knob_str(env_knobs, ("CAAR_LAPLACE_V1",)), sms)
                assert regime("lap_rows", j["E"], j["nlev"], sms=sms)["per_warp"] >= 4
    assert all(np.array_equal(v, v1_runs[0]) for v in v1_runs[1:])


def test_zz_report_regimes(capsys):
    """Not a gate: what the tests above measured, per kernel, case and knob."""
    with capsys.disabled():
        for line in REPORT:
            print(f"\n[regimes] {line}", end="")
        print()


def _knob_worker(spec_path):
    spec = json.loads(open(spec_path).read())
    for j in spec["jobs"]:
        j["range"] = tuple(j["range"])
        if "tls" in j:
            j["tls"] = tuple(j["tls"])
        np.savez(os.path.join(spec["out"], f"{j['id']}.npz"), **run_job(j))


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--knob-worker":
    _knob_worker(sys.argv[2])
