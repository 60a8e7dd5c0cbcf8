"""The argument checks of the C API, entry point by entry point, through raw ctypes calls: a rejected call returns the
exact error code (CAAR_ERR_INVALID for a bad argument, CAAR_ERR_STATE before caar_set_params), launches nothing and
leaves the caller's control and tracer time level as they were. The same calls with valid arguments succeed, so each
rejection comes from the one argument its case changes."""
import ctypes as C

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
from oracle import harness

pytestmark = pytest.mark.gpu

E, L, Q, NTL = 5, 16, 2, 3
INVALID, STATE = 1, 5
VALID = dict(nets=0, nete=E, n0=0, np1=1, nm1=2, qn0=0, mode=tb.MODE_FAST, nsteps=1, tl=0, chunk=0,
             which=tb.capi.X_VSTAR, op=tb.capi.OP_LAPLACE_SIMPLE, layout=tb.capi.LAYOUT_CXX)


def _sizes():
    return C.byref(C.c_size_t()), C.byref(C.c_size_t())


# entry point -> call(lib, handle, arguments, control, tracer time level, host arrays, extra buffer)
CALLS = {
    "caar_run": lambda lib, h, a, ctl, q, arr, buf: lib.caar_run(h, C.byref(ctl), a["nsteps"], a["mode"]),
    "caar_run_stepping": lambda lib, h, a, ctl, q, arr, buf: lib.caar_run_stepping(h, C.byref(ctl), a["nsteps"],
                                                                                   a["mode"]),
    "caar_run_rk5": lambda lib, h, a, ctl, q, arr, buf: lib.caar_run_rk5(h, C.byref(ctl), 1.0, a["nsteps"], a["mode"]),
    "caar_run_host": lambda lib, h, a, ctl, q, arr, buf: lib.caar_run_host(h, C.byref(arr), C.byref(ctl), a["mode"],
                                                                           a["chunk"]),
    "caar_host_traffic": lambda lib, h, a, ctl, q, arr, buf: lib.caar_host_traffic(h, C.byref(ctl), a["mode"],
                                                                                   *_sizes()),
    "caar_euler_step": lambda lib, h, a, ctl, q, arr, buf: lib.caar_euler_step(h, a["nets"], a["nete"], a["qn0"], Q,
                                                                               1.0, a["mode"]),
    "caar_advect_tracers": lambda lib, h, a, ctl, q, arr, buf: lib.caar_advect_tracers(
        h, a["nets"], a["nete"], C.byref(q), Q, 1.0, a["nsteps"], a["mode"]),
    "caar_sphere_wk": lambda lib, h, a, ctl, q, arr, buf: lib.caar_sphere_wk(h, a["op"], a["nets"], a["nete"],
                                                                             a["mode"]),
    "caar_norms": lambda lib, h, a, ctl, q, arr, buf: lib.caar_norms(h, a["tl"], a["nets"], a["nete"],
                                                                     (C.c_double * 3)()),
    "caar_checksums": lambda lib, h, a, ctl, q, arr, buf: lib.caar_checksums(h, a["tl"], a["nets"], a["nete"],
                                                                             C.byref(tb.capi.Checksum())),
    "caar_upload_range": lambda lib, h, a, ctl, q, arr, buf: lib.caar_upload_range(h, C.byref(arr), tb.capi.F_ALL,
                                                                                   a["nets"], a["nete"]),
    "caar_download_range": lambda lib, h, a, ctl, q, arr, buf: lib.caar_download_range(h, C.byref(arr), 0, a["nets"],
                                                                                       a["nete"]),
    "caar_extra_upload": lambda lib, h, a, ctl, q, arr, buf: lib.caar_extra_upload(h, a["which"], buf),
    "caar_extra_download": lambda lib, h, a, ctl, q, arr, buf: lib.caar_extra_download(h, a["which"], buf),
    "caar_describe": lambda lib, h, a, ctl, q, arr, buf: lib.caar_describe(h, a["mode"], C.create_string_buffer(256),
                                                                           256, None),
    "caar_upload_layout": lambda lib, h, a, ctl, q, arr, buf: lib.caar_upload_layout(h, C.byref(arr), 0, a["layout"]),
}
WITH_CONTROL = ("caar_run", "caar_run_stepping", "caar_run_rk5", "caar_run_host", "caar_host_traffic")
TRACER = ("caar_euler_step", "caar_advect_tracers")
NEED_PARAMS = WITH_CONTROL[:4] + TRACER + ("caar_sphere_wk",)
RANGED = WITH_CONTROL + TRACER + ("caar_sphere_wk", "caar_norms", "caar_checksums", "caar_upload_range",
                                  "caar_download_range")
MODED = WITH_CONTROL + TRACER + ("caar_sphere_wk", "caar_describe")
LEVELED = WITH_CONTROL + ("caar_norms", "caar_checksums")
STEPPED = ("caar_run", "caar_run_stepping", "caar_run_rk5", "caar_advect_tracers")
EXTRA = ("caar_extra_upload", "caar_extra_download")

# (entry point, case, handle: None / "fresh" (no caar_set_params) / "ready", arguments that differ from VALID, code)
CASES = (
    [(ep, "null handle", None, {}, INVALID) for ep in CALLS]
    + [(ep, "before set_params", "fresh", {}, STATE) for ep in NEED_PARAMS]
    + [(ep, f"range {r[0]}:{r[1]}", "ready", dict(nets=r[0], nete=r[1]), INVALID)
       for ep in RANGED for r in ((-1, 2), (0, E + 1), (3, 2))]
    + [(ep, "mode 7", "ready", dict(mode=7), INVALID) for ep in MODED]
    + [(ep, "time level ntl", "ready", dict(np1=NTL, tl=NTL), INVALID) for ep in LEVELED]
    + [(ep, "qn0 2", "ready", dict(qn0=2), INVALID) for ep in WITH_CONTROL + TRACER]
    + [(ep, "nsteps -1", "ready", dict(nsteps=-1), INVALID) for ep in STEPPED]
    + [(ep, f"extra array {w}", "ready", dict(which=w), INVALID) for ep in EXTRA for w in (-1, 5)]
    + [("caar_upload_layout", "layout 7", "ready", dict(layout=7), INVALID),
       ("caar_sphere_wk", "op 9", "ready", dict(op=9), INVALID),
       ("caar_run_host", "chunk_elems -2", "ready", dict(chunk=-2), INVALID)]
)


@pytest.fixture(scope="module")
def env():
    s = harness.randomize(harness.PortOracle().init(E, L, Q, NTL), seed=3)
    ready, fresh = tb.Caar(E, L, Q, NTL), tb.Caar(E, L, Q, NTL)
    ready.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    ready.upload(s.arrays)
    arr = tb.capi.Arrays(**{n: s.arrays[n].ctypes.data_as(C.POINTER(C.c_double)) for n in tb.FIELD_NAMES})
    buf = np.zeros(E * L * 32)  # the largest extra array at these dims (vstar, qtens)
    yield dict(state=s, handles={"ready": ready, "fresh": fresh}, arr=arr, buf=buf)
    ready.close()
    fresh.close()


def call(env, ep, kind, over):
    """Runs one case; returns (code, control after, tracer time level after, launches it added over both handles)."""
    lib = tb.load_library()
    a = {**VALID, **over}
    ctl = tb.capi.Control(a["nets"], a["nete"], a["n0"], a["np1"], a["nm1"], a["qn0"], 0.5)
    q = C.c_int(a["qn0"])
    handles = env["handles"].values()
    before = sum(h.launch_count() for h in handles)
    h = env["handles"][kind].h if kind else None
    rc = CALLS[ep](lib, h, a, ctl, q, env["arr"], env["buf"].ctypes.data_as(C.POINTER(C.c_double)))
    env["handles"]["ready"].sync()
    launched = sum(h.launch_count() for h in handles) - before
    return rc, (ctl.nets, ctl.nete, ctl.n0, ctl.np1, ctl.nm1, ctl.qn0, ctl.dt2), q.value, launched


@pytest.mark.parametrize("ep", list(CALLS))
def test_valid_arguments_are_accepted(env, ep):
    rc, _, _, _ = call(env, ep, "ready", {})
    assert rc == 0, tb.load_library().caar_last_error().decode()


@pytest.mark.parametrize("ep,case,kind,over,want", CASES, ids=[f"{c[0]}-{c[1]}" for c in CASES])
def test_rejected_call_changes_nothing(env, ep, case, kind, over, want):
    a = {**VALID, **over}
    rc, ctl, qn0, launched = call(env, ep, kind, over)
    assert rc == want, tb.load_library().caar_last_error().decode()
    assert launched == 0
    assert ctl == (a["nets"], a["nete"], a["n0"], a["np1"], a["nm1"], a["qn0"], 0.5)
    assert qn0 == a["qn0"]
