"""caar_vertical_remap (HOMME's PPM vertical remap for rsplit > 0) on the GPU, bit for bit against the numpy
transcription of tests/remap_oracle.py: at nlev 2 .. 131, qsize 0, 1, 4 and qsize = qsize_d = 35, every tl, both qtl,
sub-ranges, the three deformation regimes, with sentinels wherever the call must not write, and at a size where the
grid-stride walk wraps; plus run-to-run bits, launch counts and every error code, caar_run_rk5 unchanged by a kept
hybi, the composition after a strict RK5 + DSS step and a limited tracer step, partitioned handles, and Qdp offsets
past 2^31 doubles."""
import ctypes as C
import os

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
import dss_oracle as do
import remap_oracle as ro
from oracle import harness

pytestmark = pytest.mark.gpu
INVALID, UNSUPPORTED, STATE = 1, 4, 5
NAMES = ("elem_state_dp3d", "elem_state_v", "elem_state_T", "elem_state_Qdp", "elem_derived_phi")
CONSTS = (1.0 / 6.376e6, 1.0, 1004.64, 461.5, 287.04, 2.0 / 7.0)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def sentinel(rng, shape):
    return rng.integers(0x4000000000000000, 0x4100000000000000, size=shape, dtype=np.uint64).view(np.float64)


def to_slices(cols, E, L):
    """(E*16, L) columns -> [E][L][4][4]"""
    return np.ascontiguousarray(np.moveaxis(cols.reshape(E, 16, L), 2, 1)).reshape(E, L, 4, 4)


def inputs(E, L, Qd, tl, qtl, qsize, regime, seed, rng_range=None, ntl=3):
    """handle-shaped arrays: sentinels everywhere, then realistic values at dp3d, T, v (tl) and Qdp(qtl) of iq < qsize
    on the element range"""
    rng = np.random.default_rng(seed)
    a, b = rng_range or (0, E)
    A = {n: sentinel(rng, tb.field_shape(n, E, L, Qd, ntl)) for n in NAMES}
    n = b - a
    dpo = ro.columns(n * 16, L, regime, seed)
    A["elem_state_dp3d"][a:b, tl] = to_slices(dpo, n, L)
    A["elem_state_T"][a:b, tl] = rng.uniform(200.0, 300.0, (n, L, 4, 4))
    A["elem_state_v"][a:b, tl] = rng.uniform(-40.0, 40.0, (n, L, 4, 4, 2))
    for iq in range(qsize):
        A["elem_state_Qdp"][a:b, iq, qtl] = to_slices(ro.mixing_ratios(n * 16, L, seed + iq) * dpo, n, L)
    return A


def remap_handle(E, L, Qd, A, ntl=3):
    h = tb.Caar(E, L, Qd, ntl)
    hyai, hybi = ro.coordinate(L)
    h.set_params(CONSTS, np.zeros(16), ro.PS0, hyai)
    h.set_vertical_coordinate(1, hybi)
    h.upload({n: A[n] for n in NAMES}, names=NAMES)
    return h


def download(h, E, L, Qd, ntl=3):
    out = {n: np.empty(tb.field_shape(n, E, L, Qd, ntl)) for n in NAMES}
    h.download(out, names=NAMES)
    return out


def oracle(A, L, nets, nete, tl, qtl, qsize):
    W = {n: x.copy() for n, x in A.items()}
    hyai, hybi = ro.coordinate(L)
    ro.vertical_remap(W, hyai, hybi, ro.PS0, nets, nete, tl, qtl, qsize)
    return W


def run_case(c):
    E, L, Qd, qs, (a, b), tl, qtl = c["E"], c["L"], c["Qd"], c["qsize"], c["range"], c["tl"], c["qtl"]
    A = inputs(E, L, Qd, tl, qtl, qs, c["regime"], c["seed"], (a, b))
    h = remap_handle(E, L, Qd, A)
    n0 = h.launch_count()
    h.vertical_remap(tl=tl, qtl=qtl, qsize=qs, nets=a, nete=b)
    assert h.launch_count() - n0 == 2
    got = download(h, E, L, Qd)
    h.close()
    return A, got


CASES = []
for i, L in enumerate([2, 3, 5, 7, 26, 30, 72, 80, 127, 128, 131]):
    for j, regime in enumerate(ro.REGIMES):
        k = 3 * i + j
        CASES.append(dict(E=6, L=L, Qd=5, qsize=(0, 1, 4, 5)[k % 4], range=((0, 6), (1, 5), (2, 6))[k % 3],
                          tl=k % 3, qtl=(k // 3) % 2, regime=regime, seed=700 + k))
CASES += [
    dict(E=4, L=72, Qd=35, qsize=35, range=(0, 4), tl=1, qtl=1, regime="under", seed=801),
    dict(E=3, L=127, Qd=35, qsize=35, range=(1, 3), tl=2, qtl=0, regime="over", seed=802),
    # 2990 elements x 2 batches = 2990 warp items: the grid-stride walk wraps several times
    dict(E=3000, L=72, Qd=4, qsize=4, range=(5, 2995), tl=0, qtl=1, regime="under", seed=803),
]


def case_id(c):
    return f"E{c['E']}-L{c['L']}-q{c['qsize']}of{c['Qd']}-r{c['range'][0]}:{c['range'][1]}-tl{c['tl']}-qtl{c['qtl']}-{c['regime']}"


@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_remap_equals_oracle(c):
    """Every array equals the numpy transcription in every bit: the remapped slices, and the sentinels at the other time
    levels, the other Qdp level, tracers iq >= qsize, elements outside the range and a derived field."""
    A, got = run_case(c)
    want = oracle(A, c["L"], *c["range"], c["tl"], c["qtl"], c["qsize"])
    for n in NAMES:
        assert np.array_equal(bits(got[n]), bits(want[n])), n


def test_two_runs_reproduce_bits():
    c = CASES[-2]
    first, second = run_case(c)[1], run_case(c)[1]
    for n in NAMES:
        assert np.array_equal(bits(first[n]), bits(second[n])), n


def test_checks_and_counts():
    """STATE before caar_set_params and without hybi, UNSUPPORTED with rsplit == 0, INVALID for every bad argument:
    no launch and no change. 2 launches per call (qsize 0 included), none for an empty range."""
    lib = tb.load_library()
    E, L, Qd, ntl = 4, 9, 3, 3
    A = inputs(E, L, Qd, 0, 0, Qd, "under", 11)
    hyai, hybi = ro.coordinate(L)
    h = tb.Caar(E, L, Qd, ntl)
    h.upload({n: A[n] for n in NAMES}, names=NAMES)
    good = dict(nets=0, nete=E, tl=0, qtl=0, qsize=2)
    call = lambda **over: lib.caar_vertical_remap(h.h, *{**good, **over}.values())

    def unchanged(rc, **over):
        n = h.launch_count()
        assert call(**over) == rc, over
        h.sync()
        assert h.launch_count() == n, over
        got = download(h, E, L, Qd)
        for name in NAMES:
            assert np.array_equal(bits(got[name]), bits(A[name])), (name, over)

    unchanged(STATE)                                    # no caar_set_params
    h.set_params(CONSTS, np.zeros(16), ro.PS0, hyai)
    unchanged(STATE)                                    # no hybi ever given
    h.set_vertical_coordinate(1, None)
    unchanged(STATE)
    h.set_vertical_coordinate(0, hybi)
    unchanged(UNSUPPORTED)                              # Eulerian
    h.set_vertical_coordinate(2, None)                  # the hybi given before is kept
    assert lib.caar_vertical_remap(None, *good.values()) == INVALID
    for over in (dict(nets=-1), dict(nete=E + 1), dict(nets=3, nete=2), dict(tl=-1), dict(tl=ntl), dict(qtl=-1),
                 dict(qtl=2), dict(qsize=-1), dict(qsize=Qd + 1)):
        unchanged(INVALID, **over)
    for over, launches in ((dict(nets=2, nete=2), 0), (dict(qsize=0), 2), (dict(), 2), (dict(qsize=Qd), 2)):
        n = h.launch_count()
        assert call(**over) == 0, over
        h.sync()
        assert h.launch_count() - n == launches, over
    h.close()


# ---- a kept hybi changes no dynamics result -------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST], ids=["strict", "fast"])
def test_rk5_unchanged_by_hybi(mode):
    E, L = 6, 72
    s = harness.randomize(harness.PortOracle().init(E, L), seed=31)
    outs = []
    for with_hybi in (False, True):
        h = tb.Caar(E, L, s.qsize_d, s.ntl)
        h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
        if with_hybi:
            h.set_vertical_coordinate(1, ro.coordinate(L)[1])
        h.set_control(0, E, 0, 1, 2, int(s.ctl[5]), dt2=s.dt2)
        h.upload(s.arrays)
        h.run_rk5(2, 2.0, mode)
        out = {n: np.empty(tb.field_shape(n, E, L, s.qsize_d, s.ntl)) for n in harness.FIELD_NAMES}
        h.download(out, names=None)
        h.close()
        outs.append(out)
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(outs[0][n]), bits(outs[1][n])), n


# ---- one remap interval: dynamics + DSS, the limited tracer step, the remap -----------------------------------------

def test_composition_after_rk5_dss_and_limited_tracer_step():
    ne, L, Qd, qs, DT = 2, 30, 3, 3, 2.0
    gid = do.cubed_sphere_gid(ne, np.random.default_rng(41))
    E = gid.shape[0]
    s = harness.randomize(harness.PortOracle().init(E, L, qsize_d=Qd), seed=41)
    rng = np.random.default_rng(42)
    vstar = rng.uniform(-20.0, 20.0, (E, L, 4, 4, 2))
    hyai, hybi = ro.coordinate(L)
    h = tb.Caar(E, L, Qd, s.ntl)
    h.set_params(s.consts, s.dvv, ro.PS0, hyai)
    h.set_vertical_coordinate(1, hybi)
    h.set_control(0, E, 0, 1, 2, 0, dt2=s.dt2)
    h.upload(s.arrays)
    h.upload_vstar(vstar)
    h.set_connectivity(gid)
    h.run_rk5_dss(1, DT, tb.MODE_STRICT)
    tl, q, dp_tl = h.control.n0, 0, h.control.n0
    h.tracer_bounds(q, qs, dp_tl)
    h.neighbor_minmax(qs)
    q = h.advect_tracers(q, qs, 10.0, 1, tb.MODE_STRICT)
    h.limit_tracers(q, qs, dp_tl)
    h.dss(["elem_state_Qdp"], 0, q, qs, tb.DSS_PROJECT)
    pre = {n: np.empty(tb.field_shape(n, E, L, Qd, s.ntl)) for n in harness.FIELD_NAMES}
    h.download(pre, names=None)
    n0 = h.launch_count()
    h.vertical_remap(tl=tl, qtl=q, qsize=qs)
    assert h.launch_count() - n0 == 2
    got = {n: np.empty_like(x) for n, x in pre.items()}
    h.download(got, names=None)
    h.close()
    want = {n: x.copy() for n, x in pre.items()}
    ro.vertical_remap(want, hyai, hybi, ro.PS0, 0, E, tl, q, qs)
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(got[n]), bits(want[n])), n
    col = lambda x: np.moveaxis(x.reshape(E, L, 16), 1, 2).reshape(-1, L)
    dpn = ro.target_dp(col(pre["elem_state_dp3d"][:, tl]), hyai, hybi, ro.PS0)
    assert np.array_equal(bits(col(got["elem_state_dp3d"][:, tl])), bits(dpn))
    assert not np.array_equal(bits(got["elem_state_T"]), bits(pre["elem_state_T"]))


# ---- partitioned handles --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("parts", [(0, 5, 11), (0, 3, 4, 11)], ids=["2parts", "3parts"])
def test_partitioned_handles_hold_the_whole_mesh_slices(parts):
    E, L, Qd, qs, tl, qtl = 11, 72, 4, 4, 1, 0
    A = inputs(E, L, Qd, tl, qtl, qs, "under", 900)
    whole = remap_handle(E, L, Qd, A)
    whole.vertical_remap(tl=tl, qtl=qtl, qsize=qs)
    want = download(whole, E, L, Qd)
    whole.close()
    for e0, e1 in zip(parts[:-1], parts[1:]):
        h = remap_handle(e1 - e0, L, Qd, {n: np.ascontiguousarray(x[e0:e1]) for n, x in A.items()})
        h.vertical_remap(tl=tl, qtl=qtl, qsize=qs)
        got = download(h, e1 - e0, L, Qd)
        h.close()
        for n in NAMES:
            assert np.array_equal(bits(got[n]), bits(want[n][e0:e1])), (n, e0, e1)


# ---- Qdp offsets past 2^31 doubles ----------------------------------------------------------------------------------

def test_qdp_past_2_31():
    """One handle of 15 024 elements x 128 levels x 35 tracers (Qdp holds 2.15e9 doubles); the remap of the last 24
    elements, which start past 2^31 doubles of Qdp, equals the oracle, and a sample of elements before them keeps its
    bits."""
    import torch
    E, L, Qd, NT = 15024, 128, 35, 24
    E0 = E - NT
    need = 8 * sum(int(np.prod(tb.field_shape(n, E, L, Qd, 3))) for n in tb.capi.FIELD_NAMES) + (1 << 30)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB free")
    host = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    if host < 4e9:
        pytest.skip(f"needs about 4 GB of free host memory, {host / 1e9:.1f} GB free")
    assert E0 * Qd * 2 * L * 16 > 2 ** 31
    tl, qtl = 2, 1
    A = inputs(NT, L, Qd, tl, qtl, Qd, "under", 950)
    h = tb.Caar(E, L, Qd)
    hyai, hybi = ro.coordinate(L)
    h.set_params(CONSTS, np.zeros(16), ro.PS0, hyai)
    h.set_vertical_coordinate(1, hybi)
    h.upload_range({n: A[n] for n in NAMES}, E0, E, names=NAMES)
    sample = np.array([0, 1, 4000, 9000, E0 - 1])
    before = {int(e): h.download_range(int(e), int(e) + 1, names=NAMES) for e in sample}
    h.vertical_remap(tl=tl, qtl=qtl, qsize=Qd, nets=E0, nete=E)
    got = h.download_range(E0, E, names=NAMES)
    after = {int(e): h.download_range(int(e), int(e) + 1, names=NAMES) for e in sample}
    h.close()
    want = oracle(A, L, 0, NT, tl, qtl, Qd)
    for n in NAMES:
        assert np.array_equal(bits(got[n]), bits(want[n])), n
        for e in before:
            assert np.array_equal(bits(before[e][n]), bits(after[e][n])), (n, e)
