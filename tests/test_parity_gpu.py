"""GPU parity tests proper: the CUDA path, called through the C-ABI, against the CPU oracle on the same
inputs. Tolerance (BASELINE.json north_star): relative 1e-12 per field, measured as
max|a-b| / max|b| over the field; the strict kernel must be bit-identical."""
import hashlib
import json
import os

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
from oracle import harness

pytestmark = pytest.mark.gpu
TOL = 1e-12


def rel_err(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def oracle_for(nlev):
    return harness.best_oracle(nlev) if nlev in (72, 128) else harness.PortOracle()


def run_gpu(state, ncalls=1, mode=tb.MODE_FAST):
    h = tb.Caar(state.nelem, state.nlev, state.qsize_d, state.ntl)
    h.set_params(state.consts, state.dvv, state.ps0, state.hyai)
    h.set_control(*[int(x) for x in state.ctl], dt2=state.dt2)
    h.upload(state.arrays)
    h.compute_and_apply_rhs(ncalls, mode)
    h.download(state.arrays, names=None)
    nrm = h.norms()
    h.close()
    return nrm


POINTWISE = {}   # field -> worst pointwise relative error seen in this session (reported at the end, not gated)


def check(got, want, exact):
    for n in harness.FIELD_NAMES:
        if n not in harness.MUTATED or exact:
            assert np.array_equal(got.arrays[n], want.arrays[n]), n
        else:
            assert rel_err(got.arrays[n], want.arrays[n]) <= TOL, (n, rel_err(got.arrays[n], want.arrays[n]))
            b = want.arrays[n]
            mask = np.abs(b) > 1e-30 * max(float(np.max(np.abs(b))), 1e-300)
            if mask.any():   # a cancelling field (omega_p) shows a scan-carry regression here first
                e = float(np.max(np.abs(got.arrays[n][mask] - b[mask]) / np.abs(b[mask])))
                POINTWISE[n] = max(POINTWISE.get(n, 0.0), e)


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
def test_reference_default_config(mode):
    """BASELINE configs[0]: the cxx driver default, 10 elements, 1 call."""
    orc = oracle_for(72)
    want = orc.init(10)
    got = want.copy()
    orc.run(want)
    nrm = run_gpu(got, 1, mode)
    check(got, want, exact=(mode == tb.MODE_STRICT))
    assert np.max(np.abs(nrm - orc.norms(want)) / orc.norms(want)) < 1e-13


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
def test_golden_fortran_vectors(mode, golden_dir):
    """The reference's own KAT (fortran/test_mod.F90) straight against the CUDA path."""
    g = np.load(os.path.join(golden_dir, "fortran_golden.npz"))
    s = harness.PortOracle().init(3)
    s.dvv[...] = s.dvv.astype(np.float32).astype(np.float64)
    run_gpu(s, 1, mode)
    T = s.arrays["elem_state_T"][0, 1].transpose(0, 2, 1).reshape(-1)
    v1 = s.arrays["elem_state_v"][0, 1, ..., 0].transpose(0, 2, 1).reshape(-1)
    v2 = s.arrays["elem_state_v"][0, 1, ..., 1].transpose(0, 2, 1).reshape(-1)
    if mode == tb.MODE_STRICT:
        assert np.array_equal(T, g["Ttest"])
    assert rel_err(T, g["Ttest"]) < TOL and rel_err(v1, g["v1test"]) < TOL and rel_err(v2, g["v2test"]) < TOL


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
def test_committed_reference_outputs(mode, golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_outputs_E3.npz"))
    s = harness.PortOracle().init(3)
    for call in (1, 2):
        run_gpu(s, 1, mode)
        for n in harness.MUTATED:
            a = s.arrays[n]
            if n in ("elem_state_dp3d", "elem_state_v", "elem_state_T"):
                a = a[:, 1]
            if mode == tb.MODE_STRICT:
                assert np.array_equal(a, g[f"call{call}_{n}"]), (call, n)
            else:
                assert rel_err(a, g[f"call{call}_{n}"]) <= TOL, (call, n)


@pytest.mark.parametrize("nlev", [72, 128])
@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
@pytest.mark.parametrize("qn0,tls", [(0, (0, 1, 2)), (-1, (2, 0, 1)), (1, (1, 2, 0))])
def test_random_fields(nlev, mode, qn0, tls):
    """Random geometry and fields, moist and dry, rotated time levels, eta_ave_w != 1, 3 calls (accumulators)."""
    orc = oracle_for(nlev)
    want = harness.randomize(harness.PortOracle().init(37, nlev), seed=100 + nlev + qn0)
    want.ctl[2:5] = tls
    want.ctl[5] = qn0
    got = want.copy()
    orc.run(want, 3, 4)
    run_gpu(got, 3, mode)
    check(got, want, exact=(mode == tb.MODE_STRICT))


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
@pytest.mark.parametrize("n0,np1,nm1", [(0, 0, 0), (0, 1, 0), (0, 1, 1), (1, 0, 0)])
def test_time_level_aliasing(mode, n0, np1, nm1):
    """SURVEY §8f rank 2: nm1 = np1 = n0 (forward Euler / RK stages) must behave like the reference."""
    orc = oracle_for(72)
    want = harness.randomize(harness.PortOracle().init(9), seed=5)
    want.ctl[2:5] = (n0, np1, nm1)
    got = want.copy()
    orc.run(want, 2, 1)
    run_gpu(got, 2, mode)
    check(got, want, exact=(mode == tb.MODE_STRICT))


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
def test_element_range_partition(mode):
    """nets/nete: only [nets,nete) changes; disjoint ranges compose to the full run (the multi-GPU split)."""
    orc = oracle_for(72)
    base = harness.randomize(harness.PortOracle().init(11), seed=9)
    want = base.copy()
    want.ctl[0], want.ctl[1] = 3, 8
    got = want.copy()
    orc.run(want)
    run_gpu(got, 1, mode)
    check(got, want, exact=(mode == tb.MODE_STRICT))
    for n in harness.MUTATED:
        assert np.array_equal(got.arrays[n][:3], base.arrays[n][:3])
        assert np.array_equal(got.arrays[n][8:], base.arrays[n][8:])


@pytest.mark.parametrize("nlev", [2, 3, 7, 8, 13, 16, 24, 26, 30, 40, 57, 64, 65, 71, 73, 80, 81, 88, 96, 100, 104, 112,
                                  113, 120, 121, 127])
def test_other_level_counts(nlev):
    """CAAR_MODE_FAST is the fused kernel for EVERY nlev <= 128: multiples of 8 up to 64, 72, 80, 96, 112, 120, 128 have
    an instance of their own (csrc/caar_fused_more.cu), everything in between runs on the next larger instance with
    masked padding levels (26 and 30 are real E3SM level counts). 3 calls: the accumulators see the padding too."""
    orc = harness.PortOracle()
    want = harness.randomize(orc.init(7, nlev), seed=nlev)
    gs, gf = want.copy(), want.copy()
    orc.run(want, 3)
    run_gpu(gs, 3, tb.MODE_STRICT)
    run_gpu(gf, 3, tb.MODE_FAST)
    check(gs, want, exact=True)
    check(gf, want, exact=False)
    h = tb.Caar(1, nlev)
    text, fused = h.describe(tb.MODE_FAST)
    h.close()
    assert fused and "caar_fused_kernel" in text, text


def test_fast_mode_above_128_levels_says_that_it_falls_back():
    h = tb.Caar(1, 130)
    text, fused = h.describe(tb.MODE_FAST)
    h.close()
    assert not fused and "FALLBACK" in text
    orc = harness.PortOracle()
    want = harness.randomize(orc.init(3, 130), seed=1)
    got = want.copy()
    orc.run(want)
    run_gpu(got, 1, tb.MODE_FAST)
    check(got, want, exact=True)        # it IS the reference-order kernel


def test_one_shot_host_call_matches_reference_semantics():
    """caar_compute_and_apply_rhs_host == Homme::compute_and_apply_rhs(TestData&) on host arrays."""
    orc = oracle_for(72)
    want = orc.init(4)
    got = want.copy()
    orc.run(want)
    tb.compute_and_apply_rhs(got, mode=tb.MODE_STRICT)
    check(got, want, exact=True)


def test_fast_vs_strict_at_scale():
    """ne=30 (5400 elements, BASELINE configs[2]): the fast kernel against the bit-exact strict kernel on the
    GPU over the full set, plus a CPU-oracle check of the strict kernel on a slice."""
    E = 5400
    s = harness.PortOracle().init(E)
    a, b = s.copy(), s.copy()
    run_gpu(a, 2, tb.MODE_STRICT)
    run_gpu(b, 2, tb.MODE_FAST)
    for n in harness.MUTATED:
        assert rel_err(b.arrays[n], a.arrays[n]) <= TOL, n
    orc = oracle_for(72)
    s.ctl[0], s.ctl[1] = 5000, 5016
    orc.run(s, 2, 1)
    for n in harness.MUTATED:
        assert np.array_equal(a.arrays[n][5000:5016], s.arrays[n][5000:5016]), n


def test_norms_protocol():
    orc = oracle_for(72)
    s = orc.init(10)
    h = tb.Caar(10)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays)
    n0 = h.norms(1)
    assert np.max(np.abs(n0 - orc.norms(s)) / orc.norms(s)) < 1e-13
    # sums of squares over disjoint ranges add up (what the ranks all-reduce)
    tot = h.sumsq(1, 0, 10)
    parts = h.sumsq(1, 0, 4) + h.sumsq(1, 4, 10)
    assert np.max(np.abs(tot - parts) / tot) < 1e-14
    h.close()


def test_saxpby():
    rng = np.random.default_rng(3)
    for n in (1, 7, 4096, 128 * 256 * 3 + 1):
        x, y = rng.standard_normal(n), rng.standard_normal(n)
        want = x.copy()
        for _ in range(3):
            want = 3.0 * want + 5.0 * y
        tb.saxpby_host(3.0, 5.0, x, y, sweeps=3)
        assert rel_err(x, want) < 1e-15


def test_errors_are_loud():
    with pytest.raises(tb.CaarError):
        tb.Caar(0)
    h = tb.Caar(2)
    with pytest.raises(tb.CaarError):            # run before set_params
        h.compute_and_apply_rhs()
    s = harness.PortOracle().init(2)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.set_control(nete=3)
    with pytest.raises(tb.CaarError):
        h.compute_and_apply_rhs()
    h.set_control(nete=2, np1=7)
    with pytest.raises(tb.CaarError):
        h.compute_and_apply_rhs()
    h.close()


def run_gpu_host(state, ncalls=1, mode=tb.MODE_FAST, chunk=0):
    """The reference-facing call on HOST arrays (caar_run_host): no explicit upload/download."""
    h = tb.Caar(state.nelem, state.nlev, state.qsize_d, state.ntl)
    h.set_params(state.consts, state.dvv, state.ps0, state.hyai)
    h.set_control(*[int(x) for x in state.ctl], dt2=state.dt2)
    if chunk == tb.HOST_ZERO_COPY:
        tb.host_register(state.arrays)
    try:
        for _ in range(ncalls):
            h.compute_and_apply_rhs_host(state.arrays, mode, chunk)
    finally:
        if chunk == tb.HOST_ZERO_COPY:
            tb.host_unregister(state.arrays)
    traffic = h.host_traffic(mode)
    h.close()
    return traffic


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
@pytest.mark.parametrize("chunk", [0, 1, 7, 64, tb.HOST_ZERO_COPY])
@pytest.mark.parametrize("qn0,tls", [(0, (0, 1, 2)), (-1, (2, 0, 1)), (1, (0, 1, 0)), (0, (1, 1, 1))])
def test_streamed_host_call(mode, chunk, qn0, tls):
    """caar_run_host: pipelined copy-in | kernel | copy-out over ragged element chunks moves only the slices
    the routine reads/writes, and the host arrays end up exactly as the reference leaves them — every array,
    including the values the routine does not touch (other time levels, the unused Qdp level, pecnd)."""
    orc = oracle_for(72)
    want = harness.randomize(harness.PortOracle().init(23), seed=77 + chunk)
    want.ctl[0:2] = (2, 21)
    want.ctl[2:5] = tls
    want.ctl[5] = qn0
    got = want.copy()
    orc.run(want, 2, 2)
    h2d, d2h = run_gpu_host(got, 2, mode, chunk)
    check(got, want, exact=(mode == tb.MODE_STRICT))
    # traffic accounting: 13 level-fields + geometry in, 8 out per element (fewer when levels alias / dry)
    lf = 72 * 16 * 8
    nlv = 1 if tls[0] == tls[2] else 2
    extra = 73 * 16 * 8 if mode == tb.MODE_STRICT else 0
    assert h2d == 19 * (1664 + (4 * nlv + (qn0 != -1) + 4) * lf + extra)
    assert d2h == 19 * (8 * lf + extra)


@pytest.mark.parametrize("chunk", [5, tb.HOST_ZERO_COPY])
@pytest.mark.parametrize("nlev", [128, 24, 96, 30])
def test_streamed_host_call_other_nlev(nlev, chunk):
    """nlev=128 / 96 (cluster instances), 24 (one CTA per element) and 30 (reference-order kernel) through both host paths; the staged path also takes
    numpy (pageable) host memory."""
    orc = oracle_for(nlev)
    want = harness.randomize(harness.PortOracle().init(13, nlev), seed=3)
    got = want.copy()
    orc.run(want, 1, 2)
    run_gpu_host(got, 1, tb.MODE_FAST, chunk)
    check(got, want, exact=False)


def test_zero_copy_needs_mapped_host_memory():
    s = harness.PortOracle().init(3)
    h = tb.Caar(3)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    with pytest.raises(tb.CaarError):
        h.compute_and_apply_rhs_host(s.arrays, tb.MODE_FAST, tb.HOST_ZERO_COPY)
    h.close()


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
@pytest.mark.parametrize("nlev,qsize_d", [(72, 1), (72, 3), (24, 2)])
def test_f90_flat_pointer_boundary(mode, nlev, qsize_d):
    """SURVEY §8f rank 1 / §8b alt boundary: arrays in Fortran memory order in, Fortran memory order out
    (caar_upload_layout / caar_download_layout with CAAR_LAYOUT_F90, Dvv through caar_set_params_f90, no
    rmetdet passed — HOMMEXX has none). Same results as the reference on the same values."""
    orc = harness.PortOracle() if (nlev != 72 or qsize_d != 1) else oracle_for(72)
    want = harness.randomize(harness.PortOracle().init(11, nlev, qsize_d), seed=21 + qsize_d)
    want.arrays["elem_rmetdet"][...] = 1.0 / want.arrays["elem_metdet"]
    f90 = harness.to_f90(want.arrays)
    del f90["elem_rmetdet"]
    orc.run(want, 2, 2)
    h = tb.Caar(want.nelem, nlev, qsize_d, want.ntl)
    h.set_params_f90(want.consts, np.ascontiguousarray(want.dvv.T), want.ps0, want.hyai)
    h.set_control(*[int(x) for x in want.ctl], dt2=want.dt2)
    h.upload_f90(f90)
    h.compute_and_apply_rhs(2, mode)
    f90["elem_rmetdet"] = np.zeros_like(f90["elem_metdet"])
    h.download_f90(f90, names=None)
    h.close()
    got = want.copy()
    got.arrays = harness.from_f90(f90)
    check(got, want, exact=(mode == tb.MODE_STRICT))


def test_f90_boundary_against_fortran_golden(golden_dir):
    """The Fortran KAT (fortran/test_mod.F90) read straight out of the F90-layout download: no transposes."""
    g = np.load(os.path.join(golden_dir, "fortran_golden.npz"))
    s = harness.PortOracle().init(3)
    f90 = harness.to_f90(s.arrays)
    h = tb.Caar(3)
    dvv32 = s.dvv.astype(np.float32).astype(np.float64)
    h.set_params_f90(s.consts, np.ascontiguousarray(dvv32.T), s.ps0, s.hyai)
    h.upload_f90(f90)
    h.compute_and_apply_rhs(1, tb.MODE_STRICT)
    h.download_f90(f90)
    h.close()
    assert np.array_equal(f90["elem_state_T"][0, 1].reshape(-1), g["Ttest"])
    assert rel_err(f90["elem_state_v"][0, 1][:, 0].reshape(-1), g["v1test"]) < 1e-14
    assert rel_err(f90["elem_state_v"][0, 1][:, 1].reshape(-1), g["v2test"]) < 1e-14


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
def test_leapfrog_stepping_with_time_level_rotation(mode):
    """SURVEY §8f rank 2: caar_run_stepping = call + TestData::update_time_levels, 5 steps, against the
    reference doing the same on the CPU (PO/main.cpp:116-118 with the rotation enabled)."""
    orc = oracle_for(72)
    want = harness.randomize(harness.PortOracle().init(7), seed=12)
    want.dt2 = 0.5
    got = want.copy()
    for _ in range(5):
        orc.run(want, 1, 1)
        nets, nete, n0, np1, nm1, qn0 = [int(x) for x in want.ctl]
        want.ctl[:] = (nets, nete, np1, nm1, n0, qn0)
    h = tb.Caar(got.nelem, got.nlev)
    h.set_params(got.consts, got.dvv, got.ps0, got.hyai)
    h.set_control(*[int(x) for x in got.ctl], dt2=got.dt2)
    h.upload(got.arrays)
    h.run_stepping(5, mode)
    h.download(got.arrays, names=None)
    assert (h.control.n0, h.control.np1, h.control.nm1) == tuple(int(x) for x in want.ctl[2:5])
    h.close()
    for n in harness.FIELD_NAMES:
        if mode == tb.MODE_STRICT or n not in harness.MUTATED:
            assert np.array_equal(got.arrays[n], want.arrays[n]), n
        else:  # rounding differences are amplified by the 5 dependent steps: 1e-12 per step
            assert rel_err(got.arrays[n], want.arrays[n]) <= 5 * TOL, n


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
@pytest.mark.parametrize("nlev,qsize_d,qsize,qn0", [(72, 1, 1, 0), (72, 4, 3, 1), (128, 2, 2, 0), (20, 5, 5, 1), (30, 3, 3, 0),
                                                    (26, 2, 1, 1), (72, 35, 35, 0), (100, 2, 2, 1), (37, 1, 1, 0)])
def test_euler_step_tracer_rhs(mode, nlev, qsize_d, qsize, qn0):
    """SURVEY §8f rank 4: qtens = Qdp(qn0) - dt*divergence_sphere(vstar*Qdp(qn0)) against the CPU restatement, which is
    pinned to the reference's own divergence_sphere_update (tests/test_oracle_hommexx.py). Strict mode bit-exact. Level
    counts that do not fill whole slabs / warps and the reference's QSIZE_D = 35 (LV/config.h.in:10) included."""
    orc = harness.PortOracle()
    s = harness.randomize(orc.init(9, nlev, qsize_d), seed=31 + nlev)
    s.ctl[0:2] = (1, 8)
    rng = np.random.default_rng(nlev)
    vstar = rng.uniform(-40.0, 40.0, size=(9, nlev, 4, 4, 2))
    dt = 150.0
    want = np.zeros((9, qsize_d, nlev, 4, 4))
    orc.euler_step(s, vstar, want, qn0, qsize, dt)
    h = tb.Caar(9, nlev, qsize_d)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.set_control(*[int(x) for x in s.ctl], dt2=s.dt2)
    h.upload(s.arrays)
    h.upload_vstar(vstar)
    h.euler_step(qn0, qsize, dt, mode)
    got = h.download_qtens()
    h.close()
    if mode == tb.MODE_STRICT:
        assert np.array_equal(got, want)
    else:
        assert rel_err(got, want) <= TOL
    assert np.all(got[0] == 0) and np.all(got[8] == 0) and np.all(got[:, qsize:] == 0)   # outside the ranges: untouched


def run_gpu_eulerian(state, hybi, ncalls, mode, host_path=None):
    h = tb.Caar(state.nelem, state.nlev, state.qsize_d, state.ntl)
    h.set_params(state.consts, state.dvv, state.ps0, state.hyai)
    h.set_vertical_coordinate(0, hybi)
    h.set_control(*[int(x) for x in state.ctl], dt2=state.dt2)
    if host_path is None:
        h.upload(state.arrays)
        h.compute_and_apply_rhs(ncalls, mode)
        h.download(state.arrays, names=None)
    else:
        if host_path == tb.HOST_ZERO_COPY:
            tb.host_register(state.arrays)
        try:
            for _ in range(ncalls):
                h.compute_and_apply_rhs_host(state.arrays, mode, host_path)
        finally:
            if host_path == tb.HOST_ZERO_COPY:
                tb.host_unregister(state.arrays)
    h.close()


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
@pytest.mark.parametrize("nlev", [72, 128, 24, 30, 96, 26, 5, 88, 104, 125])
@pytest.mark.parametrize("qn0,tls", [(0, (0, 1, 2)), (-1, (0, 0, 0))])
def test_eulerian_vertical_coordinate(mode, nlev, qn0, tls):
    """SURVEY §8f rank 3: rsplit == 0 (eta_dot_dpdn from the divergence sum and hybi, preq_vertadv, vertical flux
    in the dp3d update) against the CPU restatement: preq_vertadv is pinned bit for bit to the reference's own code
    (tests/test_oracle_hommexx.py), the eta_dot_dpdn-from-hybi formula and the signs of the tendencies follow
    F/routine_extracted.F90:227-262,325-334,515-517, which nothing here can execute. Strict mode is bit-exact to the
    restatement; padded level counts included."""
    orc = harness.PortOracle()
    want = harness.randomize(orc.init(13, nlev), seed=nlev + 3)
    want.ctl[2:5] = tls
    want.ctl[5] = qn0
    hybi = np.linspace(0.0, 1.0, nlev + 1) ** 1.5
    got = want.copy()
    orc.run_eulerian(want, hybi, 2, 2)
    run_gpu_eulerian(got, hybi, 2, mode)
    check(got, want, exact=(mode == tb.MODE_STRICT))


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
@pytest.mark.parametrize("host_path", [6, tb.HOST_ZERO_COPY])
def test_eulerian_through_the_host_call(mode, host_path):
    """The host-array pipeline moves eta_dot_dpdn both ways on the Eulerian branch (it is really updated); on the
    zero-copy path the kernel read-modify-writes it in the caller's mapped memory."""
    orc = harness.PortOracle()
    want = harness.randomize(orc.init(21), seed=8)
    hybi = np.linspace(0.0, 1.0, 73)
    got = want.copy()
    orc.run_eulerian(want, hybi, 1, 2)
    run_gpu_eulerian(got, hybi, 1, mode, host_path=host_path)
    check(got, want, exact=(mode == tb.MODE_STRICT))
    assert not np.array_equal(got.arrays["elem_derived_eta_dot_dpdn"], harness.randomize(orc.init(21), seed=8).arrays["elem_derived_eta_dot_dpdn"])


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
def test_empty_and_single_element_ranges(mode):
    """Edge cases of the element range: [k,k) is a no-op on every entry point, a one-element range and a
    one-element handle work (the cluster launch has no minimum grid)."""
    orc = oracle_for(72)
    base = harness.randomize(harness.PortOracle().init(5), seed=2)
    got = base.copy()
    got.ctl[0:2] = (3, 3)
    run_gpu(got, 2, mode)
    run_gpu_host(got, 1, mode, 0)
    for n in harness.FIELD_NAMES:
        assert np.array_equal(got.arrays[n], base.arrays[n]), n
    want = base.copy()
    want.ctl[0:2] = (4, 5)
    got = want.copy()
    orc.run(want)
    run_gpu(got, 1, mode)
    check(got, want, exact=(mode == tb.MODE_STRICT))
    one = harness.randomize(harness.PortOracle().init(1), seed=4)
    got1 = one.copy()
    orc.run(one)
    run_gpu(got1, 1, mode)
    check(got1, one, exact=(mode == tb.MODE_STRICT))


# ---- correctness on the configurations that carry the speed claims ------------------------------------------------

def _windows(E, rng):
    mid = E // 2
    w = [(0, 64), (mid - 32, mid + 32), (E - 64, E)]
    for e in sorted(rng.choice(np.arange(64, E - 64), size=32, replace=False)):
        w.append((int(e), int(e) + 8))          # 32 random windows of 8 elements = 256 random elements
    return w


def full_size_inputs(E, L):
    """The inputs of test_full_size_runs_against_the_compiled_reference -> (td, windows, one harness.State per window
    holding that window's inputs). The closed-form init of E elements, with two thirds of the windows overwritten with
    random geometry and fields (the closed-form init has a diagonal D). tests/golden/make_golden.py runs the oracle
    on these states."""
    from tinman_sandbox_b200.testdata import TestData
    rng = np.random.default_rng(E + L)
    td = TestData(E, L).init_data()
    wins = _windows(E, rng)
    states = []
    for (a, b) in wins:
        s = harness.State(b - a, L)
        s.arrays = {n: td.arrays[n][a:b].copy() for n in harness.FIELD_NAMES}
        s.ctl = np.array([0, b - a, 0, 1, 2, 0], dtype=np.int32)
        s.dt2, s.consts, s.dvv, s.ps0, s.hyai = td.dt2, td.consts.copy(), td.dvv.copy(), td.ps0, td.hyai.copy()
        if a % 3 != 0:                            # two thirds of the windows: random data
            consts, dt2, ps0, hyai = s.consts.copy(), s.dt2, s.ps0, s.hyai.copy()
            harness.randomize(s, seed=a)
            s.consts[:], s.dt2, s.ps0, s.hyai[:] = consts, dt2, ps0, hyai      # one set of scalars per handle
            for n in harness.FIELD_NAMES:
                td.arrays[n][a:b] = s.arrays[n]
        states.append(s)
    return td, wins, states


def digest(a):
    """sha256 of an array's float64 values in C order"""
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest()


def inputs_digest(states):
    h = hashlib.sha256()
    for s in states:
        for n in harness.FIELD_NAMES:
            h.update(digest(s.arrays[n]).encode())
        for x in (s.ctl.astype(np.float64), s.consts, s.dvv, s.hyai, np.array([s.dt2, s.ps0])):
            h.update(digest(x).encode())
    return h.hexdigest()


@pytest.mark.parametrize("E,L", [(86400, 72), (49152, 128)])
def test_full_size_runs_against_the_compiled_reference(E, L, golden_dir):
    """BASELINE configs[3] (ne=120: 86400 elements, nlev=72) and the per-GPU slice of configs[4] (ne=256 over 8 GPUs:
    49152 elements, nlev=128) at FULL size on one GPU: first / middle / last 64 elements and 256 random ones on all
    seven mutated arrays after 2 calls — STRICT bit-exact, FAST <= 1e-12 of the STRICT result. The expected values are
    committed as sha256 digests per window and array (tests/golden/full_size_digests.json; the outputs themselves are
    70-125 MB): the reference's outputs on these windows, computed by the CPU restatement, which tests/test_oracle.py
    pins bit for bit to the compiled reference and to its committed outputs."""
    golden = json.load(open(os.path.join(golden_dir, "full_size_digests.json")))[f"{E}x{L}"]
    td, wins, states = full_size_inputs(E, L)
    assert inputs_digest(states) == golden["inputs"]      # otherwise the digests below are of other inputs
    assert [tuple(w) for w, _ in golden["windows"]] == wins
    h = tb.Caar(E, L)
    h.set_params(td.consts, td.dvv, td.ps0, td.hyai)
    h.set_control(*[int(x) for x in td.ctl], dt2=td.dt2)
    strict = []
    for mode in (tb.MODE_STRICT, tb.MODE_FAST):
        h.upload(td.arrays)
        h.compute_and_apply_rhs(2, mode)
        for i, ((a, b), (_, want)) in enumerate(zip(wins, golden["windows"])):
            got = h.download_range(a, b, names=harness.MUTATED)
            for n in harness.MUTATED:
                if mode == tb.MODE_STRICT:
                    assert digest(got[n]) == want[n], (a, n)
                else:
                    assert rel_err(got[n], strict[i][n]) <= TOL, (a, n, rel_err(got[n], strict[i][n]))
            if mode == tb.MODE_STRICT:
                strict.append(got)
        # and the whole set through the bit-pattern checksums: FAST and STRICT cover every element, nothing outside
        # [nets,nete) of any array is touched (sums are finite and reproducible)
        cs = h.checksums()
        assert np.all(np.isfinite(cs["sum"])) and np.all(np.isfinite(cs["energy"]))
    h.close()


@pytest.mark.parametrize("eulerian", [False, True])
def test_run_to_run_determinism(eulerian):
    """The cluster protocol of the fused kernel (relaxed barrier.cluster.arrive before the TMA issue, st.async +
    complete_tx into the peers) is the kind of code that races silently, and compute-sanitizer is closed on this pool:
    200 launches on ne=30 from identical inputs, checksummed on the device after EVERY launch with the sum of the IEEE
    bit patterns (exact, order-independent), twice — the two sequences must agree launch by launch, and the arrays that
    are pure outputs must not change from one launch to the next. Eulerian: with np1 == n0 (state updated in place)."""
    E, L, N = 5400, 72, 200
    s = harness.PortOracle().init(E, L)
    harness.randomize(s, seed=17)
    if eulerian:
        s.ctl[2:5] = (0, 0, 0)
        s.dt2 = 1e-3
    seqs = []
    for rep in range(2):
        h = tb.Caar(E, L)
        h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
        if eulerian:
            h.set_vertical_coordinate(0, np.linspace(0.0, 1.0, L + 1))
        h.set_control(*[int(x) for x in s.ctl], dt2=s.dt2)
        h.upload(s.arrays)
        bits = []
        for _ in range(N):
            h.compute_and_apply_rhs(1, tb.MODE_FAST)
            bits.append(h.checksums()["bits"].copy())
        h.close()
        seqs.append(np.array(bits))
    assert np.array_equal(seqs[0], seqs[1])
    if not eulerian:        # dp3d, v, T at np1 and phi are overwritten from unchanged inputs: identical at every launch
        for f in (0, 1, 2, 5):
            assert np.all(seqs[0][:, f] == seqs[0][0, f]), tb.CHECKSUM_FIELDS[f]
        assert len(set(seqs[0][:, 4].tolist())) > 1         # omega_p accumulates: the checksum does move


def test_checksums_against_the_oracle():
    """caar_checksums (north star: the quantities the ranks all-reduce after the timed loop): sums and sums of squares
    of the seven mutated arrays to 1e-13, the bit-pattern sums EXACTLY against the bit-exact CPU reference in strict
    mode, the energy norms against numpy; partial ranges add up (what the all-reduce relies on)."""
    orc = oracle_for(72)
    want = harness.randomize(harness.PortOracle().init(23), seed=41)
    h = tb.Caar(23)
    h.set_params(want.consts, want.dvv, want.ps0, want.hyai)
    h.set_control(*[int(x) for x in want.ctl], dt2=want.dt2)
    h.upload(want.arrays)
    h.compute_and_apply_rhs(2, tb.MODE_STRICT)
    orc.run(want, 2, 1)
    cs = h.checksums(1)
    A = want.arrays
    for f, n in enumerate(tb.CHECKSUM_FIELDS):
        a = A[n][:, 1] if n in ("elem_state_dp3d", "elem_state_v", "elem_state_T") else A[n]
        assert abs(cs["sum"][f] - a.sum()) <= 1e-13 * np.abs(a).sum(), n
        assert abs(cs["sumsq"][f] - (a * a).sum()) <= 1e-13 * (a * a).sum(), n
        assert cs["bits"][f] == np.ascontiguousarray(a).view(np.uint64).sum(dtype=np.uint64), n
    mp = A["elem_spheremp"][:, None]
    v, T, dp = A["elem_state_v"][:, 1], A["elem_state_T"][:, 1], A["elem_state_dp3d"][:, 1]
    ke = (mp * 0.5 * (v[..., 0] ** 2 + v[..., 1] ** 2) * dp).sum()
    ie = (mp * want.consts[2] * T * dp).sum()
    assert abs(cs["energy"][0] - ke) <= 1e-13 * abs(ke) and abs(cs["energy"][1] - ie) <= 1e-13 * abs(ie)
    a, b = h.checksums(1, 0, 9), h.checksums(1, 9, 23)
    assert np.array_equal(a["bits"] + b["bits"], cs["bits"])
    assert np.max(np.abs(a["sumsq"] + b["sumsq"] - cs["sumsq"]) / cs["sumsq"]) < 1e-14
    h.close()


def test_range_copies():
    s = harness.randomize(harness.PortOracle().init(12), seed=6)
    h = tb.Caar(12)
    h.upload(s.arrays)
    win = {n: np.ascontiguousarray(a[3:7]) * 2.0 for n, a in s.arrays.items()}
    h.upload_range(win, 3, 7)
    back = {n: np.zeros_like(a) for n, a in s.arrays.items()}
    h.download(back, names=None)
    for n in harness.FIELD_NAMES:
        assert np.array_equal(back[n][3:7], win[n]) and np.array_equal(back[n][:3], s.arrays[n][:3])
        assert np.array_equal(back[n][7:], s.arrays[n][7:])
    got = h.download_range(5, 12, names=harness.FIELD_NAMES)
    for n in harness.FIELD_NAMES:
        assert np.array_equal(got[n], back[n][5:12])
    with pytest.raises(tb.CaarError):
        h.download_range(5, 13)
    h.close()


def test_set_stream_orders_against_the_previous_stream():
    """caar_set_stream: work queued on the old stream is ordered before work submitted after the switch."""
    import torch
    orc = oracle_for(72)
    want = harness.randomize(harness.PortOracle().init(64), seed=13)
    got = want.copy()
    orc.run(want, 4, 2)
    h = tb.Caar(64)
    h.set_params(got.consts, got.dvv, got.ps0, got.hyai)
    h.set_control(*[int(x) for x in got.ctl], dt2=got.dt2)
    h.upload(got.arrays)
    other = torch.cuda.Stream()
    for i in range(4):                      # alternate between the handle's stream and a torch stream, no syncs
        h.set_stream(other.cuda_stream if i % 2 == 0 else 0)
        h.compute_and_apply_rhs(1, tb.MODE_STRICT, sync=False)
    h.set_stream(0)
    h.sync()
    h.download(got.arrays, names=None)
    h.close()
    check(got, want, exact=True)


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST])
@pytest.mark.parametrize("nlev", [72, 128, 30, 26, 100, 5, 16, 17, 41])
def test_weak_form_operators(mode, nlev):
    """SURVEY §8f rank 4, the hyperviscosity half: divergence_sphere_wk, laplace_simple, laplace_tensor and
    laplace_tensor_replace (LV/SphereOperators.hpp:493-636) through caar_sphere_wk against the CPU restatement, which is
    bit-identical to the reference's own code run under the Kokkos stand-in (tests/test_oracle_hommexx.py). Strict mode
    bit-exact, fast mode 1e-12 of the field maximum; a sub-range of elements leaves the rest of the output alone."""
    orc = harness.PortOracle()
    E = 9
    s = harness.randomize(orc.init(E, nlev), seed=nlev + 50)
    rng = np.random.default_rng(nlev)
    vin = rng.uniform(-40.0, 40.0, size=(E, nlev, 4, 4, 2))
    sin = rng.uniform(200.0, 300.0, size=(E, nlev, 4, 4))
    tv = rng.uniform(-1.0, 1.0, size=(E, 4, 4, 2, 2))
    h = tb.Caar(E, nlev)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays)
    h.upload_extra(tb.X_VSTAR, vin)
    h.upload_extra(tb.X_SCALAR_IN, sin)
    h.upload_extra(tb.X_TENSORVISC, tv)
    sentinel = np.full((E, nlev, 4, 4), -7.0)
    for op, name, field in ((tb.OP_DIVERGENCE_WK, "divergence_sphere_wk", vin), (tb.OP_LAPLACE_SIMPLE, "laplace_simple", sin),
                            (tb.OP_LAPLACE_TENSOR, "laplace_tensor", sin)):
        want = orc.sphere_wk(name, s, field, tv if name == "laplace_tensor" else None)
        h.upload_extra(tb.X_SCALAR_OUT, sentinel)
        h.sphere_wk(op, mode, nets=1, nete=E - 2)
        got = h.download_extra(tb.X_SCALAR_OUT, (E, nlev, 4, 4))
        assert np.all(got[0] == -7.0) and np.all(got[E - 2:] == -7.0), name
        if mode == tb.MODE_STRICT:
            assert np.array_equal(got[1:E - 2], want[1:E - 2]), name
        else:
            assert rel_err(got[1:E - 2], want[1:E - 2]) <= TOL, (name, rel_err(got[1:E - 2], want[1:E - 2]))
    want = orc.sphere_wk("laplace_tensor", s, sin, tv)
    h.upload_extra(tb.X_SCALAR_OUT, sin)
    h.sphere_wk(tb.OP_LAPLACE_TENSOR_REPLACE, mode, nets=0, nete=E)
    got = h.download_extra(tb.X_SCALAR_OUT, (E, nlev, 4, 4))
    h.close()
    if mode == tb.MODE_STRICT:
        assert np.array_equal(got, want)
    else:
        assert rel_err(got, want) <= TOL


@pytest.mark.parametrize("E,nlev", [(1, 16), (1, 20), (2, 33), (3, 128)])
def test_laplace_fewer_rows_than_a_tile(E, nlev):
    """Ranges smaller than (or barely larger than) one 32-row tile of the thread-per-level laplacians: the tile is
    zero-filled past the range on load and clipped on store."""
    orc = harness.PortOracle()
    s = harness.randomize(orc.init(E, nlev), seed=E * 100 + nlev)
    rng = np.random.default_rng(E + nlev)
    sin = rng.uniform(200.0, 300.0, size=(E, nlev, 4, 4))
    tv = rng.uniform(-1.0, 1.0, size=(E, 4, 4, 2, 2))
    h = tb.Caar(E, nlev)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays)
    h.upload_extra(tb.X_SCALAR_IN, sin)
    h.upload_extra(tb.X_TENSORVISC, tv)
    for op, name in ((tb.OP_LAPLACE_SIMPLE, "laplace_simple"), (tb.OP_LAPLACE_TENSOR, "laplace_tensor")):
        h.sphere_wk(op, tb.MODE_FAST)
        got = h.download_extra(tb.X_SCALAR_OUT, (E, nlev, 4, 4))
        want = orc.sphere_wk(name, s, sin, tv if name == "laplace_tensor" else None)
        assert rel_err(got, want) <= TOL, name
    h.close()


def test_laplace_scheduler_over_many_launches():
    """The thread-per-level laplacians draw their tiles from a global counter that every launch must leave at zero:
    300 back-to-back launches over changing element ranges (changing tile and chunk counts, queued without
    synchronisation), each checked against the oracle afterwards, and two launches of the same range bit-identical
    (the result does not depend on which warp drew which tile)."""
    orc = harness.PortOracle()
    E, L = 48, 40
    s = harness.randomize(orc.init(E, L), seed=11)
    rng = np.random.default_rng(12)
    sin = rng.uniform(200.0, 300.0, size=(E, L, 4, 4))
    tv = rng.uniform(-1.0, 1.0, size=(E, 4, 4, 2, 2))
    want = {tb.OP_LAPLACE_SIMPLE: orc.sphere_wk("laplace_simple", s, sin),
            tb.OP_LAPLACE_TENSOR: orc.sphere_wk("laplace_tensor", s, sin, tv)}
    h = tb.Caar(E, L)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays)
    h.upload_extra(tb.X_SCALAR_IN, sin)
    h.upload_extra(tb.X_TENSORVISC, tv)
    for it in range(300):
        a = int(rng.integers(0, E - 1))
        b = int(rng.integers(a + 1, E + 1))
        op = tb.OP_LAPLACE_SIMPLE if it % 2 else tb.OP_LAPLACE_TENSOR
        if it % 25 == 24:
            h.upload_extra(tb.X_SCALAR_OUT, np.full((E, L, 4, 4), -7.0))
            h.sphere_wk(op, tb.MODE_FAST, nets=a, nete=b)
            got = h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4))
            assert np.all(got[:a] == -7.0) and np.all(got[b:] == -7.0)
            assert rel_err(got[a:b], want[op][a:b]) <= TOL, (it, a, b)
        else:
            h.sphere_wk(op, tb.MODE_FAST, nets=a, nete=b, sync=False)
    h.sphere_wk(tb.OP_LAPLACE_TENSOR, tb.MODE_FAST)
    one = h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4)).copy()
    h.sphere_wk(tb.OP_LAPLACE_TENSOR, tb.MODE_FAST)
    two = h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4))
    h.close()
    assert np.array_equal(one, two)


def test_biharmonic_is_two_laplacians():
    """A property the composition offers at any size: laplace_simple applied twice through the in-place form equals the
    oracle's two applications (the hyperviscosity operator is nabla^4), ne=30-sized."""
    orc = harness.PortOracle()
    E, L = 600, 72
    s = harness.randomize(orc.init(E, L), seed=77)
    sin = np.random.default_rng(1).uniform(200.0, 300.0, size=(E, L, 4, 4))
    ones = np.zeros((E, 4, 4, 2, 2))
    ones[..., 0, 0] = ones[..., 1, 1] = 1.0                      # tensorVisc = identity: laplace_tensor == laplace_simple
    want = orc.sphere_wk("laplace_simple", s, orc.sphere_wk("laplace_simple", s, sin))
    h = tb.Caar(E, L)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays)
    h.upload_extra(tb.X_TENSORVISC, ones)
    h.upload_extra(tb.X_SCALAR_OUT, sin)
    h.sphere_wk(tb.OP_LAPLACE_TENSOR_REPLACE, tb.MODE_FAST)
    h.sphere_wk(tb.OP_LAPLACE_TENSOR_REPLACE, tb.MODE_FAST)
    got = h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4))
    h.close()
    assert rel_err(got, want) <= 2 * TOL


def test_level_local_operators_are_linear_at_scale():
    """Size-independent property at ne=120 / 4 (21600 elements, nlev=72), where no CPU oracle run is affordable for every
    element: the tracer step and laplace_tensor are linear in the field —
    op(alpha*x + beta*y) == alpha*op(x) + beta*op(y) to 1e-12 of the maximum — plus an oracle check of the last 8 elements
    (high element indices: TMA slice coordinates near the end of the arrays)."""
    orc = harness.PortOracle()
    E, L, Q = 21600, 72, 2
    rng = np.random.default_rng(5)
    s = orc.init(E, L, qsize_d=Q)
    tail = harness.randomize(orc.init(8, L, qsize_d=Q), seed=3)
    for n in harness.FIELD_NAMES:                     # random geometry and fields in the last 8 elements
        s.arrays[n][E - 8:] = tail.arrays[n]
    x = rng.uniform(0.5, 1.5, size=(E, L, 4, 4))
    y = rng.uniform(0.5, 1.5, size=(E, L, 4, 4))
    alpha, beta = 1.75, -0.625
    vstar = rng.uniform(-40.0, 40.0, size=(E, L, 4, 4, 2))
    tv = rng.uniform(-1.0, 1.0, size=(E, 4, 4, 2, 2))
    h = tb.Caar(E, L, Q)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays)
    h.upload_extra(tb.X_TENSORVISC, tv)
    h.upload_vstar(vstar)

    def lap(f):
        h.upload_extra(tb.X_SCALAR_IN, np.ascontiguousarray(f))
        h.sphere_wk(tb.OP_LAPLACE_TENSOR, tb.MODE_FAST)
        return h.download_extra(tb.X_SCALAR_OUT, (E, L, 4, 4))

    def step(q0, q1):
        s.arrays["elem_state_Qdp"][:, 0, 0] = q0
        s.arrays["elem_state_Qdp"][:, 1, 0] = q1
        h.upload(s.arrays)
        h.euler_step(0, Q, 150.0, tb.MODE_FAST)
        return h.download_qtens()

    lx, ly, lz = lap(x), lap(y), lap(alpha * x + beta * y)
    assert np.max(np.abs(lx)) > 0 and rel_err(lz, alpha * lx + beta * ly) <= 4 * TOL
    want = orc.sphere_wk("laplace_tensor", s, x, tv, nets=E - 8, nete=E)
    assert rel_err(lx[E - 8:], want[E - 8:]) <= TOL
    qa = step(x, y)
    qb = step(alpha * x + beta * y, x)
    assert rel_err(qb[:, 0], alpha * qa[:, 0] + beta * qa[:, 1]) <= 4 * TOL
    wq = np.zeros((E, Q, L, 4, 4))
    s.ctl[0:2] = (E - 8, E)
    orc.euler_step(s, vstar, wq, 0, Q, 150.0)
    assert rel_err(qb[E - 8:], wq[E - 8:]) <= TOL
    h.close()


def test_zz_report_pointwise_errors(capsys):
    """Not a gate: prints the worst POINTWISE relative error per field over every fast-mode comparison of this session
    (the gate is field-normalised, SURVEY §7); run last by name."""
    with capsys.disabled():
        for n, e in sorted(POINTWISE.items()):
            print(f"\n[pointwise] {n}: max |a-b|/|b| = {e:.3e}", end="")
        print()
