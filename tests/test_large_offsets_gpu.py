"""The tracer kernels past 2^31 doubles of Qdp: one handle of 15 024 elements x 128 levels x 35 tracers, whose Qdp
[E][35][2][128][16] holds 2.15e9 doubles (17.2 GB). Elements [0, 15 000) are an ne = 50 cubed sphere filled with one
constant state (the bulk); the last 24 are a closed ne = 2 sphere of their own (the tail), where Qdp of element 15 000,
tracer 0 starts at 2 150 400 000 doubles. Every call runs on the tail, or on the whole handle, and is checked on the
tail against the oracles of tests/ run on a 24-element state: caar_run (qn0 = 1), caar_euler_step and
caar_advect_tracers at qsize 35 (strict by bits, fast under the pointwise gates), caar_tracer_bounds and
caar_limit_tracers, caar_dss of Qdp(1) with both weightings and caar_neighbor_minmax; then the same DSS and bounds on two
partitioned handles cut inside the tail (part_start 0, 15 012, 15 024), through pack, segment move and unpack and through
interior + boundary, equal to the whole-mesh results by bits. A sample of bulk elements just before the tail keeps its
bits through every call (the bulk's Qdp values are powers of two and its spheremp 1, so the DSS maps them to
themselves).

The module skips, naming the shortfall, when the device has less free memory than the whole handle needs (about 34 GB:
its fields, qtens, two bound arrays and vstar, plus 1 GiB) or the host less than about 16 GB. Measured on an NVIDIA B200
at a 1000 W power limit: a peak of 33.6 GB of device memory in use (the whole handle), 18 s for the module."""
import os

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
import dss_oracle as do
import limiter_oracle as lo
import tracer_ssp_oracle as so
from oracle import harness
from oracle import hp_reference as hp
from test_dss_partition_gpu import exchange_dss, exchange_minmax
from test_limiter_gpu import limiter_inputs
from test_pointwise_cpu import level_local_inputs, rhs_reference
from test_pointwise_gpu import check_rhs
from test_rk5_partition_gpu import split_dss

pytestmark = pytest.mark.gpu
NE_BULK, L, QD = 50, 128, 35
E0 = 6 * NE_BULK ** 2            # 15 000: the first tail element
NT = 24                          # the tail: an ne = 2 sphere
E = E0 + NT
CUT = E0 + NT // 2               # the partition boundary inside the tail
CHUNK = 500                      # bulk elements per upload
SAMPLE = np.s_[E0 - 16:E0]       # bulk elements checked after every call
DT = 150.0
QNAMES = ("elem_state_Qdp",)
PEAK = {}                        # device bytes in use, the largest seen by this module


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def note_peak():
    import torch
    free, total = torch.cuda.mem_get_info()
    PEAK["used"] = max(PEAK.get("used", 0), total - free)


def tail_gid():
    """the whole mesh: the ne = 50 sphere, then the ne = 2 sphere with ids past the first's"""
    bulk = do.cubed_sphere_gid(NE_BULK)
    tail = do.cubed_sphere_gid(2, np.random.default_rng(2))
    return np.concatenate([bulk, tail + bulk.max() + 1]), tail


def bulk_chunk():
    """CHUNK copies of one element of a valid state; spheremp 1 and every Qdp value 2^-((3 iq + tl + k) % 16)"""
    s = harness.randomize(harness.PortOracle().init(1, L, QD), seed=5)
    s.arrays["elem_spheremp"][:] = 1.0
    iq, tl, k = np.ogrid[:QD, :2, :L]
    s.arrays["elem_state_Qdp"][0] = (2.0 ** -((3 * iq + tl + k) % 16))[..., None, None]
    return {n: np.ascontiguousarray(np.broadcast_to(a, (CHUNK,) + a.shape[1:])) for n, a in s.arrays.items()}


def fill_bulk(h, chunk, names, e1=E0):
    for e0 in range(0, e1, CHUNK):
        n = min(CHUNK, e1 - e0)
        h.upload_range({k: chunk[k][:n] for k in names}, e0, e0 + n, names=names)


def check_bulk(h, chunk, names):
    got = h.download_range(SAMPLE.start, SAMPLE.stop, names=names)
    for n in names:
        assert np.array_equal(bits(got[n]), bits(chunk[n][:SAMPLE.stop - SAMPLE.start])), n


def footprint(nelem, qtens):
    fields = sum(int(np.prod(tb.field_shape(n, nelem, L, QD, 3))) for n in tb.capi.FIELD_NAMES)
    extra = nelem * QD * L * 16 * qtens + 2 * nelem * QD * L * 2 + nelem * L * 32
    return 8 * (fields + extra)


@pytest.fixture(scope="module")
def whole():
    import torch
    need = footprint(E, True) + (1 << 30)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB free "
                    f"({(need - free) / 1e9:.1f} GB short)")
    host = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    if host < 16e9:
        pytest.skip(f"needs about 16 GB of free host memory, {host / 1e9:.1f} GB free")
    gid, tgid = tail_gid()
    chunk = bulk_chunk()
    h = tb.Caar(E, L, QD)
    fill_bulk(h, chunk, tb.capi.FIELD_NAMES)
    note_peak()
    yield dict(h=h, gid=gid, tgid=tgid, chunk=chunk)
    h.close()


def tail_state(seed, qn0):
    s, vstar, _, _ = level_local_inputs("stratified", NT, L, seed, qsize_d=QD)
    s.ctl[0:6] = (0, NT, 0, 1, 2, qn0)
    return s, vstar


def load_tail(h, s, vstar=None):
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.set_control(E0, E, *[int(x) for x in s.ctl[2:6]], dt2=s.dt2)
    h.upload_range(s.arrays, E0, E)
    if vstar is not None:
        full = np.zeros((E, L, 4, 4, 2))
        full[E0:] = vstar
        h.upload_vstar(full)


# ---- the dynamics RHS reading Qdp(qn0 = 1) ---------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST], ids=["strict", "fast"])
def test_rhs_reads_qdp_past_2_31(whole, mode):
    """caar_run, 2 calls on [15 000, 15 024) with qn0 = 1: strict equal to PortOracle by bits, fast under
    hp.k_rhs(128, 2); the bulk sample keeps every bit."""
    h = whole["h"]
    s, _ = tail_state(7100, 1)
    load_tail(h, s)
    h.compute_and_apply_rhs(2, mode)
    got = s.copy()
    got.arrays.update(h.download_range(E0, E, names=harness.FIELD_NAMES))
    check_bulk(h, whole["chunk"], harness.MUTATED + QNAMES)
    if mode == tb.MODE_STRICT:
        want = s.copy()
        harness.PortOracle().run(want, 2)
        for n in harness.FIELD_NAMES:
            assert np.array_equal(bits(got.arrays[n]), bits(want.arrays[n])), n
    else:
        check_rhs(got, s, rhs_reference(s, 2, None), L, 2, "rhs_lagrangian_fast", "tail of 15024 x 128 x 35")


# ---- the tracer step -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST], ids=["strict", "fast"])
def test_euler_step_and_advect_tracers_past_2_31(whole, mode):
    """caar_euler_step (qn0 = 1) and one step of caar_advect_tracers (qn0 = 0), qsize 35, on [15 000, 15 024): strict
    equal by bits to PortOracle.euler_step and tracer_ssp_oracle.ssp_step, fast within hp.K_EULER and k_ssp(1) u M of
    the long-double reference at every point; the bulk sample keeps its bits."""
    h = whole["h"]
    s, vstar = tail_state(7200, 1)
    load_tail(h, s, vstar)
    h.euler_step(1, QD, DT, mode, nets=E0, nete=E)
    qt = h.download_qtens()[E0:].copy()
    note_peak()
    if mode == tb.MODE_STRICT:
        want = np.zeros((NT, QD, L, 4, 4))
        harness.PortOracle().euler_step(s, vstar, want, 1, QD, DT)
        assert np.array_equal(bits(qt), bits(want))
    else:
        r, at, _ = hp.worst(qt, hp.euler_step(hp.from_state(s), vstar, 1, QD, DT))
        assert r <= hp.K_EULER, (r, at)
    q = h.advect_tracers(0, QD, DT, 1, mode, nets=E0, nete=E)
    assert q == 1
    got = h.download_range(E0, E, names=QNAMES)["elem_state_Qdp"]
    check_bulk(h, whole["chunk"], QNAMES)
    if mode == tb.MODE_STRICT:
        want = s.copy()
        assert so.ssp_step(harness.PortOracle(), want, vstar, 0, QD, DT) == 1
        assert np.array_equal(bits(got), bits(want.arrays["elem_state_Qdp"]))
    else:
        hs = hp.from_state(s)
        so.ssp_step_hp(hs, vstar, 0, QD, DT)
        ref = hs.arrays["elem_state_Qdp"]
        for lvl in (0, 1):
            r, at, _ = hp.worst(got[:, :, lvl], ref[:, :, lvl])
            assert r <= so.k_ssp(1), (lvl, r, at)


# ---- the limiter -----------------------------------------------------------------------------------------------------

def test_limiter_past_2_31(whole):
    """caar_tracer_bounds and caar_limit_tracers on [15 000, 15 024), qsize 35, Qdp(1) with dp3d(2): bounds and limited
    Qdp equal limiter_oracle by bits; the bulk's bounds stay zero and its Qdp keeps its bits."""
    h = whole["h"]
    qtl, dtl = 1, 2
    inp = limiter_inputs(NT, L, QD, 7300, dtl)
    names = ("elem_spheremp", "elem_state_dp3d", "elem_state_Qdp")
    h.upload_range({n: inp[n] for n in names}, E0, E, names=names)
    B = np.zeros((E, QD, L, 2))
    h.upload_bounds(B)
    h.tracer_bounds(qtl, QD, dtl, nets=E0, nete=E)
    h.download_bounds(B)
    wb = np.zeros((NT, QD, L, 2))
    lo.tracer_bounds(inp["elem_state_Qdp"], inp["elem_state_dp3d"], wb, 0, NT, qtl, QD, dtl)
    assert np.array_equal(bits(B[E0:]), bits(wb))
    assert not B[:E0].any()
    B[E0:] = inp["bounds"][:, :, qtl]
    h.upload_bounds(B)
    h.limit_tracers(qtl, QD, dtl, nets=E0, nete=E)
    h.download_bounds(B)
    note_peak()
    got = h.download_range(E0, E, names=QNAMES)["elem_state_Qdp"]
    wQ, wb = inp["elem_state_Qdp"].copy(), np.ascontiguousarray(inp["bounds"][:, :, qtl])
    r = lo.limit_tracers(wQ, inp["elem_state_dp3d"], inp["elem_spheremp"], wb, 0, NT, qtl, QD, dtl)
    assert np.array_equal(bits(got), bits(wQ))
    assert np.array_equal(bits(B[E0:]), bits(wb))
    assert not B[:E0].any()
    assert (r["iters"] > 1).any()
    check_bulk(h, whole["chunk"], QNAMES)


# ---- the DSS and the neighbour bounds, whole and partitioned ---------------------------------------------------------

def test_dss_and_neighbor_minmax_whole_then_partitioned(whole):
    """caar_dss of Qdp(1), qsize 35, both weightings, and caar_neighbor_minmax(35) on the whole handle equal the oracles
    on the tail by bits. Then, with the whole handle closed, two handles hold [0, 15 012) and [15 012, 15 024): pack,
    segment move and unpack, and separately pack, move, interior and boundary, give the whole-mesh tail by bits, and so
    do the exchanged bounds. The bulk sample keeps its bits throughout."""
    h, gid, chunk = whole["h"], whole["gid"], whole["chunk"]
    conn = do.Connectivity(whole["tgid"])
    rng = np.random.default_rng(7400)
    sph = rng.uniform(0.5, 2.0, (NT, 4, 4))
    Q = rng.integers(0x4000000000000000, 0x4100000000000000, size=(NT, QD, 2, L, 4, 4),
                     dtype=np.uint64).view(np.float64)
    b = np.sort(rng.standard_normal((NT, QD, L, 2)), -1)
    b[rng.random(b.shape) < 0.3] = 0.0
    b[rng.random(b.shape) < 0.5] *= -1.0
    b = np.sort(b, -1)
    h.upload_range({"elem_spheremp": sph}, E0, E, names=("elem_spheremp",))
    h.set_connectivity(gid)
    ref = {}
    for w in (do.ASSEMBLE, do.PROJECT):
        h.upload_range({"elem_state_Qdp": Q}, E0, E, names=QNAMES)
        h.dss(QNAMES, qtl=1, qsize=QD, weighting=w)
        ref[w] = h.download_range(E0, E, names=QNAMES)["elem_state_Qdp"]
        want = {"elem_spheremp": sph, "elem_state_Qdp": Q.copy()}
        do.dss_arrays(want, conn, QNAMES, qtl=1, qsize=QD, weighting=w)
        assert np.array_equal(bits(ref[w]), bits(want["elem_state_Qdp"])), w
        check_bulk(h, chunk, QNAMES)
    B = np.zeros((E, QD, L, 2))
    B[E0:] = b
    h.upload_bounds(B)
    h.neighbor_minmax(QD)
    h.download_bounds(B)
    note_peak()
    ref_b = B[E0:].copy()
    assert np.array_equal(bits(ref_b), bits(do.neighbor_minmax_np(b, conn, QD)))
    assert not B[:E0].any()
    del B
    h.close()

    ps = np.array([0, CUT, E], dtype=np.int32)
    hs = [tb.Caar(CUT, L, QD), tb.Caar(E - CUT, L, QD)]
    names = ("elem_spheremp", "elem_state_Qdp")
    fill_bulk(hs[0], chunk, names)
    tail = {"elem_spheremp": sph, "elem_state_Qdp": Q}
    for p, (a, c) in enumerate(((E0, CUT), (CUT, E))):
        off = ps[p]
        hs[p].upload_range({n: np.ascontiguousarray(tail[n][a - E0:c - E0]) for n in names}, a - off, c - off,
                           names=names)
        hs[p].set_partition(gid, ps, p)
    note_peak()

    def parts_tail():
        return np.concatenate([hs[0].download_range(E0, CUT, names=QNAMES)["elem_state_Qdp"],
                               hs[1].download_range(0, E - CUT, names=QNAMES)["elem_state_Qdp"]])

    def reload():
        hs[0].upload_range({"elem_state_Qdp": np.ascontiguousarray(Q[:CUT - E0])}, E0, CUT, names=QNAMES)
        hs[1].upload_range({"elem_state_Qdp": np.ascontiguousarray(Q[CUT - E0:])}, 0, E - CUT, names=QNAMES)

    for w in (do.ASSEMBLE, do.PROJECT):
        reload()
        exchange_dss(hs, QNAMES, qtl=1, qsize=QD, weighting=w)
        assert np.array_equal(bits(parts_tail()), bits(ref[w])), ("unpack", w)
        reload()
        split_dss(hs, QNAMES, 0, 1, QD, w, "interior_first")
        assert np.array_equal(bits(parts_tail()), bits(ref[w])), ("interior + boundary", w)
        check_bulk(hs[0], chunk, QNAMES)
    B0 = np.zeros((CUT, QD, L, 2))
    B0[E0:] = b[:CUT - E0]
    hs[0].upload_bounds(B0)
    hs[1].upload_bounds(np.ascontiguousarray(b[CUT - E0:]))
    exchange_minmax(hs, QD)
    hs[0].download_bounds(B0)
    note_peak()
    assert np.array_equal(bits(np.concatenate([B0[E0:], hs[1].download_bounds()])), bits(ref_b))
    assert not B0[:E0].any()
    for x in hs:
        x.close()


def test_zz_report_peak(capsys):
    """Not a gate: the largest device memory in use that this module saw (all processes on the device)."""
    with capsys.disabled():
        print(f"\n[large offsets] peak device memory in use {PEAK.get('used', 0) / 1e9:.1f} GB")
