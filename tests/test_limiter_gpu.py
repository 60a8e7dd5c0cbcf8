"""caar_tracer_bounds and caar_limit_tracers (HOMME's quasi-monotone limiter, limiter_option 8) on the GPU, bit for bit
against the numpy transcription of tests/limiter_oracle.py: at nlev 72, 30, 128, 5, 80 and 127, qsize < qsize_d and
qsize = qsize_d = 35, sub-ranges, both
qtl, dp_tl != qtl and a size where every warp walks many tiles, with sentinels wherever the calls must not write;
after a strict and a fast caar_advect_tracers step; at 86400 x 72 on a sample of elements, with the whole output
bounded and conserving mass; plus argument checks, launch counts and run-to-run bits."""
import ctypes as C

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
import limiter_oracle as lo
import tracer_ssp_oracle as so
from oracle import harness
from test_limiter_cpu import staircase, staircase_weights
from test_pointwise_cpu import level_local_inputs

pytestmark = pytest.mark.gpu
INVALID = 1
NAMES = ("elem_spheremp", "elem_state_dp3d", "elem_state_Qdp")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def sentinel(rng, shape):
    return rng.integers(0x4000000000000000, 0x4100000000000000, size=shape, dtype=np.uint64).view(np.float64)


def limiter_inputs(E, L, Qd, seed, dp_tl, ntl=3):
    """dict of spheremp, dp3d, Qdp (both levels of mixing ratio x times dp3d(dp_tl)) and bounds [E][Qd][L][2] for the
    level-0 and level-1 problems alike. Elements e % 7 == 5 have sumc <= 0 (zero or negative spheremp); elements
    e % 7 == 3 have dp3d = 1 and geometric spheremp with staircase mixing ratios (many passes, MAXITER); the others mix
    bounds that hold, are exceeded above, below or both, and lie wholly above or below the values (relaxation)."""
    rng = np.random.default_rng(seed)
    sph = rng.uniform(0.5, 2.0, (E, 4, 4)) * 10.0 ** rng.uniform(-2, 0, (E, 1, 1))
    dp = rng.uniform(0.5, 2.0, (E, ntl, L, 4, 4)) * 10.0 ** rng.uniform(0, 3, (E, 1, L, 1, 1))
    x = rng.uniform(0.0, 1.0, (E, Qd, 2, L, 4, 4)) * 10.0 ** rng.uniform(-3, 3, (E, Qd, 1, 1, 1, 1))
    zero = np.arange(E) % 7 == 5
    sph[zero] *= np.where(np.arange(zero.sum()) % 2 == 0, 0.0, -1.0)[:, None, None]
    xf = x.reshape(E, Qd, 2, L, 16)
    xs = np.sort(xf, -1)
    lo_, hi_ = xs[..., 0], xs[..., -1]
    span = hi_ - lo_
    cat = (np.arange(Qd)[:, None, None] + np.arange(L)[None, None, :] + np.arange(2)[None, :, None]) % 6
    cat = np.broadcast_to(cat, lo_.shape)
    pick = lambda i: xs[..., i]
    mn = np.select([cat == 2, cat == 3, cat == 4, cat == 5], [pick(4), pick(3), hi_ + span, lo_ - span], lo_ - 0.05 * span)
    mx = np.select([cat == 1, cat == 3, cat == 4, cat == 5], [pick(12), pick(11), hi_ + 2 * span, lo_ - 0.5 * span],
                   hi_ + 0.05 * span)
    stair = np.flatnonzero(np.arange(E) % 7 == 3)
    for e in stair:
        dp[e] = 1.0
        cF = staircase_weights(rng, 1)[0]
        sph[e].reshape(16)[lo.FORTRAN] = cF
        n = Qd * 2 * L
        xF, _ = staircase(rng, n, np.tile(cF, (n, 1)))
        scale = 10.0 ** rng.uniform(-3, 3, (n, 1))
        xe = np.empty((n, 16))
        xe[:, lo.FORTRAN] = xF * scale
        xf[e] = xe.reshape(Qd, 2, L, 16)
        mn[e], mx[e] = 0.0, scale.reshape(Qd, 2, L)
    Qdp = x * dp[:, dp_tl][:, None, None]
    b = np.stack([mn, mx], -1)                       # [E][Qd][2][L][2]: the bounds of each level's problems
    return dict(elem_spheremp=sph, elem_state_dp3d=dp, elem_state_Qdp=np.ascontiguousarray(Qdp), bounds=b)


def with_sentinels(inp, lo_e, hi_e, qsize, qtl, seed):
    """Qdp sentinels outside the problems (other elements, tracers iq >= qsize, the other level) and bounds [E][Qd][L][2]
    for level qtl with sentinels outside the problems."""
    rng = np.random.default_rng(seed)
    Q = inp["elem_state_Qdp"]
    for part in (np.s_[:lo_e], np.s_[hi_e:], np.s_[lo_e:hi_e, qsize:], np.s_[lo_e:hi_e, :qsize, 1 - qtl]):
        Q[part] = sentinel(rng, Q[part].shape)
    b = np.ascontiguousarray(inp["bounds"][:, :, qtl])
    for part in (np.s_[:lo_e], np.s_[hi_e:], np.s_[lo_e:hi_e, qsize:]):
        b[part] = sentinel(rng, b[part].shape)
    return b


def handle(E, L, Qd, arrays, ntl=3):
    h = tb.Caar(E, L, Qd, ntl)
    full = {n: np.ascontiguousarray(arrays[n]) for n in NAMES}
    h.upload(full, names=NAMES)
    return h


def download(h, E, L, Qd, ntl=3):
    out = {n: np.empty(tb.field_shape(n, E, L, Qd, ntl)) for n in NAMES}
    h.download(out, names=NAMES)
    return out


CASES = [
    dict(E=40, L=72, Qd=5, qsize=4, range=(0, 40), qtl=0, dp_tl=0, seed=1),
    dict(E=33, L=30, Qd=4, qsize=2, range=(3, 30), qtl=1, dp_tl=2, seed=2),
    dict(E=17, L=128, Qd=3, qsize=3, range=(1, 16), qtl=0, dp_tl=1, seed=3),
    dict(E=24, L=72, Qd=2, qsize=1, range=(4, 6), qtl=1, dp_tl=1, seed=4),
    # 2990 x 4 x 72 problems: 26910 tiles of 32, about 11 per warp of one resident wave
    dict(E=3000, L=72, Qd=5, qsize=4, range=(5, 2995), qtl=1, dp_tl=0, seed=5),
    # odd and E3SM v3 level counts; 35 of 35 tracers: no tracer outside the selection and the longest bounds rows
    dict(E=35, L=5, Qd=3, qsize=2, range=(2, 34), qtl=1, dp_tl=2, seed=6),
    dict(E=36, L=80, Qd=4, qsize=3, range=(1, 35), qtl=0, dp_tl=1, seed=7),
    dict(E=9, L=127, Qd=35, qsize=35, range=(0, 9), qtl=1, dp_tl=0, seed=8),
]


def case_id(c):
    return f"E{c['E']}-L{c['L']}-q{c['qsize']}of{c['Qd']}-r{c['range'][0]}:{c['range'][1]}-qtl{c['qtl']}-dp{c['dp_tl']}"


def run_case(c):
    """-> (inputs, bounds after caar_tracer_bounds, arrays after it, bounds and arrays after caar_limit_tracers,
    the oracle's (bounds, arrays, result) for both)"""
    E, L, Qd, qs, (a, b), qtl, dtl = c["E"], c["L"], c["Qd"], c["qsize"], c["range"], c["qtl"], c["dp_tl"]
    inp = limiter_inputs(E, L, Qd, c["seed"], dtl)
    bnd = with_sentinels(inp, a, b, qs, qtl, c["seed"])
    h = handle(E, L, Qd, inp)
    h.upload_bounds(bnd)
    n0 = h.launch_count()
    h.tracer_bounds(qtl, qs, dtl, nets=a, nete=b)
    gb1, ga1 = h.download_bounds(), download(h, E, L, Qd)
    h.upload_bounds(bnd)
    h.limit_tracers(qtl, qs, dtl, nets=a, nete=b)
    gb2, ga2 = h.download_bounds(), download(h, E, L, Qd)
    assert h.launch_count() - n0 == 2
    h.close()
    wb1 = bnd.copy()
    lo.tracer_bounds(inp["elem_state_Qdp"], inp["elem_state_dp3d"], wb1, a, b, qtl, qs, dtl)
    wb2, wQ = bnd.copy(), inp["elem_state_Qdp"].copy()
    r = lo.limit_tracers(wQ, inp["elem_state_dp3d"], inp["elem_spheremp"], wb2, a, b, qtl, qs, dtl)
    return inp, (gb1, ga1, gb2, ga2), (wb1, wb2, wQ, r)


@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_kernels_equal_oracle(c):
    """Both calls equal the numpy transcription in every bit: the bounds (sentinels outside the problems kept), the
    limited Qdp (sentinels at other elements, tracers iq >= qsize and the other level kept), the relaxed bounds; dp3d and
    spheremp untouched, Qdp untouched by caar_tracer_bounds."""
    inp, (gb1, ga1, gb2, ga2), (wb1, wb2, wQ, r) = run_case(c)
    assert np.array_equal(bits(gb1), bits(wb1))
    assert np.array_equal(bits(ga1["elem_state_Qdp"]), bits(inp["elem_state_Qdp"]))
    assert np.array_equal(bits(gb2), bits(wb2))
    assert np.array_equal(bits(ga2["elem_state_Qdp"]), bits(wQ))
    for ga in (ga1, ga2):
        for n in ("elem_spheremp", "elem_state_dp3d"):
            assert np.array_equal(bits(ga[n]), bits(inp[n])), n
    if r is not None and c["E"] >= 33:   # the mix reaches what it is for
        assert (r["exit"] == lo.EXIT_NONE).any() and (r["exit"] == lo.EXIT_MAXITER).any() and (r["iters"] >= 10).any()
        assert not np.array_equal(bits(wQ), bits(inp["elem_state_Qdp"]))


# ---- composition with the tracer step ------------------------------------------------------------------------------

QNAMES = ("elem_Dinv", "elem_metdet", "elem_rmetdet", "elem_spheremp", "elem_state_dp3d", "elem_state_Qdp")
DT = 150.0


@pytest.mark.parametrize("L", [72, 30])
def test_strict_step_composition(L):
    """bounds(qn0) -> strict caar_advect_tracers -> limit(new qn0), on a sub-range with qsize < qsize_d: equal in every
    bit to tracer_ssp_oracle.ssp_step between the oracle's bounds and limiter."""
    E, Qd, qs, a, b, dtl = 9, 4, 3, 1, 8, 1
    s, vstar, _, _ = level_local_inputs("randomize", E, L, 6100 + L, qsize_d=Qd)
    want = s.copy()
    want.ctl[0:2] = (a, b)
    h = tb.Caar(E, L, Qd, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays, names=QNAMES)
    h.upload_vstar(vstar)
    h.tracer_bounds(0, qs, dtl, nets=a, nete=b)
    q = h.advect_tracers(0, qs, DT, 1, tb.MODE_STRICT, nets=a, nete=b)
    h.limit_tracers(q, qs, dtl, nets=a, nete=b)
    got = {"elem_state_Qdp": np.empty_like(s.arrays["elem_state_Qdp"])}
    h.download(got, names=("elem_state_Qdp",))
    gb = h.download_bounds()
    h.close()
    wb = np.zeros((E, Qd, L, 2))
    A = want.arrays
    lo.tracer_bounds(A["elem_state_Qdp"], A["elem_state_dp3d"], wb, a, b, 0, qs, dtl)
    qw = so.ssp_step(harness.PortOracle(), want, vstar, 0, qs, DT)
    assert qw == q
    r = lo.limit_tracers(A["elem_state_Qdp"], A["elem_state_dp3d"], A["elem_spheremp"], wb, a, b, q, qs, dtl)
    assert np.array_equal(bits(got["elem_state_Qdp"]), bits(A["elem_state_Qdp"]))
    assert np.array_equal(bits(gb), bits(wb))
    assert (r["iters"] > 1).any()       # the step left values outside the bounds of its input


def test_fast_step_then_limiter():
    """The GPU limiter on the Qdp a fast caar_advect_tracers step left equals the oracle limiter on the downloaded Qdp."""
    E, L, Qd, qs, dtl = 12, 72, 3, 3, 0
    s, vstar, _, _ = level_local_inputs("randomize", E, L, 6200, qsize_d=Qd)
    h = tb.Caar(E, L, Qd, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    h.upload(s.arrays, names=QNAMES)
    h.upload_vstar(vstar)
    h.tracer_bounds(1, qs, dtl)
    q = h.advect_tracers(1, qs, DT, 1, tb.MODE_FAST)
    mid = {"elem_state_Qdp": np.empty_like(s.arrays["elem_state_Qdp"])}
    h.download(mid, names=("elem_state_Qdp",))
    b0 = h.download_bounds()
    h.limit_tracers(q, qs, dtl)
    got = {"elem_state_Qdp": np.empty_like(s.arrays["elem_state_Qdp"])}
    h.download(got, names=("elem_state_Qdp",))
    gb = h.download_bounds()
    h.close()
    wQ = mid["elem_state_Qdp"].copy()
    r = lo.limit_tracers(wQ, s.arrays["elem_state_dp3d"], s.arrays["elem_spheremp"], b0, 0, E, q, qs, dtl)
    assert np.array_equal(bits(got["elem_state_Qdp"]), bits(wQ))
    assert np.array_equal(bits(gb), bits(b0))
    assert (r["iters"] > 1).any()


# ---- full size ------------------------------------------------------------------------------------------------------

def test_full_size_86400x72():
    """86400 x 72, qsize 4 (a pool of 343 elements tiled over the handle): bounds of Qdp(0), limiter on Qdp(1) = Qdp(0)
    perturbed by up to 5 %. A seeded sample of 48 elements equals the oracle bit for bit; over every problem the result
    lies in its relaxed bounds to 1e-12 and keeps its mass to 1e-12."""
    E, L, Qd, POOL, dtl = 86400, 72, 4, 343, 0
    rng = np.random.default_rng(6300)
    sph = rng.uniform(0.5, 2.0, (POOL, 4, 4))
    dp = rng.uniform(0.5, 2.0, (POOL, 3, L, 4, 4)) * 10.0 ** rng.uniform(0, 3, (POOL, 1, L, 1, 1))
    x0 = rng.uniform(0.0, 1.0, (POOL, Qd, 1, L, 4, 4)) * 10.0 ** rng.uniform(-3, 3, (POOL, Qd, 1, L, 1, 1))
    x1 = x0 * rng.uniform(0.95, 1.05, x0.shape)
    pool = dict(elem_spheremp=sph, elem_state_dp3d=dp,
                elem_state_Qdp=np.concatenate([x0, x1], 2) * dp[:, dtl][:, None, None])
    h = tb.Caar(E, L, Qd)
    for e0 in range(0, E, POOL):
        e1 = min(E, e0 + POOL)
        h.upload_range({n: np.ascontiguousarray(v[:e1 - e0]) for n, v in pool.items()}, e0, e1, names=NAMES)
    n0 = h.launch_count()
    h.tracer_bounds(0, Qd, dtl)
    h.limit_tracers(1, Qd, dtl)
    assert h.launch_count() - n0 == 2
    Qg = np.empty(tb.field_shape("elem_state_Qdp", E, L, Qd))
    h.download({"elem_state_Qdp": Qg}, names=("elem_state_Qdp",))
    bg = h.download_bounds()
    h.close()
    sample = np.sort(rng.choice(E, 48, replace=False))
    P = sample % POOL
    wQ, wb = pool["elem_state_Qdp"][P].copy(), np.zeros((48, Qd, L, 2))
    lo.tracer_bounds(wQ, dp[P], wb, 0, 48, 0, Qd, dtl)
    lo.limit_tracers(wQ, dp[P], sph[P], wb, 0, 48, 1, Qd, dtl)
    assert np.array_equal(bits(Qg[sample]), bits(wQ))
    assert np.array_equal(bits(bg[sample]), bits(wb))
    for e0 in range(0, E, 4 * POOL):   # bounded and mass-conserving, chunk by chunk
        e1 = min(E, e0 + 4 * POOL)
        idx = np.arange(e0, e1) % POOL
        d = dp[idx, dtl][:, None]                               # [n][1][L][4][4]
        x = Qg[e0:e1, :, 1] / d
        mn, mx = bg[e0:e1, ..., 0][..., None, None], bg[e0:e1, ..., 1][..., None, None]
        scale = np.maximum(np.abs(mn), np.abs(mx))
        assert np.all(x >= mn - 1e-12 * scale) and np.all(x <= mx + 1e-12 * scale)
        c = sph[idx][:, None, None] * d
        m0 = (c * pool["elem_state_Qdp"][idx, :, 1] / d).reshape(e1 - e0, Qd, L, 16).sum(-1)
        m1 = (c * x).reshape(e1 - e0, Qd, L, 16).sum(-1)
        assert np.all(np.abs(m1 - m0) <= 1e-12 * np.abs(m0))


# ---- checks, counts, reproducibility ---------------------------------------------------------------------------------

def test_checks_counts_and_no_params():
    """Every argument error returns CAAR_ERR_INVALID, launches nothing and leaves Qdp and the bounds as they were; the
    calls need no caar_set_params; each call with work is one launch, an empty range or qsize 0 none."""
    lib = tb.load_library()
    E, L, Qd, ntl = 6, 16, 3, 3
    inp = limiter_inputs(E, L, Qd, 7, 0)
    h = handle(E, L, Qd, inp)                    # caar_set_params is never called
    bnd = np.ascontiguousarray(inp["bounds"][:, :, 0])
    h.upload_bounds(bnd)
    buf = np.zeros(E * Qd * L * 2)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    assert lib.caar_bounds_upload(None, dp(buf)) == INVALID and lib.caar_bounds_download(None, dp(buf)) == INVALID
    assert lib.caar_bounds_upload(h.h, None) == INVALID and lib.caar_bounds_download(h.h, None) == INVALID
    good = dict(nets=0, nete=E, qtl=0, qsize=2, dp_tl=1)
    bad = [dict(nets=-1), dict(nete=E + 1), dict(nets=4, nete=3), dict(qtl=-1), dict(qtl=2), dict(dp_tl=-1),
           dict(dp_tl=ntl), dict(qsize=-1), dict(qsize=Qd + 1)]
    for fn in (lib.caar_tracer_bounds, lib.caar_limit_tracers):
        # the good calls of the previous function rewrote the bounds (and the limiter Qdp): start each from the inputs
        h.upload({n: np.ascontiguousarray(inp[n]) for n in NAMES}, names=NAMES)
        h.upload_bounds(bnd)
        Q0, B0 = download(h, E, L, Qd)["elem_state_Qdp"], h.download_bounds()
        assert np.array_equal(bits(B0), bits(bnd))
        assert fn(None, *good.values()) == INVALID
        for over in bad:
            a = {**good, **over}
            n = h.launch_count()
            assert fn(h.h, *a.values()) == INVALID, (fn, over)
            h.sync()
            assert h.launch_count() == n, over
            assert np.array_equal(bits(download(h, E, L, Qd)["elem_state_Qdp"]), bits(Q0)), over
            assert np.array_equal(bits(h.download_bounds()), bits(B0)), over
        for over, launches in ((dict(), 1), (dict(nets=3, nete=3), 0), (dict(qsize=0), 0), (dict(qsize=Qd), 1)):
            n = h.launch_count()
            assert fn(h.h, *{**good, **over}.values()) == 0, over
            h.sync()
            assert h.launch_count() - n == launches, over
    h.close()
    fresh = tb.Caar(E, L, Qd)                      # bounds are zero on first use
    assert not fresh.download_bounds().any()
    fresh.close()


def test_two_runs_reproduce_bits():
    c = CASES[-1]
    runs = [run_case(c)[1] for _ in range(2)]
    for a, b in zip(runs[0][2:], runs[1][2:]):
        if isinstance(a, dict):
            a, b = a["elem_state_Qdp"], b["elem_state_Qdp"]
        assert np.array_equal(bits(a), bits(b))
