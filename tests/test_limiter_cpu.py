"""The two transcriptions of HOMME's quasi-monotone limiter in tests/limiter_oracle.py, on the CPU: they agree bit for
bit on a mix of random problems; on dyadic hand cases, where every operation is exact, they give the answers an exact
rational transcription gives; their outputs have the properties the algorithm promises; and four defective limiters
each fail at least one of these checks."""
import math
from fractions import Fraction as F

import numpy as np
import pytest

import limiter_oracle as lo

U = 2.0 ** -53
CATEGORIES = ("in_bounds", "over", "under", "both", "relax_low", "relax_high", "sumc_le_0", "staircase")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def staircase_weights(rng, n):
    """(n, 16) weights falling geometrically from point 0, by a ratio in [0.2, 1] per point"""
    return rng.uniform(0.2, 1.0, n)[:, None] ** np.arange(16) * rng.uniform(0.9, 1.1, (n, 16))


def staircase(rng, n, c=None):
    """n problems that saturate about one point per pass (many passes, often MAXITER): with weights c falling
    geometrically (staircase_weights unless given), point 0 is over maxp = 1 and point j sits so that pass j pushes it
    over by a fraction f of that pass's increment -> (x, c), both permuted over the points unless c is given."""
    given = c is not None
    c = staircase_weights(rng, n) if c is None else c
    f = rng.uniform(0.3, 0.95, n)
    E = rng.uniform(0.1, 2.0, n) * c[:, 0]
    x = np.empty((n, 16))
    x[:, 0] = 1.0 + E / c[:, 0]
    moved = np.zeros(n)
    for j in range(1, 16):
        inc = E / c[:, j:].sum(1)
        x[:, j] = 1.0 - (moved + inc * (1 - f))
        moved += inc
        E = f * inc * c[:, j]
    if given:
        return x, c
    perm = rng.permuted(np.tile(np.arange(16), (n, 1)), axis=1)
    return np.take_along_axis(x, perm, 1), np.take_along_axis(c, perm, 1)


def random_problems(n, seed):
    """n problems, an equal share of each of CATEGORIES -> dict(p, d, w (n, 16) in C order; minp, maxp (n,); cat)."""
    rng = np.random.default_rng(seed)
    cat = np.arange(n) % len(CATEGORIES)
    x = rng.uniform(0.0, 1.0, (n, 16)) * rng.uniform(1e-3, 1e3, (n, 1))
    d = rng.uniform(0.5, 2.0, (n, 16)) * 10.0 ** rng.uniform(-2, 3, (n, 1))
    w = rng.uniform(0.5, 2.0, (n, 16)) * 10.0 ** rng.uniform(-6, 0, (n, 1))
    xs = np.sort(x, 1)
    lo_, hi_ = xs[:, 0], xs[:, -1]
    span = hi_ - lo_
    minp, maxp = lo_ - rng.uniform(0, 0.1, n) * span, hi_ + rng.uniform(0, 0.1, n) * span
    pick = lambda k: xs[np.arange(n), rng.integers(k[0], k[1], n)]
    over, under = cat == 1, cat == 2
    both = cat == 3
    maxp = np.where(over | both, pick((8, 15)), maxp)
    minp = np.where(under | both, pick((1, 8)), minp)
    minp = np.where(cat == 4, hi_ + span, minp)           # the bounds above every value: minp relaxes
    maxp = np.where(cat == 4, hi_ + 2 * span, maxp)
    maxp = np.where(cat == 5, lo_ - span * 0.5, maxp)     # below every value: maxp relaxes
    minp = np.where(cat == 5, lo_ - span, minp)
    nz = cat == 6                                        # sumc <= 0: zero or negative weights
    w[nz] = np.where(rng.random((nz.sum(), 1)) < 0.5, 0.0, -w[nz])
    st = cat == 7
    xs7, c7 = staircase(rng, int(st.sum()))
    scale = x[st, :1]
    x[st] = xs7 * scale
    w[st] = c7 / d[st]
    minp[st], maxp[st] = 0.0, scale[:, 0]
    return dict(p=x * d, d=d, w=w, minp=minp, maxp=maxp, cat=cat)


def run_scalar(pr, idx=None):
    idx = range(len(pr["minp"])) if idx is None else idx
    out = dict(p=[], minp=[], maxp=[], x=[], iters=[], exit=[])
    for i in idx:
        r = lo.limit_problem(pr["p"][i], pr["d"][i], pr["w"][i], float(pr["minp"][i]), float(pr["maxp"][i]))
        for k, v in zip(("p", "minp", "maxp", "x", "iters", "exit"), r):
            out[k].append(v)
    return {k: np.array(v) for k, v in out.items()}


def run_np(pr, defect=None, idx=slice(None)):
    return lo.limit_np(pr["p"][idx], pr["d"][idx], pr["w"][idx], pr["minp"][idx], pr["maxp"][idx], defect=defect)


def compare(a, b):
    """names of the outputs in which two limiter results differ (bits, or counts)"""
    bad = [k for k in ("p", "minp", "maxp", "x") if not np.array_equal(bits(a[k]), bits(b[k]))]
    return bad + [k for k in ("iters", "exit") if not np.array_equal(a[k], b[k])]


@pytest.fixture(scope="module")
def mix():
    pr = random_problems(100_008, 8100)
    return pr, run_np(pr)


def test_scalar_and_numpy_agree_bit_for_bit(mix, capsys):
    """10^5 problems of every category: the literal scalar transcription and the vectorised one give the same Qdp,
    relaxed bounds, pass counts and exits. The mix covers relaxation on both sides, sumc <= 0, >= 10 passes, MAXITER."""
    pr, got = mix
    want = run_scalar(pr)
    assert compare(got, want) == []
    hist = np.bincount(got["iters"], minlength=lo.MAXITER + 1)
    n_max, n_ws0 = int((got["exit"] == lo.EXIT_MAXITER).sum()), int((got["exit"] == lo.EXIT_WS0).sum())
    with capsys.disabled():
        print(f"\n[limiter] passes histogram {hist.tolist()}; MAXITER exits {n_max}; ws == 0 exits {n_ws0}")
    assert (got["iters"] >= 10).sum() > 1000 and n_max > 0
    assert (got["exit"] == lo.EXIT_NONE).sum() == (pr["cat"] == 6).sum()
    assert (got["minp"] < pr["minp"]).sum() > 1000 and (got["maxp"] > pr["maxp"]).sum() > 1000   # relaxation
    moved = ~np.all(bits(got["p"]) == bits(pr["p"] / pr["d"] * pr["d"]), axis=1)
    for k in (1, 2, 3):
        assert moved[pr["cat"] == k].mean() > 0.9, CATEGORIES[k]


# ---- hand cases: dyadic inputs, exact arithmetic ---------------------------------------------------------------------

def limit_exact(p, d, w, minp, maxp):
    """The same algorithm in exact rational arithmetic -> (p, minp, maxp) as Fractions, C order."""
    c = [F(w[o]) * F(d[o]) for o in lo.FORTRAN]
    x = [F(p[o]) / F(d[o]) for o in lo.FORTRAN]
    minp, maxp = F(minp), F(maxp)
    sumc = sum(c)
    if sumc <= 0:
        return [F(v) for v in p], minp, maxp
    mass = sum(ci * xi for ci, xi in zip(c, x))
    minp = min(minp, mass / sumc)
    maxp = max(maxp, mass / sumc)
    for _ in range(lo.MAXITER):
        add = F(0)
        for n in range(16):
            if x[n] > maxp:
                add += (x[n] - maxp) * c[n]
                x[n] = maxp
            if x[n] < minp:
                add -= (minp - x[n]) * c[n]
                x[n] = minp
        if abs(add) <= F(lo.TOL) * abs(mass):
            break
        sel = [(x[n] < maxp) if add > 0 else (x[n] > minp) for n in range(16)]
        ws = sum(c[n] for n in range(16) if sel[n])
        if ws == 0:
            break
        x = [x[n] + add / ws if sel[n] else x[n] for n in range(16)]
    out = [F(0)] * 16
    for n, o in enumerate(lo.FORTRAN):
        out[o] = x[n] * F(d[o])
    return out, minp, maxp


def _two_pass():
    """c = 1 at the over point (x = 10), 8 at a point 0.25 below maxp = 2, and 8 spread over the other 14 (12 x 0.5,
    2 x 1) at x = 1: pass 1 spreads 8 over a weight of 16 and pushes the heavy point over by 0.25, pass 2 spreads the
    2 it gives back over 8; every value is dyadic."""
    c = np.array([1.0, 8.0] + [0.5] * 12 + [1.0, 1.0])
    x = np.array([10.0, 1.75] + [1.0] * 14)
    return x, c, 0.0, 2.0, np.array([2.0, 2.0] + [1.75] * 14), (0.0, 2.0)


HAND = {
    # name: (x, c, minp, maxp, x wanted, bounds wanted), x and c in Fortran point order
    "one_over_spreads_evenly": (np.array([17.0] + [1.0] * 15), np.ones(16), 0.0, 2.0, np.full(16, 2.0), (0.0, 2.0)),
    "one_under_spreads_evenly": (np.array([-15.0] + [3.0] * 15), np.ones(16), 0.0, 4.0,
                                 np.array([0.0] + [2.0] * 15), (0.0, 4.0)),
    "relax_max": (np.full(16, 3.0), np.ones(16), 0.0, 2.0, np.full(16, 3.0), (0.0, 3.0)),
    "relax_min": (np.full(16, 0.5), np.full(16, 0.25), 1.0, 2.0, np.full(16, 0.5), (0.5, 2.0)),
    "two_passes": _two_pass(),
    "sumc_zero": (np.array([9.0] + [1.0] * 15), np.zeros(16), 0.0, 2.0, np.array([9.0] + [1.0] * 15), (0.0, 2.0)),
}


def hand_problem(name):
    """(p, d, w) in C order with d = 2 (so p = 2 x and w = c/2, still dyadic), minp, maxp, wanted p, wanted bounds."""
    x, c, mn, mx, xw, bw = HAND[name]
    xc, cc, xwc = np.empty(16), np.empty(16), np.empty(16)
    xc[lo.FORTRAN], cc[lo.FORTRAN], xwc[lo.FORTRAN] = x, c, xw
    d = np.full(16, 2.0)
    return xc * d, d, cc / d, mn, mx, xwc * d, bw


def hand_failures(defect=None):
    """names of the hand cases on which limit_np(defect) misses the exact answer"""
    bad = []
    for name in HAND:
        p, d, w, mn, mx, pw, bw = hand_problem(name)
        r = lo.limit_np(p[None], d[None], w[None], np.array([mn]), np.array([mx]), defect=defect)
        if not (np.array_equal(r["p"][0], pw) and (r["minp"][0], r["maxp"][0]) == bw):
            bad.append(name)
    return bad


@pytest.mark.parametrize("name", list(HAND))
def test_hand_case_is_exact(name):
    p, d, w, mn, mx, pw, bw = hand_problem(name)
    ep, emn, emx = limit_exact(p, d, w, mn, mx)
    assert [F(v) for v in pw] == ep and (F(bw[0]), F(bw[1])) == (emn, emx)      # the worked answer is the exact one
    sp, smn, smx, _, _, _ = lo.limit_problem(p, d, w, mn, mx)
    assert [F(v) for v in sp] == ep and (F(smn), F(smx)) == (emn, emx)
    assert hand_failures() == []


# ---- properties --------------------------------------------------------------------------------------------------

def property_failures(pr, r):
    """names of the promised properties that the limiter result r on problems pr violates"""
    bad = []
    p, d, w = pr["p"], pr["d"], pr["w"]
    F_ = lo.FORTRAN
    with np.errstate(all="ignore"):
        c, x0 = w * d, p / d
        act = r["exit"] != lo.EXIT_NONE
        # in bounds on a tolerance exit
        t = r["exit"] == lo.EXIT_TOL
        if not np.all((r["x"][t] >= r["minp"][t, None]) & (r["x"][t] <= r["maxp"][t, None])):
            bad.append("in_bounds_after_tolerance_exit")
        # mass within TOL |mass| plus rounding: each pass rounds at most 3 operations on every point's share
        m = act & (r["exit"] != lo.EXIT_WS0)
        cm, xm0, xm1 = c[m], x0[m], r["x"][m]
        mass0 = np.array([math.fsum(v) for v in cm * xm0])
        mass1 = np.array([math.fsum(v) for v in cm * xm1])
        big = np.maximum(np.abs(xm0), np.maximum(np.abs(r["minp"][m]), np.abs(r["maxp"][m]))[:, None])
        S = (np.abs(cm) * big).sum(1)
        allow = lo.TOL * np.abs(mass0) + 64 * (r["iters"][m] + 2) * U * S
        if not np.all(np.abs(mass1 - mass0) <= allow):
            bad.append("mass_conserved")
        # a problem in bounds changes by the p/d*d round trip only
        inb = act & np.all((x0 >= pr["minp"][:, None]) & (x0 <= pr["maxp"][:, None]), axis=1)
        if not np.array_equal(bits(r["p"][inb]), bits(x0[inb] * d[inb])):
            bad.append("in_bounds_unchanged")
        # sumc <= 0 untouched
        sumc = np.zeros(len(p))
        for o in F_:
            sumc = sumc + c[:, o]
        z = sumc <= 0
        if not (np.array_equal(bits(r["p"][z]), bits(p[z])) and np.array_equal(bits(r["minp"][z]), bits(pr["minp"][z]))
                and np.array_equal(bits(r["maxp"][z]), bits(pr["maxp"][z])) and np.array_equal(z, ~act)):
            bad.append("sumc_le_0_untouched")
        # the relaxed bounds are written back
        mass = np.zeros(len(p))
        for o in F_:
            mass = mass + c[:, o] * x0[:, o]
        emin = np.where(act & (mass < pr["minp"] * sumc), mass / sumc, pr["minp"])
        emax = np.where(act & (mass > pr["maxp"] * sumc), mass / sumc, pr["maxp"])
        if not (np.array_equal(bits(r["minp"]), bits(emin)) and np.array_equal(bits(r["maxp"]), bits(emax))):
            bad.append("relaxed_bounds_written")
    return bad


def test_properties(mix):
    pr, r = mix
    assert property_failures(pr, r) == []


@pytest.mark.parametrize("defect", lo.DEFECTS)
def test_defect_is_caught(mix, defect):
    """Each defective limiter fails the bit comparison with the scalar transcription, a hand case or a property."""
    pr, _ = mix
    idx = np.arange(0, len(pr["minp"]), 50)
    sub = {k: v[idx] for k, v in pr.items()}
    r = run_np(pr, defect)
    caught = property_failures(pr, r) + hand_failures(defect)
    caught += ["bits_vs_scalar"] if compare(run_np(sub, defect), run_scalar(sub)) else []
    assert caught, defect
