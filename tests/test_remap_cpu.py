"""The two transcriptions of HOMME's PPM vertical remap (tests/remap_oracle.py) agree bit for bit at nlev 2 .. 128 in
three deformation regimes, and the remap has the properties HOMME relies on: column mass conserved, a constant mixing
ratio kept, the identity where dp_star == dp, no new extrema under a deformation of under one cell. Each defect of
remap_oracle.DEFECTS is told apart from the scalar transcription."""
import numpy as np
import pytest

import remap_oracle as ro

LEVELS = [2, 3, 5, 26, 72, 127, 128]


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def problem(N, L, regime, seed):
    """dpo, dpn (N, L) and three fields: mass of a mixing ratio, T*dpo and v*dpo"""
    dpo = ro.columns(N, L, regime, seed)
    hyai, hybi = ro.coordinate(L)
    dpn = ro.target_dp(dpo, hyai, hybi, ro.PS0)
    rng = np.random.default_rng(seed + 1)
    q = ro.mixing_ratios(N, L, seed + 2)
    T = 200.0 + 100.0 * rng.random((N, L))
    v = rng.uniform(-40.0, 40.0, (N, L))
    return dpo, dpn, [q * dpo, T * dpo, v * dpo], q


@pytest.mark.parametrize("regime", ro.REGIMES)
@pytest.mark.parametrize("L", LEVELS)
def test_scalar_and_numpy_agree(L, regime):
    N = 6 if L <= 72 else 3
    dpo, dpn, fields, _ = problem(N, L, regime, 100 + L)
    got = ro.remap_np(dpo, dpn, fields)
    for c in range(N):
        want = ro.remap_column(list(dpo[c]), list(dpn[c]), [list(f[c]) for f in fields])
        for g, w in zip(got, want):
            assert np.array_equal(bits(g[c]), bits(np.array(w))), (c,)
    if regime == "over" and L >= 26:   # the regime reaches the extrapolation of cell k-1
        kid = ro.grid_np(dpo, dpn)["kid"][:, 1:]
        assert (kid == np.arange(L)[None, :]).any()


@pytest.mark.parametrize("regime", ro.REGIMES)
@pytest.mark.parametrize("L", LEVELS)
def test_mass_conserved_and_constant_kept(L, regime):
    dpo, dpn, fields, _ = problem(40, L, regime, 200 + L)
    const = 3.7e-3 * dpo
    out = ro.remap_np(dpo, dpn, fields + [const])
    for f, g in zip(fields, out):
        m0, m1 = f.sum(1), g.sum(1)
        assert np.all(np.abs(m1 - m0) <= 1e-12 * np.abs(f).sum(1))
    assert np.allclose(out[-1] / dpn, 3.7e-3, rtol=1e-12, atol=0)


@pytest.mark.parametrize("L", LEVELS)
def test_identity_when_dp_star_is_dp(L):
    dpo, dpn, fields, _ = problem(30, L, "identity", 300 + L)
    assert np.allclose(dpn, dpo, rtol=1e-14, atol=0)
    out = ro.remap_np(dpo, dpn, fields)
    for f, g in zip(fields, out):
        assert np.allclose(g / dpn, f / dpo, rtol=1e-12, atol=1e-12 * np.abs(f / dpo).max())


@pytest.mark.parametrize("L", LEVELS)
def test_no_new_extrema_under_one_cell(L):
    dpo, dpn, fields, q = problem(40, L, "under", 400 + L)
    out = ro.remap_np(dpo, dpn, fields[:1])[0] / dpn
    lo, hi = q.min(1, keepdims=True), q.max(1, keepdims=True)
    tol = 1e-12 * np.abs(q).max(1, keepdims=True)
    assert np.all(out >= lo - tol) and np.all(out <= hi + tol)


@pytest.mark.parametrize("defect", ro.DEFECTS)
def test_defects_are_caught(defect):
    """Every defective numpy remap differs from the scalar transcription somewhere on the deformed inputs."""
    L, N = 26, 6
    dpo, dpn, fields, _ = problem(N, L, "under", 500)
    bad = ro.remap_np(dpo, dpn, fields, defect=defect)
    differs = False
    for c in range(N):
        want = ro.remap_column(list(dpo[c]), list(dpn[c]), [list(f[c]) for f in fields])
        differs |= any(not np.array_equal(bits(b[c]), bits(np.array(w))) for b, w in zip(bad, want))
    assert differs


def test_handle_arrays_only_the_selection_changes():
    """vertical_remap on handle-shaped arrays changes T, v, dp3d at tl and Qdp(qtl) of iq < qsize on [nets, nete) only,
    and equals remap_np on the same columns."""
    E, L, Qd, ntl, tl, qtl, qs, a, b = 5, 7, 3, 3, 2, 1, 2, 1, 4
    rng = np.random.default_rng(7)
    dp = rng.uniform(0.5, 2.0, (E, ntl, L, 4, 4)) * 1000.0
    A = dict(elem_state_dp3d=dp, elem_state_v=rng.uniform(-9, 9, (E, ntl, L, 4, 4, 2)),
             elem_state_T=rng.uniform(200, 300, (E, ntl, L, 4, 4)), elem_state_Qdp=rng.uniform(0, 1, (E, Qd, 2, L, 4, 4)))
    B = {n: x.copy() for n, x in A.items()}
    hyai, hybi = ro.coordinate(L)
    ro.vertical_remap(B, hyai, hybi, ro.PS0, a, b, tl, qtl, qs)
    changed = {n: ~np.equal(bits(A[n]), bits(B[n])) for n in A}
    assert not changed["elem_state_dp3d"][:a].any() and not changed["elem_state_dp3d"][b:].any()
    assert not changed["elem_state_dp3d"][:, [0, 1]].any() and changed["elem_state_dp3d"][a:b, tl].all()
    assert not changed["elem_state_Qdp"][:, qs:].any() and not changed["elem_state_Qdp"][:, :, 1 - qtl].any()
    assert not changed["elem_state_T"][:, :tl].any() and not changed["elem_state_v"][:a].any()
    col = lambda x: np.moveaxis(x.reshape(b - a, L, 16), 1, 2).reshape(-1, L)
    dpo = col(A["elem_state_dp3d"][a:b, tl])
    want = ro.remap_np(dpo, ro.target_dp(dpo, hyai, hybi, ro.PS0), [col(A["elem_state_Qdp"][a:b, 1, qtl])])[0]
    assert np.array_equal(bits(col(B["elem_state_Qdp"][a:b, 1, qtl])), bits(want))
