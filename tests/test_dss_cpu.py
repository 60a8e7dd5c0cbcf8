"""tests/dss_oracle.py on the CPU: the cubed-sphere generator has HOMME's point multiplicities and neighbour counts, its
permutation and orientation keep adjacency; the two transcriptions of the DSS and of neighbor_minmax agree bit for bit on
cubed and random meshes; the DSS output is continuous, conserves mass and leaves a continuous field where it was; and
four deliberately wrong variants are each caught by these checks."""
import numpy as np
import pytest

import dss_oracle as do


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def adjacency(gid):
    """set of frozensets of the element-block positions sharing each id -> the element graph as sorted pairs"""
    conn = do.Connectivity(gid)
    return {(e, n) for e, nb in enumerate(conn.neighbours) for n in nb}


# ---- the mesh generator ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("ne", range(1, 7))
def test_cubed_sphere_multiplicities(ne):
    """24 ne^2 interior points (1 copy), 24 ne^2 edge points (2), 6 ne^2 - 6 vertices shared by 4 and the 8 cube corners
    shared by 3; with ne >= 2 every element has 8 neighbours except the 24 at the cube's corners, which have 7."""
    for rng in (None, np.random.default_rng(ne)):
        conn = do.Connectivity(do.cubed_sphere_gid(ne, rng))
        counts = np.bincount(conn.mult, minlength=5)
        assert tuple(counts[1:]) == (24 * ne * ne, 24 * ne * ne, 8, 6 * ne * ne - 6)
        if ne >= 2:
            deg = np.array([len(x) for x in conn.neighbours])
            assert (deg == 7).sum() == 24 and (deg == 8).sum() == 6 * ne * ne - 24


@pytest.mark.parametrize("ne", [2, 3, 4])
def test_permutation_and_orientation_keep_adjacency(ne):
    """The permuted, rotated mesh is the plain one relabelled: the same element graph under the permutation, and within
    each element the same points shared with the same neighbours."""
    rng = np.random.default_rng(10 + ne)
    plain = do.cubed_sphere_gid(ne)
    perm = np.random.default_rng(10 + ne).permutation(plain.shape[0])
    mixed = do.cubed_sphere_gid(ne, rng)
    assert np.array_equal(np.sort(mixed.reshape(-1)), np.sort(plain.reshape(-1)))
    for e in range(plain.shape[0]):   # element e of the mixed mesh is plain element perm[e], its ids rearranged
        assert sorted(mixed[e].reshape(-1)) == sorted(plain[perm[e]].reshape(-1))
    a, b = adjacency(plain), adjacency(mixed)
    assert {(int(perm[e]), int(perm[n])) for e, n in b} == a


def test_random_mesh_has_what_spheres_lack():
    conn = do.Connectivity(do.random_gid(30, np.random.default_rng(1), 8))
    assert conn.M == 8 and (conn.mult > 4).any()
    assert conn.groups[0][:2] == [0, 5]              # two points of one element with one id


# ---- the two transcriptions -----------------------------------------------------------------------------------------

def meshes():
    rng = np.random.default_rng(2)
    return {"cube1": do.cubed_sphere_gid(1), "cube3": do.cubed_sphere_gid(3, rng), "random8": do.random_gid(25, rng, 8),
            "random3": do.random_gid(9, rng, 3)}


MESHES = meshes()


def inputs(conn, seed, X=6):
    rng = np.random.default_rng(seed)
    f = rng.standard_normal((conn.E * 16, X)) * 10.0 ** rng.uniform(-2, 2, (conn.E * 16, 1))
    s = rng.uniform(0.5, 2.0, conn.E * 16) * 10.0 ** rng.uniform(-3, 0, conn.E * 16)
    return f, s


def scalar_all(f, s, conn, w):
    return np.array([do.dss_scalar(f[:, j].tolist(), s.tolist(), conn, w) for j in range(f.shape[1])]).T


@pytest.mark.parametrize("w", [do.ASSEMBLE, do.PROJECT], ids=["assemble", "project"])
@pytest.mark.parametrize("name", list(MESHES))
def test_transcriptions_agree_and_dss_properties(name, w):
    conn = do.Connectivity(MESHES[name])
    f, s = inputs(conn, 3)
    a, b = do.dss_np(f, s, conn, w), scalar_all(f, s, conn, w)
    assert np.array_equal(bits(a), bits(b))
    check_continuous(a, conn)
    check_mass(f, a, s, w)


def check_continuous(out, conn):
    for c in range(1, conn.M):
        has = conn.mult > c
        assert np.array_equal(bits(out[conn.idx[has, c]]), bits(out[conn.idx[has, 0]])), c


def check_mass(f, out, s, w):
    """ASSEMBLE: sum spheremp * out = sum in; PROJECT: sum spheremp * out = sum spheremp * in; per column, ~1e-15"""
    got = (s[:, None] * out).sum(0)
    want = f.sum(0) if w == do.ASSEMBLE else (s[:, None] * f).sum(0)
    scale = np.abs(f).sum(0) if w == do.ASSEMBLE else (s[:, None] * np.abs(f)).sum(0)
    assert np.all(np.abs(got - want) <= 4e-15 * scale), np.max(np.abs(got - want) / scale)


@pytest.mark.parametrize("name", ["cube3", "random8"])
def test_project_keeps_a_continuous_field(name):
    """PROJECT of a continuous field returns it up to rounding: n products, n - 1 adds, the n - 1 adds of m, 1/m and the
    last product give at most (2n + 1) u relative for a point of n copies (u = 2^-53), with weights of one magnitude.
    Most points come back within 2 ulp."""
    conn = do.Connectivity(MESHES[name])
    f, _ = inputs(conn, 4)
    s = np.random.default_rng(4).uniform(0.5, 2.0, conn.E * 16)
    cont = do.dss_np(f, s, conn, do.ASSEMBLE)           # any continuous field
    out = do.dss_np(cont, s, conn, do.PROJECT)
    n = np.empty(conn.E * 16)
    for c in range(conn.M):
        n[conn.idx[conn.mult > c, c]] = conn.mult[conn.mult > c]
    assert np.all(np.abs(out - cont) <= (2 * n[:, None] + 1) * 2.0 ** -53 * np.abs(cont))
    assert np.mean(np.abs(out - cont) <= 2 * np.spacing(np.abs(cont))) > 0.99


def test_dss_arrays_slices_like_the_handle():
    """dss_arrays touches exactly the selected slice (dp3d at tl, v components separately, Qdp(qtl) of iq < qsize)."""
    gid = MESHES["cube3"]
    conn = do.Connectivity(gid)
    E, L, Qd = conn.E, 3, 3
    rng = np.random.default_rng(5)
    A = {"elem_spheremp": rng.uniform(0.5, 2, (E, 4, 4)), "elem_state_v": rng.standard_normal((E, 3, L, 4, 4, 2)),
         "elem_state_Qdp": rng.standard_normal((E, Qd, 2, L, 4, 4))}
    B = {k: v.copy() for k, v in A.items()}
    do.dss_arrays(B, conn, ("elem_state_v", "elem_state_Qdp"), tl=2, qtl=1, qsize=2, weighting=do.PROJECT)
    s = A["elem_spheremp"].reshape(-1)
    for c in range(2):
        for k in range(L):
            want = do.dss_scalar(A["elem_state_v"][:, 2, k, :, :, c].reshape(-1).tolist(), s.tolist(), conn, do.PROJECT)
            assert np.array_equal(bits(B["elem_state_v"][:, 2, k, :, :, c].reshape(-1)), bits(np.array(want)))
    for iq in range(2):
        for k in range(L):
            want = do.dss_scalar(A["elem_state_Qdp"][:, iq, 1, k].reshape(-1).tolist(), s.tolist(), conn, do.PROJECT)
            assert np.array_equal(bits(B["elem_state_Qdp"][:, iq, 1, k].reshape(-1)), bits(np.array(want)))
    assert np.array_equal(bits(B["elem_state_v"][:, :2]), bits(A["elem_state_v"][:, :2]))
    assert np.array_equal(bits(B["elem_state_Qdp"][:, 2]), bits(A["elem_state_Qdp"][:, 2]))
    assert np.array_equal(bits(B["elem_state_Qdp"][:, :, 0]), bits(A["elem_state_Qdp"][:, :, 0]))


@pytest.mark.parametrize("name", list(MESHES))
def test_neighbor_minmax_transcriptions_agree(name):
    conn = do.Connectivity(MESHES[name])
    rng = np.random.default_rng(6)
    b = np.sort(rng.standard_normal((conn.E, 3, 5, 2)), -1)
    a, c = do.neighbor_minmax_np(b, conn, 2), do.neighbor_minmax_scalar(b, conn, 2)
    assert np.array_equal(bits(a), bits(c))
    assert np.array_equal(bits(a[:, 2]), bits(b[:, 2]))
    check_neighbour_bounds(MESHES[name], b, a, 2)


def check_neighbour_bounds(gid, b, out, qsize):
    """Brute force from the ids: every element's bounds are the min / max over itself and every element it shares an id
    with."""
    g = gid.reshape(gid.shape[0], 16)
    for e in range(g.shape[0]):
        near = [n for n in range(g.shape[0]) if np.intersect1d(g[e], g[n]).size] or [e]
        assert np.array_equal(out[e, :qsize, :, 0], b[near, :qsize, :, 0].min(0))
        assert np.array_equal(out[e, :qsize, :, 1], b[near, :qsize, :, 1].max(0))


# ---- the defective variants are caught ----------------------------------------------------------------------------------

@pytest.mark.parametrize("defect", do.DEFECTS)
def test_defective_dss_is_caught(defect):
    """Each wrong DSS fails at least one of: agreement with the scalar transcription, continuity, mass."""
    caught = False
    for name in ("cube3", "random8"):
        conn = do.Connectivity(MESHES[name])
        f, s = inputs(conn, 7, X=2)
        for w in (do.ASSEMBLE, do.PROJECT):
            bad = do.dss_np(f, s, conn, w, defect)
            checks = [lambda: np.testing.assert_array_equal(bits(bad), bits(scalar_all(f, s, conn, w))),
                      lambda: check_continuous(bad, conn), lambda: check_mass(f, bad, s, w)]
            for chk in checks:
                try:
                    chk()
                except AssertionError:
                    caught = True
    assert caught, defect


def test_neighbour_set_without_vertex_neighbours_is_caught():
    gid = do.cubed_sphere_gid(3)
    bad = do.Connectivity(gid, defect="edges_only")
    deg = np.array([len(x) for x in bad.neighbours])
    assert not ((deg == 7).sum() == 24 and (deg == 8).sum() == 6 * 9 - 24)
    b = np.sort(np.random.default_rng(8).standard_normal((gid.shape[0], 1, 4, 2)), -1)
    with pytest.raises(AssertionError):
        check_neighbour_bounds(gid, b, do.neighbor_minmax_np(b, bad, 1), 1)
