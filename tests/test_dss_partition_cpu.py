"""The partitioned DSS and neighbor_minmax of tests/dss_partition_oracle.py (pack, segment moves, unpack in numpy) equal,
bit for bit, dss_oracle's whole-mesh transcriptions: exact cubed spheres ne = 1..6, plain and permuted, and random meshes
with up to 8 copies per point, cut into 1, 2, 3 and 7 blocks, with blocks of one element, a block that shares no point
and points whose copies lie in 3 or 4 parts. A variant that sums the received copies after the local ones is caught."""
import numpy as np
import pytest

import dss_oracle as do
import dss_partition_oracle as dpo

NPARTS = (1, 2, 3, 7)


def mesh(kind, rng):
    if kind.startswith("cube"):
        ne, permuted = int(kind[4]), kind.endswith("p")
        return do.cubed_sphere_gid(ne, rng if permuted else None)
    gid = do.random_gid(40, rng, 8).reshape(40, 16)
    gid[-1] = (1 << 62) + np.arange(16)    # the last element shares no point: as the last block, neither does its part
    return gid.reshape(40, 4, 4)


MESHES = [f"cube{ne}{p}" for ne in range(1, 7) for p in ("", "p")] + ["random8"]


def partitions(E, rng, gid):
    out = []
    for n in NPARTS:
        if n > E:
            continue
        out.append(dpo.block_partition(E, n, rng))
    if gid is not None and E >= 3:   # the last element alone as the last block
        out.append(np.array([0, 1, E - 1, E], dtype=np.int32))
    return out


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def points_values(E, rng, X=3):
    f = rng.integers(0x4000000000000000, 0x4100000000000000, size=(16 * E, X), dtype=np.uint64).view(np.float64)
    s = rng.uniform(0.5, 2.0, 16 * E)
    return f, s


@pytest.mark.parametrize("kind", MESHES)
def test_partitioned_dss_equals_whole_mesh(kind):
    rng = np.random.default_rng(MESHES.index(kind))
    gid = mesh(kind, rng)
    E = gid.shape[0]
    conn = do.Connectivity(gid)
    f, s = points_values(E, rng)
    for ps in partitions(E, rng, gid if kind == "random8" else None):
        for w in (do.ASSEMBLE, do.PROJECT):
            want = do.dss_np(f, s, conn, w)
            got = dpo.dss_partitioned(gid, ps, f, s, w)
            assert np.array_equal(bits(got), bits(want)), (kind, list(ps), w)


@pytest.mark.parametrize("kind", ["cube2", "cube3p", "random8"])
def test_partitioned_neighbor_minmax_equals_whole_mesh(kind):
    rng = np.random.default_rng(100 + MESHES.index(kind))
    gid = mesh(kind, rng)
    E, Qd, L = gid.shape[0], 3, 5
    conn = do.Connectivity(gid)
    b = np.sort(rng.standard_normal((E, Qd, L, 2)), -1)
    b[rng.random(b.shape) < 0.2] = 0.0
    b[rng.random(b.shape) < 0.5] *= -1.0                # -0.0 and +0.0 side by side: the order decides which survives
    b = np.sort(b, -1)
    for ps in partitions(E, rng, gid if kind == "random8" else None):
        for qs in (0, 2, Qd):
            want = do.neighbor_minmax_np(b, conn, qs)
            got = dpo.neighbor_minmax_partitioned(gid, ps, b, qs)
            assert np.array_equal(bits(got), bits(want)), (kind, list(ps), qs)


def spread(gid, ps):
    """the number of parts that hold a copy of each point"""
    part_of = np.searchsorted(ps, np.arange(ps[-1]), side="right") - 1
    out = {}
    for c, g in enumerate(np.asarray(gid).reshape(-1)):
        out.setdefault(int(g), set()).add(int(part_of[c // 16]))
    return {g: len(v) for g, v in out.items()}


def test_points_in_3_and_4_parts_and_segment_sizes():
    """A cube corner with its three elements in three one-element blocks, and a point of a random mesh in four parts:
    bit for bit with the whole-mesh DSS and neighbor_minmax; the segment sizes agree pairwise; the isolated last
    element sends and receives nothing."""
    rng = np.random.default_rng(5)
    cube = do.cubed_sphere_gid(2)                  # element 0 of faces x=0, y=0, z=0 (elements 0, 8, 16) share (0,0,0)
    ps3 = np.array([0, 1, 8, 9, 16, 17, 24], dtype=np.int32)
    assert spread(cube, ps3)[int(cube[0, 0, 0])] == 3
    rnd = mesh("random8", np.random.default_rng(1))
    conn = do.Connectivity(rnd)
    g = next(g for g in conn.groups if len({c // 16 for c in g}) >= 4)
    els = sorted({c // 16 for c in g})[:4]
    ps4 = np.array(sorted({0, els[1], els[2], els[3], 39, 40}), dtype=np.int32)
    assert spread(rnd, ps4)[int(rnd.reshape(-1)[g[0]])] >= 4
    for gid, ps in ((cube, ps3), (rnd, ps4)):
        E = gid.shape[0]
        f, s = points_values(E, rng)
        b = np.sort(rng.standard_normal((E, 2, 3, 2)), -1)
        c = do.Connectivity(gid)
        for w in (do.ASSEMBLE, do.PROJECT):
            assert np.array_equal(bits(dpo.dss_partitioned(gid, ps, f, s, w)), bits(do.dss_np(f, s, c, w)))
        assert np.array_equal(bits(dpo.neighbor_minmax_partitioned(gid, ps, b, 2)), bits(do.neighbor_minmax_np(b, c, 2)))
        parts = [dpo.Part(gid, ps, p) for p in range(len(ps) - 1)]
        for p in parts:
            for q in parts:
                assert len(p.send[q.part]) == len(q.recv[p.part])
                assert len(p.send_el[q.part]) == len(q.recv_el[p.part])
    assert not any(parts[-1].send) and not any(parts[-1].recv) and not any(parts[-1].send_el)


def test_remote_after_local_defect_is_caught():
    rng = np.random.default_rng(11)
    caught = 0
    for kind in ("cube3p", "random8"):
        gid = mesh(kind, rng)
        E = gid.shape[0]
        f, s = points_values(E, rng)
        ps = dpo.block_partition(E, 3, rng)
        for w in (do.ASSEMBLE, do.PROJECT):
            want = do.dss_np(f, s, do.Connectivity(gid), w)
            bad = dpo.dss_partitioned(gid, ps, f, s, w, defect="remote_after_local")
            caught += not np.array_equal(bits(bad), bits(want))
    assert caught == 4
