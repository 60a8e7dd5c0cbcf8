"""caar_dss_interior / caar_dss_boundary transcribed in tests/rk5_partition_oracle.py: on permuted cubed spheres
ne = 1..6 and random meshes with up to 8 copies per point, cut into 1, 2, 3, 5 and 8 uneven blocks (and a block that
shares no point), every local group is interior or boundary and never both, every copy pack sends lies in a boundary
group, and interior then boundary, or boundary then interior, equals dss_partition_oracle's unpack bit for bit without
writing the receive buffer. A split with a boundary group in the interior set, or a boundary pass that writes a remote
copy's slot, is caught."""
import numpy as np
import pytest

import dss_oracle as do
import dss_partition_oracle as dpo
import rk5_partition_oracle as rpo

NPARTS = (1, 2, 3, 5, 8)
MESHES = [f"cube{ne}p" for ne in range(1, 7)] + ["random8"]


def mesh(kind, rng):
    if kind.startswith("cube"):
        return do.cubed_sphere_gid(int(kind[4]), rng)
    gid = do.random_gid(40, rng, 8).reshape(40, 16)
    gid[-1] = (1 << 62) + np.arange(16)    # the last element shares no point: as the last block, no boundary group
    return gid.reshape(40, 4, 4)


def partitions(E, rng, isolated):
    out = [dpo.block_partition(E, n, rng) for n in NPARTS if n <= E]
    if isolated:
        out.append(np.array([0, 1, E - 1, E], dtype=np.int32))
    return out


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def values(E, rng):
    f = rng.integers(0x4000000000000000, 0x4100000000000000, size=(16 * E, 3), dtype=np.uint64).view(np.float64)
    return f, rng.uniform(0.5, 2.0, 16 * E)


@pytest.mark.parametrize("kind", MESHES)
def test_split_covers_the_groups_and_equals_unpack(kind):
    rng = np.random.default_rng(MESHES.index(kind))
    gid = mesh(kind, rng)
    E = gid.shape[0]
    f, s = values(E, rng)
    no_boundary = 0
    for ps in partitions(E, rng, kind == "random8"):
        for p in range(len(ps) - 1):
            pt = rpo.SplitPart(gid, ps, p)
            assert sorted(pt.interior + pt.boundary) == list(range(len(pt.groups)))
            assert not set(pt.interior) & set(pt.boundary)
            local = lambda c: pt.e0 <= c // 16 < pt.e1
            assert all(all(local(c) for c in pt.groups[i]) for i in pt.interior)
            assert all(any(not local(c) for c in pt.groups[i]) for i in pt.boundary)
            bcopies = {c for i in pt.boundary for c in pt.groups[i]}
            assert all(c in bcopies for seg in pt.send for c in seg)
            no_boundary += not pt.boundary
        for w in (do.ASSEMBLE, do.PROJECT):
            want = dpo.dss_partitioned(gid, ps, f, s, w)
            for order in ("interior_first", "boundary_first"):
                got, kept = rpo.dss_split(gid, ps, f, s, w, order)
                assert kept, (kind, list(ps), w, order)
                assert np.array_equal(bits(got), bits(want)), (kind, list(ps), w, order)
    assert no_boundary >= 1          # the one-block partition, and the isolated block of random8


def test_defective_splits_are_caught():
    rng = np.random.default_rng(17)
    for kind in ("cube3p", "random8"):
        gid = mesh(kind, rng)
        E = gid.shape[0]
        f, s = values(E, rng)
        ps = dpo.block_partition(E, 3, rng)
        for w in (do.ASSEMBLE, do.PROJECT):
            want = dpo.dss_partitioned(gid, ps, f, s, w)
            for order in ("interior_first", "boundary_first"):
                bad, kept = rpo.dss_split(gid, ps, f, s, w, order, defect="boundary_in_interior")
                assert kept and not np.array_equal(bits(bad), bits(want)), (kind, w, order)
                bad, kept = rpo.dss_split(gid, ps, f, s, w, order, defect="boundary_writes_remote")
                assert np.array_equal(bits(bad), bits(want)) and not kept, (kind, w, order)
