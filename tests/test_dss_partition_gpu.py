"""caar_set_partition, caar_dss_pack / caar_dss_unpack, caar_neighbor_minmax_pack / caar_neighbor_minmax_unpack and
caar_halo_segments on the GPU: N handles on one device hold the blocks of a mesh, and torch copies move the segments
between them. The assembled fields of every handle equal, bit for bit, one whole-mesh handle's caar_dss and the oracle,
at nlev 72, 30, 128 and at 2, 3, 5, 7, 26, 80, 127 and 131, with every value outside the selection unchanged and both
exchange buffers NaN wherever the current call does not write them (the whole send buffer before every pack, the whole
receive buffer outside the moved segments); ne = 60 in 4
parts and ne = 120 in 8 parts; neighbor_minmax with -0.0 / +0.0; the limited tracer step run partitioned; nparts == 1;
argument errors, launch counts and pairwise segment sizes."""
import ctypes as C

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
import dss_oracle as do
import dss_partition_oracle as dpo
from oracle import harness
from test_pointwise_cpu import level_local_inputs

pytestmark = pytest.mark.gpu
INVALID, UNSUPPORTED, STATE_ERR = 1, 4, 5
F = {n: tb.capi.FIELD_BIT[n] for n in tb.DSS_FIELDS}
ALL4 = tuple(tb.DSS_FIELDS)
SEL_NAMES = ("elem_spheremp",) + ALL4
STATE_NAMES = ("elem_state_dp3d", "elem_state_v", "elem_state_T")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def random_fields(E, L, Qd, ntl, seed):
    rng = np.random.default_rng(seed)
    out = {"elem_spheremp": rng.uniform(0.5, 2.0, (E, 4, 4))}
    for n in ALL4:
        shape = tb.field_shape(n, E, L, Qd, ntl)
        out[n] = rng.integers(0x4000000000000000, 0x4100000000000000, size=shape, dtype=np.uint64).view(np.float64)
    return out


def part_handles(gid, ps, L, Qd, ntl, arrays, names=SEL_NAMES):
    hs = []
    for p in range(len(ps) - 1):
        h = tb.Caar(int(ps[p + 1] - ps[p]), L, Qd, ntl)
        h.upload({n: np.ascontiguousarray(arrays[n][ps[p]:ps[p + 1]]) for n in names}, names=names)
        h.set_partition(gid, ps, p)
        hs.append(h)
    return hs


def upload_parts(hs, ps, arrays, names):
    for p, h in enumerate(hs):
        h.upload({n: np.ascontiguousarray(arrays[n][ps[p]:ps[p + 1]]) for n in names}, names=names)


def download_parts(hs, ps, E, L, Qd, ntl, names):
    out = {n: np.empty(tb.field_shape(n, E, L, Qd, ntl)) for n in names}
    for p, h in enumerate(hs):
        part = {n: np.empty(tb.field_shape(n, int(ps[p + 1] - ps[p]), L, Qd, ntl)) for n in names}
        h.download(part, names=names)
        for n in names:
            out[n][ps[p]:ps[p + 1]] = part[n]
    return out


def whole_buffers(h):
    """(send, recv): views of the whole of a handle's two exchange buffers, which are sized for the largest selection of
    either exchange"""
    Qd = h.shape_args[2]
    segs = [h.halo_segments(op, names, Qd) for op, names in ((tb.HALO_DSS, ALL4), (tb.HALO_MINMAX, ()))]
    return tuple(max((s[i] for s in segs), key=lambda t: t.numel()) for i in (0, 1))


def nan_fill(hs, which):
    """a NaN bit pattern over the whole send (0) or receive (1) buffer of every handle: a record a pack leaves
    unwritten, or a read outside the current selection's segments, is then a NaN in a compared value, not a stale
    record of an earlier call"""
    import torch
    for h in hs:
        whole_buffers(h)[which].view(torch.int64).fill_(0x7FF8DEADBEEF0001)
    torch.cuda.synchronize()       # the handles run on streams of their own


def move_segments(hs, op, names, qsize):
    """segment p->q of part p's send buffer to segment p of part q's receive buffer, each whole receive buffer NaN
    first; checks that the segment sizes agree pairwise"""
    import torch
    segs = [h.halo_segments(op, names, qsize) for h in hs]
    nan_fill(hs, 1)
    for q, (_, recv, _, ro) in enumerate(segs):
        for p, (send, _, so_, _) in enumerate(segs):
            assert so_[q + 1] - so_[q] == ro[p + 1] - ro[p], (p, q)
            if p == q:
                assert so_[q + 1] == so_[q]
            elif ro[p + 1] > ro[p]:
                recv[ro[p]:ro[p + 1]].copy_(send[so_[q]:so_[q + 1]])
    torch.cuda.synchronize()


def exchange_dss(hs, names, tl=0, qtl=0, qsize=0, weighting=tb.DSS_ASSEMBLE):
    nan_fill(hs, 0)
    for h in hs:
        h.dss_pack(names, tl=tl, qtl=qtl, qsize=qsize, weighting=weighting)
    move_segments(hs, tb.HALO_DSS, names, qsize)
    for h in hs:
        h.dss_unpack(names, tl=tl, qtl=qtl, qsize=qsize, weighting=weighting)


def exchange_minmax(hs, qsize):
    nan_fill(hs, 0)
    for h in hs:
        h.neighbor_minmax_pack(qsize)
    move_segments(hs, tb.HALO_MINMAX, (), qsize)
    for h in hs:
        h.neighbor_minmax_unpack(qsize)


def isolated_random(rng):
    gid = do.random_gid(40, rng, 8).reshape(40, 16)
    gid[-1] = (1 << 62) + np.arange(16)          # a last block of one element that shares no point
    return gid.reshape(40, 4, 4)


MESHES = {
    "cube2": lambda rng: do.cubed_sphere_gid(2, rng),
    "cube3": lambda rng: do.cubed_sphere_gid(3, rng),
    "cube5": lambda rng: do.cubed_sphere_gid(5, rng),
    "random8": isolated_random,
}
# mesh, nlev, partition: a number of random blocks (the first of one element), or part_start itself. After nlev 72, 30
# and 128, the tails of the level batches: L % 4 = 0, 1, 2, 3 and L < 4 (dss_slice, dss_pack_kernel and
# dss_boundary_kernel's last batch), on groups of up to 4 copies (cube*) and more (random8), with one-element parts
CASES = [("cube2", 72, 3), ("cube2", 30, [0, 1, 8, 9, 16, 17, 24]), ("cube3", 30, 7), ("cube5", 128, 2),
         ("random8", 72, [0, 1, 39, 40]), ("random8", 30, 3), ("cube3", 72, 1),
         ("cube2", 2, 3), ("random8", 3, [0, 1, 39, 40]), ("cube3", 5, 7), ("cube2", 7, [0, 1, 8, 9, 16, 17, 24]),
         ("random8", 7, 3), ("random8", 26, 4), ("cube3", 80, 4), ("cube5", 127, 3), ("random8", 131, [0, 1, 39, 40]),
         ("cube2", 131, 2)]
SELECTIONS = [(n,) for n in ALL4] + [ALL4]


@pytest.mark.parametrize("mesh,L,parts", CASES, ids=[f"{m}-L{L}-{p if isinstance(p, int) else len(p) - 1}"
                                                      for m, L, p in CASES])
def test_partitioned_dss_equals_whole_mesh(mesh, L, parts):
    """Every selection with both weightings, tl and qtl cycling, qsize < qsize_d: the concatenated parts equal the
    whole-mesh caar_dss and the oracle in every bit of every field; the fields outside the selection are unchanged."""
    idx = CASES.index((mesh, L, parts))
    rng = np.random.default_rng(idx)
    gid = MESHES[mesh](rng)
    E, Qd, ntl = gid.shape[0], 4, 3
    ps = np.array(parts, dtype=np.int32) if not isinstance(parts, int) else dpo.block_partition(E, parts, rng)
    conn = do.Connectivity(gid)
    inp = random_fields(E, L, Qd, ntl, 13 * L + idx)
    whole = tb.Caar(E, L, Qd, ntl)
    whole.upload(inp, names=SEL_NAMES)
    whole.set_connectivity(gid)
    hs = part_handles(gid, ps, L, Qd, ntl, inp)
    i = 0
    for names in SELECTIONS:
        for w in (do.ASSEMBLE, do.PROJECT):
            tl, qtl, qs = i % ntl, (i // 3) % 2, 3 if i % 2 else 1
            i += 1
            whole.upload(inp, names=ALL4)
            upload_parts(hs, ps, inp, ALL4)
            whole.dss(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
            exchange_dss(hs, names, tl, qtl, qs, w)
            got = download_parts(hs, ps, E, L, Qd, ntl, ALL4)
            ref = {n: np.empty(tb.field_shape(n, E, L, Qd, ntl)) for n in ALL4}
            whole.download(ref, names=ALL4)
            want = {n: inp[n].copy() for n in SEL_NAMES}
            do.dss_arrays(want, conn, names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
            for n in ALL4:
                assert np.array_equal(bits(got[n]), bits(ref[n])), (names, w, n)
                assert np.array_equal(bits(got[n]), bits(want[n])), (names, w, n)
    for h in hs + [whole]:
        h.close()


@pytest.mark.parametrize("ne,nparts", [(60, 4), (120, 8)])
def test_large_meshes(ne, nparts):
    """ne = 60 in 4 parts (each part's walk wraps) and ne = 120 in 8: dp3d, v and T assembled at once, bit for bit with
    one whole-mesh handle; at ne = 60 also Qdp with PROJECT."""
    gid = do.cubed_sphere_gid(ne, np.random.default_rng(ne) if ne == 60 else None)
    E, L, Qd, ntl = gid.shape[0], 72, 2, 1
    ps = np.array([(E * p) // nparts for p in range(nparts + 1)], dtype=np.int32)
    rng = np.random.default_rng(ne)
    inp = {"elem_spheremp": rng.uniform(0.5, 2.0, (E, 4, 4))}
    names = STATE_NAMES + (("elem_state_Qdp",) if ne == 60 else ())
    for n in names:
        inp[n] = rng.uniform(1.0, 3.0, tb.field_shape(n, E, L, Qd, ntl))
    sel = ("elem_spheremp",) + names
    whole = tb.Caar(E, L, Qd, ntl)
    whole.upload(inp, names=sel)
    whole.set_connectivity(gid)
    hs = part_handles(gid, ps, L, Qd, ntl, inp, sel)
    runs = [(STATE_NAMES, 0, do.ASSEMBLE)] + ([(("elem_state_Qdp",), 2, do.PROJECT)] if ne == 60 else [])
    for sel_names, qs, w in runs:
        whole.dss(sel_names, tl=0, qtl=1, qsize=qs, weighting=w)
        exchange_dss(hs, sel_names, 0, 1, qs, w)
    ref = {n: np.empty(tb.field_shape(n, E, L, Qd, ntl)) for n in names}
    whole.download(ref, names=names)
    got = download_parts(hs, ps, E, L, Qd, ntl, names)
    for n in names:
        assert np.array_equal(bits(got[n]), bits(ref[n])), n
        assert not np.array_equal(bits(got[n]), bits(inp[n])), n
    for h in hs + [whole]:
        h.close()


MINMAX_CASES = [("cube3", 7, 30), ("random8", [0, 1, 39, 40], 30), ("cube2", 1, 30), ("cube3", 7, 3),
                ("random8", [0, 1, 39, 40], 5), ("cube2", 3, 80), ("random8", 3, 127), ("cube5", 4, 131)]


@pytest.mark.parametrize("mesh,parts,L", MINMAX_CASES,
                         ids=[f"{m}-{p if isinstance(p, int) else 'parts1'}" + ("" if L == 30 else f"-L{L}")
                              for m, p, L in MINMAX_CASES])
def test_partitioned_neighbor_minmax(mesh, parts, L):
    """Random bounds with -0.0 and +0.0 side by side, qsize 3 of 4 then 1: the parts equal the whole-mesh
    caar_neighbor_minmax and the oracle bit for bit; tracer 3 untouched."""
    rng = np.random.default_rng(21)
    gid = MESHES[mesh](rng)
    E, Qd = gid.shape[0], 4
    ps = np.array(parts, dtype=np.int32) if not isinstance(parts, int) else dpo.block_partition(E, parts, rng)
    conn = do.Connectivity(gid)
    b = np.sort(rng.standard_normal((E, Qd, L, 2)), -1)
    b[rng.random(b.shape) < 0.3] = 0.0
    b[rng.random(b.shape) < 0.5] *= -1.0
    b = np.ascontiguousarray(np.sort(b, -1))
    whole = tb.Caar(E, L, Qd)
    whole.set_connectivity(gid)
    whole.upload_bounds(b)
    hs = []
    for p in range(len(ps) - 1):
        h = tb.Caar(int(ps[p + 1] - ps[p]), L, Qd)
        h.set_partition(gid, ps, p)
        h.upload_bounds(np.ascontiguousarray(b[ps[p]:ps[p + 1]]))
        hs.append(h)
    want = b
    for qs in (3, 1):
        whole.neighbor_minmax(qs)
        exchange_minmax(hs, qs)
        want = do.neighbor_minmax_np(want, conn, qs)
        got = np.concatenate([h.download_bounds() for h in hs])
        assert np.array_equal(bits(got), bits(whole.download_bounds())), qs
        assert np.array_equal(bits(got), bits(want)), qs
    assert np.array_equal(bits(got[:, 3]), bits(b[:, 3]))
    for h in hs + [whole]:
        h.close()


QNAMES = ("elem_Dinv", "elem_metdet", "elem_rmetdet", "elem_spheremp", "elem_state_dp3d", "elem_state_Qdp")


def test_limited_tracer_step_partitioned():
    """bounds -> exchanged neighbor_minmax -> strict caar_advect_tracers -> limiter -> exchanged caar_dss(Qdp, PROJECT)
    on a permuted ne = 2 sphere in 3 parts equals the same step on one handle, bit for bit, bounds included."""
    gid = do.cubed_sphere_gid(2, np.random.default_rng(2))
    E, L, Qd, qs, dtl, DT = gid.shape[0], 30, 3, 2, 1, 150.0
    ps = np.array([0, 1, 13, 24], dtype=np.int32)
    s, vstar, _, _ = level_local_inputs("randomize", E, L, 6400, qsize_d=Qd)

    def handle(e0, e1):
        h = tb.Caar(e1 - e0, L, Qd, s.ntl)
        h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
        h.upload({n: np.ascontiguousarray(s.arrays[n][e0:e1]) for n in QNAMES}, names=QNAMES)
        h.upload_vstar(np.ascontiguousarray(vstar[e0:e1]))
        return h
    whole = handle(0, E)
    whole.set_connectivity(gid)
    whole.tracer_bounds(0, qs, dtl)
    whole.neighbor_minmax(qs)
    q = whole.advect_tracers(0, qs, DT, 1, tb.MODE_STRICT)
    whole.limit_tracers(q, qs, dtl)
    whole.dss(("elem_state_Qdp",), qtl=q, qsize=qs, weighting=tb.DSS_PROJECT)
    hs = []
    for p in range(3):
        h = handle(int(ps[p]), int(ps[p + 1]))
        h.set_partition(gid, ps, p)
        h.tracer_bounds(0, qs, dtl)
        hs.append(h)
    exchange_minmax(hs, qs)
    for h in hs:
        assert h.advect_tracers(0, qs, DT, 1, tb.MODE_STRICT) == q
        h.limit_tracers(q, qs, dtl)
    exchange_dss(hs, ("elem_state_Qdp",), qtl=q, qsize=qs, weighting=tb.DSS_PROJECT)
    want = {"elem_state_Qdp": np.empty_like(s.arrays["elem_state_Qdp"])}
    whole.download(want, names=("elem_state_Qdp",))
    got = download_parts(hs, ps, E, L, Qd, s.ntl, ("elem_state_Qdp",))
    assert np.array_equal(bits(got["elem_state_Qdp"]), bits(want["elem_state_Qdp"]))
    assert np.array_equal(bits(np.concatenate([h.download_bounds() for h in hs])), bits(whole.download_bounds()))
    assert not np.array_equal(bits(want["elem_state_Qdp"]), bits(s.arrays["elem_state_Qdp"]))
    for h in hs + [whole]:
        h.close()


def test_one_part_and_local_meaning_kept():
    """nparts == 1: caar_dss_unpack equals caar_dss bit for bit, with no segment at all. After caar_set_partition,
    caar_dss and caar_neighbor_minmax on a part equal caar_set_connectivity on the part's slice of the map."""
    rng = np.random.default_rng(31)
    gid = do.cubed_sphere_gid(3, rng)
    E, L, Qd, ntl = gid.shape[0], 30, 2, 2
    inp = random_fields(E, L, Qd, ntl, 31)
    one = part_handles(gid, [0, E], L, Qd, ntl, inp)[0]
    ref = tb.Caar(E, L, Qd, ntl)
    ref.upload(inp, names=SEL_NAMES)
    ref.set_connectivity(gid)
    send, recv, so_, ro = one.halo_segments(tb.HALO_DSS, ALL4, 2)
    assert list(so_) == [0, 0] and list(ro) == [0, 0]
    for w in (do.ASSEMBLE, do.PROJECT):
        k = one.launch_count()
        one.dss_pack(ALL4, tl=1, qtl=1, qsize=2, weighting=w)
        assert one.launch_count() == k                 # a part that shares no point packs nothing
        one.dss_unpack(ALL4, tl=1, qtl=1, qsize=2, weighting=w)
        assert one.launch_count() == k + 1
        ref.dss(ALL4, tl=1, qtl=1, qsize=2, weighting=w)
        a = {n: np.empty(tb.field_shape(n, E, L, Qd, ntl)) for n in ALL4}
        one.download(a, names=ALL4)
        b = {n: np.empty_like(a[n]) for n in ALL4}
        ref.download(b, names=ALL4)
        for n in ALL4:
            assert np.array_equal(bits(a[n]), bits(b[n])), (w, n)
    ps = np.array([0, 20, E], dtype=np.int32)
    part = tb.Caar(int(ps[2] - ps[1]), L, Qd, ntl)
    sl = tb.Caar(int(ps[2] - ps[1]), L, Qd, ntl)
    bnd = np.ascontiguousarray(np.sort(rng.standard_normal((int(ps[2] - ps[1]), Qd, L, 2)), -1))
    for h in (part, sl):
        h.upload({n: np.ascontiguousarray(inp[n][20:]) for n in SEL_NAMES}, names=SEL_NAMES)
        h.upload_bounds(bnd)
    part.set_partition(gid, ps, 1)
    sl.set_connectivity(gid[20:])
    for h in (part, sl):
        h.dss(ALL4, tl=0, qtl=0, qsize=2, weighting=tb.DSS_PROJECT)
        h.neighbor_minmax(2)
    a = {n: np.empty(tb.field_shape(n, E - 20, L, Qd, ntl)) for n in ALL4}
    b = {n: np.empty_like(a[n]) for n in ALL4}
    part.download(a, names=ALL4)
    sl.download(b, names=ALL4)
    for n in ALL4:
        assert np.array_equal(bits(a[n]), bits(b[n])), n
    assert np.array_equal(bits(part.download_bounds()), bits(sl.download_bounds()))
    # a later caar_set_connectivity replaces the partition
    part.set_connectivity(gid[20:])
    assert tb.load_library().caar_dss_pack(part.h, F["elem_state_T"], 0, 0, 0, 0) == STATE_ERR
    for h in (one, ref, part, sl):
        h.close()


def test_segments_are_the_selection():
    """Segment sizes: DSS records of 1 + (fields' values per level) * L doubles, bounds rows of qsize * L * 2; equal
    pairwise across parts; the receive segments of a part sum to the records it reads. At nlev 16 with qsize_d 3, and at
    nlev 127 with qsize_d 35, where the record of every field and tracer (1 + 39 * 127 doubles) is odd and the largest
    the buffers are sized for."""
    rng = np.random.default_rng(41)
    gid = do.cubed_sphere_gid(2, rng)
    ps = np.array([0, 5, 11, 24], dtype=np.int32)
    parts = [dpo.Part(gid, ps, p) for p in range(3)]
    for L, Qd in ((16, 3), (127, 35)):
        hs = []
        for p in range(3):
            h = tb.Caar(int(ps[p + 1] - ps[p]), L, Qd, 2)
            h.set_partition(gid, ps, p)
            hs.append(h)
        for names, qs, per in ((("elem_state_T",), 0, 1), (("elem_state_v",), 0, 2), (ALL4, 2, 6), (ALL4, 3, 7),
                               (("elem_state_Qdp",), 0, 0), (ALL4, Qd, 4 + Qd)):
            for h, pt in zip(hs, parts):
                _, _, so_, ro = h.halo_segments(tb.HALO_DSS, names, qs)
                nv = 1 + per * L if per else 0
                assert list(np.diff(so_)) == [len(x) * nv for x in pt.send], (L, names, qs)
                assert list(np.diff(ro)) == [len(x) * nv for x in pt.recv], (L, names, qs)
        for qs in (1, 3, Qd):
            for h, pt in zip(hs, parts):
                _, _, so_, ro = h.halo_segments(tb.HALO_MINMAX, (), qs)
                assert list(np.diff(so_)) == [len(x) * qs * L * 2 for x in pt.send_el], (L, qs)
                assert list(np.diff(ro)) == [len(x) * qs * L * 2 for x in pt.recv_el], (L, qs)
        for h, pt in zip(hs, parts):      # what nan_fill covers: the largest selection of either exchange
            nv, row = 1 + (4 + Qd) * L, Qd * L * 2
            send, recv = whole_buffers(h)
            assert send.numel() == max(sum(map(len, pt.send)) * nv, sum(map(len, pt.send_el)) * row), L
            assert recv.numel() == max(sum(map(len, pt.recv)) * nv, sum(map(len, pt.recv_el)) * row), L
        for h in hs:
            h.close()


# ---- argument errors and launch counts ------------------------------------------------------------------------------

E_, L_, Q_, NTL_ = 24, 16, 2, 3
PS_ = (0, 10, 24)
GOOD_DSS = dict(mask=F["elem_state_T"] | F["elem_state_Qdp"], tl=0, qtl=0, qsize=2, weighting=0)
DSS_BAD = ([dict(mask=tb.capi.FIELD_BIT["elem_spheremp"]), dict(mask=1 << 16), dict(tl=-1), dict(tl=NTL_),
            dict(qtl=-1), dict(qtl=2), dict(qsize=-1), dict(qsize=Q_ + 1), dict(weighting=2), dict(weighting=-1)])
PART_BAD = [("null gid", dict(gid=None), INVALID), ("null part_start", dict(ps=None), INVALID),
            ("nparts 0", dict(nparts=0), INVALID), ("part -1", dict(part=-1), INVALID),
            ("part 2", dict(part=2), INVALID), ("start 1", dict(ps=(1, 10, 24)), INVALID),
            ("end 23", dict(ps=(0, 10, 23), nglob=23), INVALID), ("end != nelem_global", dict(ps=(0, 10, 25)), INVALID),
            ("not ascending", dict(ps=(0, 10, 10, 24), nparts=3, part=2), INVALID),
            ("block size", dict(ps=(0, 9, 24)), INVALID), ("layout 2", dict(layout=2), INVALID),
            ("2^27 elements", dict(nglob=1 << 27, ps=(0, 10, 1 << 27)), UNSUPPORTED)]
ENTRIES = ("caar_dss_pack", "caar_dss_unpack")
ERR_CASES = (
    [(ep, "null handle", None, {}, INVALID) for ep in ENTRIES + ("caar_neighbor_minmax_pack",
                                                               "caar_neighbor_minmax_unpack", "caar_halo_segments",
                                                               "caar_set_partition")]
    + [(ep, "not partitioned", k, {}, STATE_ERR) for ep in ENTRIES + ("caar_neighbor_minmax_pack",
                                                                       "caar_neighbor_minmax_unpack",
                                                                       "caar_halo_segments")
       for k in ("bare", "connected")]
    + [(ep, f"{k}={v}", "ready", {k: v}, INVALID) for ep in ENTRIES for o in DSS_BAD for k, v in o.items()]
    + [(ep, f"qsize={q}", "ready", dict(qsize=q), INVALID) for ep in ("caar_neighbor_minmax_pack",
                                                                      "caar_neighbor_minmax_unpack") for q in (-1, Q_ + 1)]
    + [("caar_halo_segments", c, "ready", o, INVALID) for c, o in
       (("op 2", dict(op=2)), ("op -1", dict(op=-1)), ("mask", dict(mask=1 << 16)), ("qsize 3", dict(qsize=Q_ + 1)),
        ("null output", dict(null_out=True)))]
    + [("caar_set_partition", c, "ready", o, code) for c, o, code in PART_BAD]
)


@pytest.fixture(scope="module")
def env():
    gid = do.cubed_sphere_gid(2, np.random.default_rng(4))
    s = harness.randomize(harness.PortOracle().init(E_, L_, Q_, NTL_), seed=4)
    hs = {k: tb.Caar(PS_[2] - PS_[1], L_, Q_, NTL_) for k in ("bare", "connected", "ready")}
    for k, h in hs.items():
        h.upload({n: np.ascontiguousarray(a[PS_[1]:]) for n, a in s.arrays.items()})
        if k == "connected":
            h.set_connectivity(gid[PS_[1]:])
        if k == "ready":
            h.set_partition(gid, PS_, 1)
        h.upload_bounds(np.sort(np.random.default_rng(5).standard_normal((PS_[2] - PS_[1], Q_, L_, 2)), -1))
    yield dict(gid=gid, handles=hs)
    for h in hs.values():
        h.close()


def call(env, ep, kind, over):
    lib = tb.load_library()
    h = env["handles"][kind].h if kind else None
    if ep in ENTRIES:
        a = {**GOOD_DSS, **over}
        return getattr(lib, ep)(h, a["mask"], a["tl"], a["qtl"], a["qsize"], a["weighting"])
    if ep in ("caar_neighbor_minmax_pack", "caar_neighbor_minmax_unpack"):
        return getattr(lib, ep)(h, over.get("qsize", 2))
    if ep == "caar_halo_segments":
        sp, rp = C.c_void_p(), C.c_void_p()
        so_, ro = (C.c_size_t * 3)(), (C.c_size_t * 3)()
        if over.get("null_out"):
            return lib.caar_halo_segments(h, 0, 0, 0, None, C.byref(rp), so_, ro)
        return lib.caar_halo_segments(h, over.get("op", 0), over.get("mask", 0), over.get("qsize", 0), C.byref(sp),
                                      C.byref(rp), so_, ro)
    gid = np.ascontiguousarray(env["gid"])
    ps = over.get("ps", PS_)
    psa = None if ps is None else np.ascontiguousarray(ps, dtype=np.int32)
    nparts = over.get("nparts", 2 if ps is None else len(ps) - 1)
    return lib.caar_set_partition(h, None if "gid" in over else gid.ctypes.data_as(C.POINTER(C.c_longlong)),
                                  over.get("nglob", E_), None if psa is None else psa.ctypes.data_as(C.POINTER(C.c_int)),
                                  nparts, over.get("part", 1), over.get("layout", 0))


def snapshot(h):
    out = {n: np.empty(tb.field_shape(n, PS_[2] - PS_[1], L_, Q_, NTL_)) for n in ALL4}
    h.download(out, names=ALL4)
    out["bounds"] = h.download_bounds()
    return out


@pytest.mark.parametrize("ep,case,kind,over,want", ERR_CASES, ids=[f"{c[0]}-{c[1]}-{c[2]}" for c in ERR_CASES])
def test_rejected_call_changes_nothing(env, ep, case, kind, over, want):
    before = {k: snapshot(h) for k, h in env["handles"].items()}
    launches = {k: h.launch_count() for k, h in env["handles"].items()}
    segs = env["handles"]["ready"].halo_segments(tb.HALO_DSS, ALL4, 2)
    rc = call(env, ep, kind, over)
    assert rc == want, tb.load_library().caar_last_error().decode()
    for k, h in env["handles"].items():
        h.sync()
        assert h.launch_count() == launches[k]
        after = snapshot(h)
        for n in after:
            assert np.array_equal(bits(after[n]), bits(before[k][n])), (k, n)
    after = env["handles"]["ready"].halo_segments(tb.HALO_DSS, ALL4, 2)
    assert after[0].data_ptr() == segs[0].data_ptr() and list(after[2]) == list(segs[2])   # the partition stays


def test_launch_counts(env):
    """1 per pack (a part with records to send) and unpack with work, 0 for an empty selection; set_partition and
    halo_segments launch nothing."""
    lib = tb.load_library()
    h = env["handles"]["ready"]
    for ep in ENTRIES:
        for args, n in (((0, 0, 0, 0, 0), 0), ((F["elem_state_Qdp"], 0, 0, 0, 0), 0),
                        ((F["elem_state_Qdp"], 0, 1, 1, 1), 1), ((F["elem_state_v"], 2, 0, 0, 0), 1),
                        ((sum(F.values()), 1, 1, 2, 1), 1)):
            k = h.launch_count()
            assert getattr(lib, ep)(h.h, *args) == 0
            h.sync()
            assert h.launch_count() - k == n, (ep, args)
    for ep in ("caar_neighbor_minmax_pack", "caar_neighbor_minmax_unpack"):
        for qs, n in ((0, 0), (1, 1), (2, 1)):
            k = h.launch_count()
            assert getattr(lib, ep)(h.h, qs) == 0
            assert h.launch_count() - k == n, (ep, qs)
    k = h.launch_count()
    h.set_partition(env["gid"], PS_, 1)
    h.halo_segments(tb.HALO_MINMAX, (), 2)
    assert h.launch_count() == k
