"""caar_rk5_stage, caar_dss_interior and caar_dss_boundary on the GPU, bit for bit: the five public stages compose to
caar_run_rk5 and, with caar_dss after each, to caar_run_rk5_dss (strict and fast, Lagrangian and Eulerian, nlev 72, 30,
5, 80 and 127, 2 steps); interior + boundary in either order, and interior queued before pack, equal caar_dss_unpack and
the whole-mesh caar_dss for every selection, at the level counts of tests/test_dss_partition_gpu.py's CASES; several
handles on one GPU step HOMME's RK5 step with the split DSS and equal one whole-mesh caar_run_rk5_dss (nlev 72, 80, 127
and 5); ne = 120 in 8 parts; rejected calls; and two ranks over NCCL
(partition.run_rk5_dss)."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
import dss_oracle as do
import dss_partition_oracle as dpo
import rk5_partition_oracle as rpo
from oracle import harness
from test_dss_partition_gpu import (ALL4, CASES, MESHES, SEL_NAMES, SELECTIONS, download_parts, move_segments,
                                    nan_fill, part_handles, random_fields, upload_parts)

pytestmark = pytest.mark.gpu
INVALID, STATE_ERR = 1, 5
F = {n: tb.capi.FIELD_BIT[n] for n in tb.DSS_FIELDS}
STATE = ("elem_state_dp3d", "elem_state_v", "elem_state_T")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = 2.0


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


# ---- the public stages ----------------------------------------------------------------------------------------------

def rk5_state(ne, L, seed, E_part=None):
    gid = do.cubed_sphere_gid(ne, np.random.default_rng(seed))
    s = harness.randomize(harness.PortOracle().init(gid.shape[0], L), seed=seed)
    s.ctl[0:2] = (0, s.nelem)
    s.ctl[2:5] = (0, 1, 2)
    return s, gid


def rk5_handle(s, hybi, e0=0, e1=None):
    e1 = s.nelem if e1 is None else e1
    h = tb.Caar(e1 - e0, s.nlev, s.qsize_d, s.ntl)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    if hybi is not None:
        h.set_vertical_coordinate(0, hybi)
    h.set_control(0, e1 - e0, *[int(x) for x in s.ctl[2:6]], dt2=s.dt2)
    h.upload({n: np.ascontiguousarray(a[e0:e1]) for n, a in s.arrays.items()})
    return h


def download_all(h, s, E):
    out = {n: np.empty(tb.field_shape(n, E, s.nlev, s.qsize_d, s.ntl)) for n in harness.FIELD_NAMES}
    h.download(out, names=None)
    return out


@pytest.mark.parametrize("mode", [tb.MODE_STRICT, tb.MODE_FAST], ids=["strict", "fast"])
@pytest.mark.parametrize("eulerian", [False, True], ids=["lagrangian", "eulerian"])
@pytest.mark.parametrize("L", [72, 30, 5, 80, 127])
def test_stages_compose_to_run_rk5_and_run_rk5_dss(mode, eulerian, L):
    """2 steps: stages 0..4 + update_time_levels equal caar_run_rk5, and with caar_dss(V|T|DP3D, *tl) after every
    stage equal caar_run_rk5_dss, in every bit of every array; 1, 1, 1, 1, 2 launches; *tl = nm1, np1, np1, np1, np1."""
    s, gid = rk5_state(3, L, 60 + L + eulerian)
    hybi = np.linspace(0.0, 1.0, L + 1) ** 1.5 if eulerian else None
    for dss in (False, True):
        ref, got = rk5_handle(s, hybi), rk5_handle(s, hybi)
        for h in (ref, got):
            h.set_connectivity(gid)
        (ref.run_rk5_dss if dss else ref.run_rk5)(2, DT, mode)
        for _ in range(2):
            c = got.control
            want_tl = [c.nm1] + [c.np1] * 4
            for k in range(5):
                n = got.launch_count()
                tl = got.rk5_stage(k, DT, mode, sync=False)
                assert tl == want_tl[k] and got.launch_count() - n == (2 if k == 4 else 1), (k, tl)
                if dss:
                    got.dss(STATE, tl=tl, sync=False)
            got.update_time_levels()
        a, b = download_all(ref, s, s.nelem), download_all(got, s, s.nelem)
        assert (ref.control.n0, ref.control.np1, ref.control.nm1) == (got.control.n0, got.control.np1, got.control.nm1)
        for n in harness.FIELD_NAMES:
            assert np.array_equal(bits(a[n]), bits(b[n])), (dss, n)
        for h in (ref, got):
            h.close()


# ---- interior + boundary --------------------------------------------------------------------------------------------

def split_dss(hs, names, tl, qtl, qs, w, order):
    if order == "interior_before_pack":
        for h in hs:
            h.dss_interior(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
    nan_fill(hs, 0)
    for h in hs:
        h.dss_pack(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
    move_segments(hs, tb.HALO_DSS, names, qs)
    for h in hs:
        if order == "interior_first":
            h.dss_interior(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
        h.dss_boundary(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
        if order == "boundary_first":
            h.dss_interior(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)


@pytest.mark.parametrize("mesh,L,parts", CASES, ids=[f"{m}-L{L}-{p if isinstance(p, int) else len(p) - 1}"
                                                      for m, L, p in CASES])
def test_interior_and_boundary_equal_unpack(mesh, L, parts):
    """Every selection with both weightings, tl and qtl cycling, qsize < qsize_d, in three orders: the parts equal
    caar_dss_unpack's parts and the whole-mesh caar_dss in every bit of all four fields (outside the selection the
    inputs stay); each call launches once when its part has such groups and never otherwise."""
    idx = CASES.index((mesh, L, parts))
    rng = np.random.default_rng(idx)
    gid = MESHES[mesh](rng)
    E, Qd, ntl = gid.shape[0], 4, 3
    ps = np.array(parts, dtype=np.int32) if not isinstance(parts, int) else dpo.block_partition(E, parts, rng)
    inp = random_fields(E, L, Qd, ntl, 17 * L + idx)
    whole = tb.Caar(E, L, Qd, ntl)
    whole.upload(inp, names=SEL_NAMES)
    whole.set_connectivity(gid)
    hs, us = part_handles(gid, ps, L, Qd, ntl, inp), part_handles(gid, ps, L, Qd, ntl, inp)
    split = [rpo.SplitPart(gid, ps, p) for p in range(len(ps) - 1)]
    lib = tb.load_library()
    i = 0
    for names in SELECTIONS:
        for w in (do.ASSEMBLE, do.PROJECT):
            tl, qtl, qs = i % ntl, (i // 3) % 2, 3 if i % 2 else 1
            i += 1
            whole.upload(inp, names=ALL4)
            whole.dss(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
            ref = {n: np.empty(tb.field_shape(n, E, L, Qd, ntl)) for n in ALL4}
            whole.download(ref, names=ALL4)
            upload_parts(us, ps, inp, ALL4)
            nan_fill(us, 0)
            for h in us:
                h.dss_pack(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
            move_segments(us, tb.HALO_DSS, names, qs)
            for h in us:
                h.dss_unpack(names, tl=tl, qtl=qtl, qsize=qs, weighting=w)
            unpacked = download_parts(us, ps, E, L, Qd, ntl, ALL4)
            for order in ("interior_first", "boundary_first", "interior_before_pack"):
                upload_parts(hs, ps, inp, ALL4)
                split_dss(hs, names, tl, qtl, qs, w, order)
                got = download_parts(hs, ps, E, L, Qd, ntl, ALL4)
                for n in ALL4:
                    assert np.array_equal(bits(got[n]), bits(unpacked[n])), (names, w, order, n)
                    assert np.array_equal(bits(got[n]), bits(ref[n])), (names, w, order, n)
                    if n not in names:
                        assert np.array_equal(bits(got[n]), bits(inp[n])), (names, w, order, n)
            for h, pt in zip(hs, split):
                for ep, groups in (("caar_dss_interior", pt.interior), ("caar_dss_boundary", pt.boundary)):
                    k = h.launch_count()
                    assert getattr(lib, ep)(h.h, sum(F[n] for n in names), tl, qtl, qs, w) == 0
                    assert h.launch_count() - k == (1 if groups else 0), (ep, names)
                    assert getattr(lib, ep)(h.h, 0, tl, qtl, qs, w) == 0
                    assert getattr(lib, ep)(h.h, F["elem_state_Qdp"], tl, qtl, 0, w) == 0
                    assert h.launch_count() - k == (1 if groups else 0), (ep, names)
    if len(ps) == 2:
        assert not split[0].boundary and split[0].interior      # nparts == 1: no boundary launch at all
    for h in hs + us + [whole]:
        h.close()


# ---- HOMME's step across handles of one GPU -------------------------------------------------------------------------

def step_parts(hs, nsteps, dt, mode):
    """partition.run_rk5_dss's sequence with device copies for the transport"""
    for _ in range(nsteps):
        for k in range(5):
            tls = [h.rk5_stage(k, dt, mode, sync=False) for h in hs]
            nan_fill(hs, 0)
            for h, tl in zip(hs, tls):
                h.dss_pack(STATE, tl=tl)
            move_segments(hs, tb.HALO_DSS, STATE, 0)
            for h, tl in zip(hs, tls):
                h.dss_interior(STATE, tl=tl, sync=False)
                h.dss_boundary(STATE, tl=tl, sync=False)
        for h in hs:
            h.update_time_levels()


STEP_CASES = [(4, 3, tb.MODE_STRICT, 72), (4, 3, tb.MODE_FAST, 72), (30, 4, tb.MODE_FAST, 72),
              (4, 3, tb.MODE_FAST, 80), (4, 3, tb.MODE_STRICT, 127), (4, 3, tb.MODE_STRICT, 5)]


@pytest.mark.parametrize("ne,nparts,mode,L", STEP_CASES,
                         ids=[f"ne{ne}-{n}-{'strict' if m == tb.MODE_STRICT else 'fast'}" + ("" if L == 72 else f"-L{L}")
                              for ne, n, m, L in STEP_CASES])
def test_partitioned_rk5_step_equals_whole_mesh(ne, nparts, mode, L):
    """2 RK5 steps with the split DSS after every stage on nparts handles of one GPU equal one whole-mesh
    caar_run_rk5_dss in every bit of every array (ne = 4 permuted with a one-element block; ne = 30 in even blocks), at
    nlev 72, 80, 127 and 5."""
    s, gid = rk5_state(ne, L, 70 + ne + (L != 72) * L)
    E = s.nelem
    rng = np.random.default_rng(ne)
    ps = dpo.block_partition(E, nparts, rng) if ne == 4 else \
        np.array([(E * p) // nparts for p in range(nparts + 1)], dtype=np.int32)
    whole = rk5_handle(s, None)
    whole.set_connectivity(gid)
    whole.run_rk5_dss(2, DT, mode)
    hs = []
    for p in range(nparts):
        h = rk5_handle(s, None, int(ps[p]), int(ps[p + 1]))
        h.set_partition(gid, ps, p)
        hs.append(h)
    step_parts(hs, 2, DT, mode)
    want = download_all(whole, s, E)
    got = download_parts(hs, ps, E, s.nlev, s.qsize_d, s.ntl, harness.FIELD_NAMES)
    for n in harness.FIELD_NAMES:
        assert np.array_equal(bits(got[n]), bits(want[n])), n
    assert all((h.control.n0, h.control.np1, h.control.nm1) == (whole.control.n0, whole.control.np1,
                                                                 whole.control.nm1) for h in hs)
    for h in hs + [whole]:
        h.close()


def test_ne120_in_8_parts():
    """ne = 120 x 72 in 8 parts: one split DSS of dp3d, v and T equals the whole-mesh caar_dss: every part's
    caar_checksums bits for dp3d, v and T equal the whole handle's over the part's range, and sampled elements are
    equal exactly."""
    ne, L, nparts = 120, 72, 8
    gid = do.cubed_sphere_gid(ne)
    E = gid.shape[0]
    ps = np.array([(E * p) // nparts for p in range(nparts + 1)], dtype=np.int32)
    rng = np.random.default_rng(120)
    inp = {"elem_spheremp": rng.uniform(0.5, 2.0, (E, 4, 4))}
    for n in STATE:
        inp[n] = rng.uniform(1.0, 3.0, tb.field_shape(n, E, L, 1, 1))
    sel = ("elem_spheremp",) + STATE
    whole = tb.Caar(E, L, 1, 1)
    whole.upload(inp, names=sel)
    whole.set_connectivity(gid)
    whole.dss(STATE, tl=0)
    hs = part_handles(gid, ps, L, 1, 1, inp, sel)
    split_dss(hs, STATE, 0, 0, 0, do.ASSEMBLE, "interior_first")
    sample = np.sort(rng.choice(E, 64, replace=False))
    for p, h in enumerate(hs):
        a = h.checksums(0, 0, int(ps[p + 1] - ps[p]))["bits"][:3]
        b = whole.checksums(0, int(ps[p]), int(ps[p + 1]))["bits"][:3]
        assert np.array_equal(a, b), p
        for e in sample[(sample >= ps[p]) & (sample < ps[p + 1])]:
            x = h.download_range(int(e - ps[p]), int(e - ps[p]) + 1, names=STATE)
            y = whole.download_range(int(e), int(e) + 1, names=STATE)
            for n in STATE:
                assert np.array_equal(bits(x[n]), bits(y[n])), (p, e, n)
    for h in hs + [whole]:
        h.close()


# ---- rejected calls -------------------------------------------------------------------------------------------------

E_, L_, Q_, NTL_ = 24, 16, 2, 3
PS_ = (0, 10, 24)
GOOD_DSS = dict(mask=F["elem_state_T"] | F["elem_state_Qdp"], tl=0, qtl=0, qsize=2, weighting=0)
DSS_BAD = ([dict(mask=tb.capi.FIELD_BIT["elem_spheremp"]), dict(mask=1 << 16), dict(tl=-1), dict(tl=NTL_),
            dict(qtl=-1), dict(qtl=2), dict(qsize=-1), dict(qsize=Q_ + 1), dict(weighting=2), dict(weighting=-1)])
SPLIT = ("caar_dss_interior", "caar_dss_boundary")
STAGE_BAD = [("null control", dict(ctl=None)), ("range -1", dict(nets=-1)), ("range 0:15", dict(nete=15)),
             ("levels 0,0,1", dict(tls=(0, 0, 1))), ("levels 0,1,1", dict(tls=(0, 1, 1))),
             ("level 3", dict(tls=(0, 1, 3))), ("qn0 2", dict(qn0=2)), ("mode 7", dict(mode=7)),
             ("stage -1", dict(stage=-1)), ("stage 5", dict(stage=5)), ("null tl", dict(tl=None))]
ERR_CASES = (
    [(ep, "null handle", None, {}, INVALID) for ep in SPLIT + ("caar_rk5_stage",)]
    + [(ep, "not partitioned", k, {}, STATE_ERR) for ep in SPLIT for k in ("bare", "connected")]
    + [(ep, f"{k}={v}", "ready", {k: v}, INVALID) for ep in SPLIT for o in DSS_BAD for k, v in o.items()]
    + [("caar_rk5_stage", "before set_params", "noparams", {}, STATE_ERR)]
    + [("caar_rk5_stage", c, "ready", o, INVALID) for c, o in STAGE_BAD]
)


@pytest.fixture(scope="module")
def env():
    gid = do.cubed_sphere_gid(2, np.random.default_rng(4))
    s = harness.randomize(harness.PortOracle().init(E_, L_, Q_, NTL_), seed=4)
    hs = {k: tb.Caar(PS_[2] - PS_[1], L_, Q_, NTL_) for k in ("bare", "connected", "noparams", "ready")}
    for k, h in hs.items():
        if k != "noparams":
            h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
        h.upload({n: np.ascontiguousarray(a[PS_[1]:]) for n, a in s.arrays.items()})
        if k == "connected":
            h.set_connectivity(gid[PS_[1]:])
        if k in ("ready", "noparams"):
            h.set_partition(gid, PS_, 1)
    yield dict(gid=gid, handles=hs)
    for h in hs.values():
        h.close()


def call(env, ep, kind, over):
    lib = tb.load_library()
    h = env["handles"][kind].h if kind else None
    if ep in SPLIT:
        a = {**GOOD_DSS, **over}
        return getattr(lib, ep)(h, a["mask"], a["tl"], a["qtl"], a["qsize"], a["weighting"]), None, None
    tls = over.get("tls", (0, 1, 2))
    n = PS_[2] - PS_[1]
    ctl = tb.capi.Control(over.get("nets", 0), over.get("nete", n), *tls, over.get("qn0", 0), 0.5)
    tl = C.c_int(-7)
    rc = lib.caar_rk5_stage(h, None if "ctl" in over else C.byref(ctl), 1.0, over.get("stage", 0),
                            over.get("mode", tb.MODE_FAST), None if "tl" in over else C.byref(tl))
    return rc, (ctl.nets, ctl.nete, ctl.n0, ctl.np1, ctl.nm1, ctl.qn0, ctl.dt2), tl.value


def snapshot(h):
    out = {n: np.empty(tb.field_shape(n, PS_[2] - PS_[1], L_, Q_, NTL_)) for n in harness.FIELD_NAMES}
    h.download(out, names=None)
    return out


@pytest.mark.parametrize("ep,case,kind,over,want", ERR_CASES, ids=[f"{c[0]}-{c[1]}-{c[2]}" for c in ERR_CASES])
def test_rejected_call_changes_nothing(env, ep, case, kind, over, want):
    before = {k: snapshot(h) for k, h in env["handles"].items()}
    launches = {k: h.launch_count() for k, h in env["handles"].items()}
    rc, ctl, tl = call(env, ep, kind, over)
    assert rc == want, tb.load_library().caar_last_error().decode()
    for k, h in env["handles"].items():
        h.sync()
        assert h.launch_count() == launches[k]
        after = snapshot(h)
        for n in after:
            assert np.array_equal(bits(after[n]), bits(before[k][n])), (k, n)
    if ctl is not None:
        n = PS_[2] - PS_[1]
        assert ctl == (over.get("nets", 0), over.get("nete", n), *over.get("tls", (0, 1, 2)), over.get("qn0", 0), 0.5)
        assert tl == -7


def test_stage_launch_counts_and_empty_range(env):
    """1 launch per stage, 2 for stage 4; none for an empty element range, which still reports *tl."""
    lib = tb.load_library()
    h = env["handles"]["ready"]
    for nets, nete, per in ((0, PS_[2] - PS_[1], (1, 1, 1, 1, 2)), (3, 3, (0,) * 5)):
        ctl = tb.capi.Control(nets, nete, 0, 1, 2, 0, 0.5)
        for k in range(5):
            tl = C.c_int(-7)
            n = h.launch_count()
            assert lib.caar_rk5_stage(h.h, C.byref(ctl), 1.0, k, tb.MODE_FAST, C.byref(tl)) == 0
            assert h.launch_count() - n == per[k] and tl.value == (2 if k == 0 else 1)
        assert (ctl.n0, ctl.np1, ctl.nm1) == (0, 1, 2)
    h.sync()


# ---- two ranks over NCCL --------------------------------------------------------------------------------------------

E2, L2 = 96, 30
PS2 = [0, 37, 96]
WORKER = r'''
import os, sys
root, out = sys.argv[1], sys.argv[2]
sys.path[:0] = [root, os.path.join(root, "tests")]
import numpy as np
import torch
import torch.distributed as dist
import tinman_sandbox_b200 as tb
from tinman_sandbox_b200 import partition
import test_rk5_partition_gpu as t

dist.init_process_group("nccl")
r = dist.get_rank()
torch.cuda.set_device(r)
s, gid = t.rk5_state(4, t.L2, 91)
e0, e1 = t.PS2[r], t.PS2[r + 1]
h = tb.Caar(e1 - e0, s.nlev, s.qsize_d, s.ntl, device=r)
h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
h.set_control(0, e1 - e0, *[int(x) for x in s.ctl[2:6]], dt2=s.dt2)
h.upload({n: np.ascontiguousarray(a[e0:e1]) for n, a in s.arrays.items()})
h.set_partition(gid, t.PS2, r)
partition.run_rk5_dss(h, 2, t.DT, tb.MODE_FAST)
h.sync()
res = t.download_all(h, s, e1 - e0)
res["levels"] = np.array([h.control.n0, h.control.np1, h.control.nm1])
np.savez(os.path.join(out, f"rank{r}.npz"), **res)
h.close()
dist.destroy_process_group()
'''


def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def test_two_ranks_run_rk5_dss(tmp_path):
    """partition.run_rk5_dss on two ranks (a permuted ne = 4 sphere, blocks of 37 and 59 elements), 2 fast steps: the
    slices concatenate to one whole-mesh handle's caar_run_rk5_dss in every bit of every array."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    worker = tmp_path / "worker.py"
    worker.write_text(WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), str(worker), ROOT, str(tmp_path)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    ranks = [np.load(tmp_path / f"rank{r}.npz") for r in range(2)]
    s, gid = rk5_state(4, L2, 91)
    h = rk5_handle(s, None)
    h.set_connectivity(gid)
    h.run_rk5_dss(2, DT, tb.MODE_FAST)
    want = download_all(h, s, E2)
    levels = (h.control.n0, h.control.np1, h.control.nm1)
    h.close()
    for r in ranks:
        assert tuple(r["levels"]) == levels
    for n in harness.FIELD_NAMES:
        got = np.concatenate([r[n] for r in ranks])
        assert np.array_equal(bits(got), bits(want[n])), n
