#!/usr/bin/env python
"""Times caar_dss, caar_neighbor_minmax and caar_run_rk5_dss on resident data over cubed-sphere connectivity.
    python tools/dss_bench.py [--reps 10] [--parts N]
With --parts N it times only the exchange across partitioned handles (parts_case below: pack, copies, unpack,
interior and boundary alone and summed) and HOMME's RK5 step on N handles of one GPU (parts_rk5_case). Otherwise it prints one JSON
line per case:
  state DSS (v, T, dp3d; ASSEMBLE) at 86400 x 72 (ne = 120) and 48600 x 128 (ne = 90)
  Qdp DSS (PROJECT) at 86400 x 72 with qsize 4 and 21600 x 72 (ne = 60) with qsize 35
  caar_neighbor_minmax at the two Qdp sizes
each in two element orders: "panel" (face by face, row by row: close to HOMME's space-filling order, neighbours a face
row apart) and "shuffled" (a random permutation with rotated element blocks: the neighbours of a group are anywhere, the
adversarial case for L2); and caar_run_rk5 against caar_run_rk5_dss at 86400 x 72 in fast mode, alternating call by call.
spheremp is 1, so ASSEMBLE and PROJECT both average the copies and the data stays bounded over repeated in-place calls.
Reported: min and median ms of --reps calls between CUDA events on the handle's stream, the compulsory bytes (every
selected value read and written once), GB/s over them, the fraction of the device-to-device copy rate measured in the
same process, the byte-bound time at that rate, and the card's name, power limit and SM clocks from a read-only
nvidia-smi query. A second pass under torch.profiler gives each case's kernel time (it writes no trace)."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
import tinman_sandbox_b200 as tb  # noqa: E402
from rk5_bench import copy_peak_gbps, gpu_info  # noqa: E402

import dss_oracle as do  # noqa: E402
from oracle import harness  # noqa: E402

STATE = ("elem_state_dp3d", "elem_state_v", "elem_state_T")


def mesh(ne, order):
    return do.cubed_sphere_gid(ne, np.random.default_rng(ne) if order == "shuffled" else None)


def timed(h, fn, reps):
    fn()
    h.sync()
    ms = []
    for _ in range(reps):
        h.timer_start()
        fn()
        ms.append(h.timer_stop())
    return min(ms), float(np.median(ms))


def kernel_ms(fn, h, reps, name):
    """mean device time of the kernels whose name contains `name`, over reps calls under torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    h.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        h.sync()
    ev = [e for e in prof.key_averages() if name in e.key]
    total = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in ev)
    count = sum(e.count for e in ev)
    torch.cuda.synchronize()
    return total / 1e3 / count if count else None


def report(case, order, E, L, nbytes, best, med, kms, peak, info):
    print(json.dumps(dict(case=case, order=order, E=E, L=L, bytes_gb=round(nbytes / 1e9, 3), min_ms=round(best, 4),
                          median_ms=round(med, 4), kernel_ms=None if kms is None else round(kms, 4),
                          gbps=round(nbytes / best / 1e6, 1), of_copy_rate=round(nbytes / best / 1e6 / peak, 3),
                          bound_ms=round(nbytes / peak / 1e6, 3), copy_gbps=round(peak, 1), **info)), flush=True)


def dss_cases(reps, peak, info):
    for case, ne, L, Qd, qs in (("state", 120, 72, 1, 0), ("state", 90, 128, 1, 0), ("qdp", 120, 72, 4, 4),
                                ("qdp", 60, 72, 35, 35)):
        E = 6 * ne * ne
        h = tb.Caar(E, L, Qd, 3 if case == "state" else 1)
        h.upload({"elem_spheremp": np.ones((E, 4, 4))}, names=("elem_spheremp",))
        for order in ("panel", "shuffled"):
            h.set_connectivity(mesh(ne, order))
            if case == "state":
                fn = lambda: h.dss(STATE, tl=1, sync=False)
                nbytes = 2 * 4 * E * L * 16 * 8
            else:
                fn = lambda: h.dss(("elem_state_Qdp",), tl=0, qtl=1, qsize=qs, weighting=tb.DSS_PROJECT, sync=False)
                nbytes = 2 * qs * E * L * 16 * 8
            best, med = timed(h, fn, reps)
            report(f"dss_{case}" + (f"_q{qs}" if qs else ""), order, E, L, nbytes, best, med,
                   kernel_ms(fn, h, reps, "dss_kernel"), peak, info)
            if case == "qdp":
                fn = lambda: h.neighbor_minmax(qs, sync=False)
                nbytes = 2 * qs * E * L * 16
                best, med = timed(h, fn, reps)
                report(f"neighbor_minmax_q{qs}", order, E, L, nbytes, best, med,
                       kernel_ms(fn, h, reps, "neighbor_minmax"), peak, info)
        h.close()


def rk5_case(reps, peak, info):
    E, L, P = 86400, 72, 257
    pool = harness.PortOracle().init(P, L)
    pool.arrays["elem_spheremp"][...] = 1.0
    h = tb.Caar(E, L)
    h.set_params(pool.consts, pool.dvv, pool.ps0, pool.hyai)
    h.set_control(0, E, 0, 1, 2, int(pool.ctl[5]), dt2=pool.dt2)
    for e0 in range(0, E, P):
        e1 = min(E, e0 + P)
        h.upload_range({n: np.ascontiguousarray(a[:e1 - e0]) for n, a in pool.arrays.items()}, e0, e1)
    h.set_connectivity(mesh(120, "panel"))
    runs = {"rk5": lambda: h.run_rk5(1, 1.0, tb.MODE_FAST, sync=False),
            "rk5_dss": lambda: h.run_rk5_dss(1, 1.0, tb.MODE_FAST, sync=False)}
    ms = {k: [] for k in runs}
    for k, fn in runs.items():
        fn()
    h.sync()
    for _ in range(reps):
        for k, fn in runs.items():
            h.timer_start()
            fn()
            ms[k].append(h.timer_stop())
    h.close()
    for k, nbytes in (("rk5", 90.7e9), ("rk5_dss", 122.5e9)):
        report(f"step_{k}", "panel", E, L, nbytes, min(ms[k]), float(np.median(ms[k])), None, peak, info)


def parts_case(nparts, reps, peak, info):
    """N handles on one GPU hold the blocks of the ne = 120 mesh (86400 x 72, panel order; blocks as
    partition.element_range cuts them) and assemble dp3d, v and T (ASSEMBLE). Timed with CUDA events on one stream,
    alternating rep by rep, on one non-default stream: caar_dss_pack on every part, the segment copies (one torch copy_ per non-empty segment,
    cudaMemcpyAsync), caar_dss_unpack on every part, and caar_dss on one handle that holds the whole mesh. Bytes:
    pack reads and writes every record, the copies read and write every segment, unpack and the whole-mesh DSS read and
    write every value once (unpack also reads the records). Also reported: the host time of caar_set_partition per
    part and the largest number of boundary copies a part sends."""
    import torch
    from tinman_sandbox_b200.partition import element_range
    ne, L = 120, 72
    E = 6 * ne * ne
    gid = mesh(ne, "panel")
    ps = [element_range(p, nparts, E)[0] for p in range(nparts)] + [E]
    stream = torch.cuda.Stream()      # not the default stream: caar_set_stream(h, 0) means the handle's own
    whole = tb.Caar(E, L, 1, 1)
    whole.upload({"elem_spheremp": np.ones((E, 4, 4))}, names=("elem_spheremp",))
    whole.set_connectivity(gid)
    whole.set_stream(stream.cuda_stream)
    hs, build_ms = [], []
    for p in range(nparts):
        h = tb.Caar(ps[p + 1] - ps[p], L, 1, 1)
        h.upload({"elem_spheremp": np.ones((ps[p + 1] - ps[p], 4, 4))}, names=("elem_spheremp",))
        t0 = time.perf_counter()
        h.set_partition(gid, ps, p)
        build_ms.append((time.perf_counter() - t0) * 1e3)
        h.set_stream(stream.cuda_stream)
        hs.append(h)
    segs = [h.halo_segments(tb.HALO_DSS, STATE, 0) for h in hs]
    moves = [(segs[q][1][segs[q][3][p]:segs[q][3][p + 1]], segs[p][0][segs[p][2][q]:segs[p][2][q + 1]])
             for q in range(nparts) for p in range(nparts) if segs[q][3][p + 1] > segs[q][3][p]]

    def copies():
        with torch.cuda.stream(stream):
            for dst, src in moves:
                dst.copy_(src)
    def split():
        for h in hs:
            h.dss_interior(STATE, tl=0, sync=False)
            h.dss_boundary(STATE, tl=0, sync=False)
    runs = {"pack": lambda: [h.dss_pack(STATE, tl=0, sync=False) for h in hs], "copies": copies,
            "unpack": lambda: [h.dss_unpack(STATE, tl=0, sync=False) for h in hs],
            "interior": lambda: [h.dss_interior(STATE, tl=0, sync=False) for h in hs],
            "boundary": lambda: [h.dss_boundary(STATE, tl=0, sync=False) for h in hs],
            "interior_boundary": split,
            "whole_dss": lambda: whole.dss(STATE, tl=0, sync=False)}
    nv = 1 + 4 * L
    sent = sum(int(s[2][-1]) for s in segs) * 8
    value_bytes = 2 * 4 * E * L * 16 * 8
    nbytes = {"pack": 2 * sent, "copies": 2 * sent, "unpack": value_bytes + sent, "interior": value_bytes - 2 * sent,
              "boundary": 3 * sent, "interior_boundary": value_bytes + sent, "whole_dss": value_bytes}
    for fn in runs.values():
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in runs}
    for _ in range(reps):
        for k, fn in runs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    for k in runs:
        report(f"parts{nparts}_{k}", "panel", E, L, nbytes[k], min(ms[k]), float(np.median(ms[k])), None, peak, info)
    records = max(int(s[2][-1]) for s in segs) // nv
    print(json.dumps(dict(case=f"parts{nparts}_set_partition", E=E, host_ms_max=round(max(build_ms), 1),
                          host_ms_mean=round(float(np.mean(build_ms)), 1), max_send_records=records,
                          max_send_fraction=round(records / (16 * max(np.diff(ps))), 4), **info)), flush=True)
    for h in hs + [whole]:
        h.close()


def parts_rk5_case(nparts, reps, peak, info):
    """HOMME's RK5 step on N handles of one GPU holding the blocks of the ne = 120 mesh (86400 x 72, fast mode), per
    stage: caar_rk5_stage on every part, caar_dss_pack on every part, the segment copies, caar_dss_interior and
    caar_dss_boundary on every part (partition.run_rk5_dss's sequence with device copies for the transport), against
    caar_run_rk5_dss on one handle that holds the whole mesh, alternating step by step on one stream. The bytes are
    rk5_case's step_rk5_dss model."""
    import torch
    from tinman_sandbox_b200.partition import element_range
    ne, L, P = 120, 72, 257
    E = 6 * ne * ne
    gid = mesh(ne, "panel")
    ps = [element_range(p, nparts, E)[0] for p in range(nparts)] + [E]
    pool = harness.PortOracle().init(P, L)
    pool.arrays["elem_spheremp"][...] = 1.0
    stream = torch.cuda.Stream()

    def handle(e0, e1):
        h = tb.Caar(e1 - e0, L)
        h.set_params(pool.consts, pool.dvv, pool.ps0, pool.hyai)
        h.set_control(0, e1 - e0, 0, 1, 2, int(pool.ctl[5]), dt2=pool.dt2)
        for a0 in range(0, e1 - e0, P):
            a1 = min(e1 - e0, a0 + P)
            h.upload_range({n: np.ascontiguousarray(a[:a1 - a0]) for n, a in pool.arrays.items()}, a0, a1)
        h.set_stream(stream.cuda_stream)
        return h
    whole = handle(0, E)
    whole.set_connectivity(gid)
    hs = []
    for p in range(nparts):
        h = handle(ps[p], ps[p + 1])
        h.set_partition(gid, ps, p)
        hs.append(h)
    segs = [h.halo_segments(tb.HALO_DSS, STATE, 0) for h in hs]
    moves = [(segs[q][1][segs[q][3][p]:segs[q][3][p + 1]], segs[p][0][segs[p][2][q]:segs[p][2][q + 1]])
             for q in range(nparts) for p in range(nparts) if segs[q][3][p + 1] > segs[q][3][p]]

    def step():
        for k in range(5):
            tls = [h.rk5_stage(k, 1.0, tb.MODE_FAST, sync=False) for h in hs]
            for h, tl in zip(hs, tls):
                h.dss_pack(STATE, tl=tl, sync=False)
            with torch.cuda.stream(stream):
                for dst, src in moves:
                    dst.copy_(src)
            for h, tl in zip(hs, tls):
                h.dss_interior(STATE, tl=tl, sync=False)
            for h, tl in zip(hs, tls):
                h.dss_boundary(STATE, tl=tl, sync=False)
        for h in hs:
            h.update_time_levels()
    runs = {"parts": step, "whole": lambda: whole.run_rk5_dss(1, 1.0, tb.MODE_FAST, sync=False)}
    for fn in runs.values():
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in runs}
    for _ in range(reps):
        for k, fn in runs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    for k in runs:
        report(f"parts{nparts}_step_rk5_dss_{k}", "panel", E, L, 122.5e9, min(ms[k]), float(np.median(ms[k])), None,
               peak, info)
    for h in hs + [whole]:
        h.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--parts", type=int, default=0, help="time the exchange over this many handles of the ne = 120 mesh")
    args = ap.parse_args()
    info = gpu_info()
    peak = copy_peak_gbps()
    if args.parts:
        parts_case(args.parts, args.reps, peak, info)
        parts_rk5_case(args.parts, max(3, args.reps // 2), peak, info)
        return
    dss_cases(args.reps, peak, info)
    rk5_case(max(3, args.reps // 2), peak, info)


if __name__ == "__main__":
    main()
