"""Element partition across ranks — the reference's own nets/nete hook (pointers_only/data_structures.hpp:58-66,
compute_and_apply_rhs.cpp:65-74) applied per GPU: rank g of G owns the contiguous block
[floor(g*E/G), floor((g+1)*E/G)). compute_and_apply_rhs has no inter-element coupling; the DSS and the neighbour
limiter bounds do, and ``halo_exchange`` assembles them across ranks with point-to-point sends of the segments that
caar_dss_pack / caar_neighbor_minmax_pack write (HOMME's bndry_exchangeV). ``run_rk5_dss`` runs HOMME's RK5 step with
that exchange after every stage, the interior points assembled while the segments are in flight. The other exchanges
of a job are the final sums of the three squared norms and of the checksums."""
from __future__ import annotations

import numpy as np

from .capi import HALO_DSS, MODE_FAST


def element_range(rank: int, world: int, nelem: int):
    if not (0 <= rank < world) or nelem < 0:
        raise ValueError("bad partition arguments")
    return (nelem * rank) // world, (nelem * (rank + 1)) // world


def reduce_norms(local_sumsq, all_reduce_sum=None):
    """local sums of squares (v, T, dp3d) -> global 2-norms. all_reduce_sum(np.ndarray) -> np.ndarray sums over
    ranks (torch.distributed with NCCL on GPUs, gloo in the CPU tests); None = single rank."""
    s = np.asarray(local_sumsq, dtype=np.float64)
    if all_reduce_sum is not None:
        s = all_reduce_sum(s)
    return np.sqrt(s)


def reduce_checksums(local, all_reduce_sum=None):
    """Per-rank caar_checksums (dict with float64 `sum`, `sumsq`, `energy` and uint64 `bits`) -> the job's: the doubles are
    summed as doubles, the bit-pattern sums as 64-bit integers with wrap-around (exact, independent of the partition).
    all_reduce_sum(np.ndarray) -> np.ndarray sums over ranks for float64 AND int64 arrays; None = single rank."""
    f = np.concatenate([np.asarray(local["sum"], dtype=np.float64), np.asarray(local["sumsq"], dtype=np.float64),
                        np.asarray(local["energy"], dtype=np.float64)])
    b = np.asarray(local["bits"], dtype=np.uint64).view(np.int64).copy()
    if all_reduce_sum is not None:
        f = all_reduce_sum(f)
        b = all_reduce_sum(b)
    n = len(local["sum"])
    return {"sum": f[:n], "sumsq": f[n:2 * n], "energy": f[2 * n:], "bits": b.view(np.uint64)}


def _post_segments(send, recv, so, ro, group):
    """Posts the receive and the send of every non-empty segment between this rank and each other rank of `group` as
    one batch of point-to-point ops on views of the handle's buffers -> the works to wait on."""
    import torch.distributed as dist

    me = dist.get_rank(group)
    ops = []
    for q in range(len(so) - 1):
        if q == me:
            continue
        peer = q if group is None else dist.get_global_rank(group, q)
        if ro[q + 1] > ro[q]:
            ops.append(dist.P2POp(dist.irecv, recv[ro[q]:ro[q + 1]], peer, group))
        if so[q + 1] > so[q]:
            ops.append(dist.P2POp(dist.isend, send[so[q]:so[q + 1]], peer, group))
    return dist.batch_isend_irecv(ops) if ops else []


def halo_exchange(caar, op, mask, qsize, group=None, tl=None, qtl=0, weighting=0):
    """One exchange of a rank of a torch.distributed job whose rank r (in `group`) holds part r of the partition given
    to caar.set_partition: pack, send and receive every non-empty segment with point-to-point ops on views of the
    handle's buffers, wait, unpack. op is HALO_DSS (mask: the names of the fields, with tl, qtl, qsize, weighting as
    in Caar.dss) or HALO_MINMAX (the limiter bounds of tracers < qsize; mask is ignored). Returns after the unpack
    has been queued on the handle's stream."""
    import torch

    names = tuple(mask) if op == HALO_DSS else ()
    if op == HALO_DSS:
        caar.dss_pack(names, tl=tl, qtl=qtl, qsize=qsize, weighting=weighting, sync=True)
    else:
        caar.neighbor_minmax_pack(qsize, sync=True)
    send, recv, so, ro = caar.halo_segments(op, names, qsize)
    for w in _post_segments(send, recv, so, ro, group):
        w.wait()
    torch.cuda.synchronize(send.device)   # the received segments are in place before the handle's stream reads them
    if op == HALO_DSS:
        caar.dss_unpack(names, tl=tl, qtl=qtl, qsize=qsize, weighting=weighting, sync=False)
    else:
        caar.neighbor_minmax_unpack(qsize, sync=False)


STATE = ("elem_state_dp3d", "elem_state_v", "elem_state_T")


def run_rk5_dss(caar, nsteps, dt, mode=MODE_FAST, group=None):
    """nsteps of HOMME's RK5 dynamics step (tstep_type 5) with the exchanged DSS of v, T and dp3d after every stage, on
    the part this rank holds (rank r of `group` holds part r of caar.set_partition; caar.control spans the part). Per
    stage: rk5_stage, dss_pack, the segment sends and receives, dss_interior, a wait on the receives, dss_boundary;
    after stage 4 the control rotates. The handle's stream becomes torch's current stream (caar_set_stream), so the
    NCCL ops wait on the pack, the interior launch runs while the segments are in flight, and work.wait() orders the
    boundary launch after the receives; there is no host synchronisation inside the step. Over a block partition the
    parts end with the slices of caar_run_rk5_dss on one handle of the whole mesh, bit for bit. Returns with the work
    queued; the handle stays on torch's current stream."""
    import torch

    caar.set_stream(torch.cuda.current_stream(caar.device).cuda_stream)
    send, recv, so, ro = caar.halo_segments(HALO_DSS, STATE, 0)
    for _ in range(nsteps):
        for stage in range(5):
            tl = caar.rk5_stage(stage, dt, mode, sync=False)
            caar.dss_pack(STATE, tl=tl, sync=False)
            works = _post_segments(send, recv, so, ro, group)
            caar.dss_interior(STATE, tl=tl, sync=False)
            for w in works:
                w.wait()
            caar.dss_boundary(STATE, tl=tl, sync=False)
        caar.update_time_levels()
