"""Element partition across ranks — the reference's own nets/nete hook (pointers_only/data_structures.hpp:58-66,
compute_and_apply_rhs.cpp:65-74) applied per GPU: rank g of G owns the contiguous block
[floor(g*E/G), floor((g+1)*E/G)). compute_and_apply_rhs has no inter-element coupling; the DSS and the neighbour
limiter bounds do, and ``halo_exchange`` assembles them across ranks with point-to-point sends of the segments that
caar_dss_pack / caar_neighbor_minmax_pack write (HOMME's bndry_exchangeV). The other exchanges of a job are the final
sums of the three squared norms and of the checksums."""
from __future__ import annotations

import numpy as np


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


def halo_exchange(caar, op, mask, qsize, group=None, tl=None, qtl=0, weighting=0):
    """One exchange of a rank of a torch.distributed job whose rank r (in `group`) holds part r of the partition given
    to caar.set_partition: pack, send and receive every non-empty segment with point-to-point ops on views of the
    handle's buffers, wait, unpack. op is HALO_DSS (mask: the names of the fields, with tl, qtl, qsize, weighting as
    in Caar.dss) or HALO_MINMAX (the limiter bounds of tracers < qsize; mask is ignored). Returns after the unpack
    has been queued on the handle's stream."""
    import torch
    import torch.distributed as dist

    from .capi import HALO_DSS

    names = tuple(mask) if op == HALO_DSS else ()
    if op == HALO_DSS:
        caar.dss_pack(names, tl=tl, qtl=qtl, qsize=qsize, weighting=weighting, sync=True)
    else:
        caar.neighbor_minmax_pack(qsize, sync=True)
    send, recv, so, ro = caar.halo_segments(op, names, qsize)
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
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()
    torch.cuda.synchronize(send.device)   # the received segments are in place before the handle's stream reads them
    if op == HALO_DSS:
        caar.dss_unpack(names, tl=tl, qtl=qtl, qsize=qsize, weighting=weighting, sync=False)
    else:
        caar.neighbor_minmax_unpack(qsize, sync=False)
