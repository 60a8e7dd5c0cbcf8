#!/usr/bin/env python
"""Times HOMME's RK5 dynamics step across the GPUs of one box, one rank per GPU, each holding its block of the ne = 120
mesh (86400 x 72 in total, panel order, blocks as partition.element_range cuts them; fast mode):
    python -m torch.distributed.run --nproc-per-node=N tools/rk5_partition_bench.py [--steps 10]
Three variants, alternating step by step:
  overlap     partition.run_rk5_dss: per stage rk5_stage, dss_pack, the NCCL sends and receives, dss_interior while
              the segments are in flight, then dss_boundary
  no_overlap  the same step with dss_pack, the NCCL exchange, a wait, then dss_unpack (nothing runs during the exchange)
  rk5         caar_run_rk5: the five stages and the combination with no DSS
A step is timed with CUDA events on torch's current stream of every rank after a barrier; rank 0 prints one JSON line
per variant with the min and median over --steps of the slowest rank's time, and the card's name, power limit and SM
clocks from a read-only nvidia-smi query, and the device-to-device copy rate measured in the same process."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
import tinman_sandbox_b200 as tb  # noqa: E402
from tinman_sandbox_b200 import partition  # noqa: E402
from rk5_bench import copy_peak_gbps, gpu_info  # noqa: E402

import dss_oracle as do  # noqa: E402
from oracle import harness  # noqa: E402

STATE = partition.STATE


def no_overlap_step(h, dt, send, recv, so, ro):
    for k in range(5):
        tl = h.rk5_stage(k, dt, tb.MODE_FAST, sync=False)
        h.dss_pack(STATE, tl=tl, sync=False)
        for w in partition._post_segments(send, recv, so, ro, None):
            w.wait()
        h.dss_unpack(STATE, tl=tl, sync=False)
    h.update_time_levels()


def main():
    import torch
    import torch.distributed as dist
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--ne", type=int, default=120)
    args = ap.parse_args()
    dist.init_process_group("nccl")
    r, n = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(r)
    E, L, P = 6 * args.ne * args.ne, 72, 257
    ps = [partition.element_range(p, n, E)[0] for p in range(n)] + [E]
    e0, e1 = ps[r], ps[r + 1]
    pool = harness.PortOracle().init(P, L)
    pool.arrays["elem_spheremp"][...] = 1.0
    h = tb.Caar(e1 - e0, L, device=r)
    h.set_params(pool.consts, pool.dvv, pool.ps0, pool.hyai)
    h.set_control(0, e1 - e0, 0, 1, 2, int(pool.ctl[5]), dt2=pool.dt2)
    for a0 in range(0, e1 - e0, P):
        a1 = min(e1 - e0, a0 + P)
        h.upload_range({k: np.ascontiguousarray(a[:a1 - a0]) for k, a in pool.arrays.items()}, a0, a1)
    h.set_partition(do.cubed_sphere_gid(args.ne), ps, r)
    stream = torch.cuda.current_stream()
    h.set_stream(stream.cuda_stream)
    send, recv, so, ro = h.halo_segments(tb.HALO_DSS, STATE, 0)
    runs = {"overlap": lambda: partition.run_rk5_dss(h, 1, 1.0),
            "no_overlap": lambda: no_overlap_step(h, 1.0, send, recv, so, ro),
            "rk5": lambda: h.run_rk5(1, 1.0, tb.MODE_FAST, sync=False)}
    for fn in runs.values():
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in runs}
    for _ in range(args.steps):
        for k, fn in runs.items():
            dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            t = torch.tensor([a.elapsed_time(b)], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms[k].append(float(t.item()))
    info = gpu_info() if r == 0 else {}
    peak = copy_peak_gbps() if r == 0 else 0.0
    if r == 0:
        for k, v in ms.items():
            print(json.dumps(dict(case=f"rk5_partition_{k}", gpus=n, E=E, L=L, min_ms=round(min(v), 3),
                                  median_ms=round(float(np.median(v)), 3), copy_gbps=round(peak, 1), **info)),
                  flush=True)
    h.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
