#!/usr/bin/env python
"""Times caar_vertical_remap (HOMME's PPM vertical remap for rsplit > 0) on resident data.
    python tools/remap_bench.py [--configs 86400x72q0,86400x72q4,21600x72q35,49152x128q4] [--reps 10]
Prints one JSON line per configuration and regime:
  identity  dp_star == dp to rounding (the target of a surface pressure near ps0)
  under     every interface moved by under half of the thinner adjacent layer: a deformation under one cell
The remap changes dp3d, T, v and Qdp in place, so before every timed call the four arrays are restored from device copies
(device-to-device copies on the handle's stream); only the call is inside the CUDA events. Reported: min and median ms
over --reps calls, GB/s over the compulsory bytes (64 B per column and level for dp3d, T and v read and written, 16 B per
tracer), the fraction of the device-to-device copy rate measured in the same process, the byte-bound time at that rate,
and the card's name, power limit and SM clocks from a read-only nvidia-smi query."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
import tinman_sandbox_b200 as tb  # noqa: E402
from limiter_bench import device_view  # noqa: E402
from rk5_bench import copy_peak_gbps, gpu_info  # noqa: E402

import remap_oracle as ro  # noqa: E402

POOL = 257
CONSTS = (1.0 / 6.376e6, 1.0, 1004.64, 461.5, 287.04, 2.0 / 7.0)
STATE = ("elem_state_dp3d", "elem_state_v", "elem_state_T", "elem_state_Qdp")


def remap_bytes(E, L, qsize):
    return E * 16.0 * L * (64.0 + 16.0 * qsize)


def pool_arrays(L, Q, regime, rng):
    """POOL elements of dp3d, v, T (time level 0) and Qdp (level 0) in the regime"""
    cols = lambda c: np.ascontiguousarray(np.moveaxis(c.reshape(POOL, 16, L), 2, 1)).reshape(POOL, L, 4, 4)
    dpo = ro.columns(POOL * 16, L, regime, 5)
    dp = np.repeat(cols(dpo)[:, None], 3, 1)
    v = rng.uniform(-40.0, 40.0, (POOL, 3, L, 4, 4, 2))
    T = rng.uniform(200.0, 300.0, (POOL, 3, L, 4, 4))
    Q = np.zeros((POOL, Q, 2, L, 4, 4))
    for iq in range(Q.shape[1]):
        Q[:, iq, 0] = cols(ro.mixing_ratios(POOL * 16, L, 10 + iq) * dpo)
    return dict(elem_state_dp3d=dp, elem_state_v=v, elem_state_T=T, elem_state_Qdp=Q)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="86400x72q0,86400x72q4,21600x72q35,49152x128q4")
    ap.add_argument("--regimes", default="identity,under")
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    info = gpu_info()
    peak = copy_peak_gbps()
    for cfg in args.configs.split(","):
        el, q = cfg.split("q")
        E, L = (int(x) for x in el.split("x"))
        qs = int(q)
        Qd = max(qs, 1)
        for regime in args.regimes.split(","):
            pool = pool_arrays(L, Qd, regime, np.random.default_rng(11))
            h = tb.Caar(E, L, Qd)
            hyai, hybi = ro.coordinate(L)
            h.set_params(CONSTS, np.zeros(16), ro.PS0, hyai)
            h.set_vertical_coordinate(1, hybi)
            stream = torch.cuda.current_stream()
            h.set_stream(stream.cuda_stream)
            for e0 in range(0, E, POOL):
                e1 = min(E, e0 + POOL)
                h.upload_range({n: np.ascontiguousarray(v[:e1 - e0]) for n, v in pool.items()}, e0, e1, names=STATE)
            ptr = h.device_pointers()
            views = [device_view(ptr[n], int(np.prod(tb.field_shape(n, E, L, Qd, 3)))) for n in STATE]
            saved = [x.clone() for x in views]
            ms = []
            for r in range(args.reps + 1):
                for x, s in zip(views, saved):
                    x.copy_(s)
                h.timer_start()
                h.vertical_remap(tl=0, qtl=0, qsize=qs, sync=False)
                t = h.timer_stop()
                if r:   # the first call warms up
                    ms.append(t)
            h.set_stream(None)
            del views, saved
            torch.cuda.empty_cache()
            h.close()
            by = remap_bytes(E, L, qs)
            best, med = min(ms), float(np.median(ms))
            rec = {"config": cfg, "regime": regime, "nelem": E, "nlev": L, "qsize": qs, "reps": args.reps,
                   "ms_min": round(best, 4), "ms_median": round(med, 4), "bytes": by,
                   "GBps": round(by / (best * 1e-3) / 1e9, 1),
                   "frac_copy_peak": round(by / (best * 1e-3) / 1e9 / peak, 4),
                   "byte_bound_ms_at_copy_peak": round(by / (peak * 1e9) * 1e3, 3),
                   "copy_peak_GBps": round(peak, 1), "gpu": info}
            print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
