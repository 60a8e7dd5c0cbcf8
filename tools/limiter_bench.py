#!/usr/bin/env python
"""Times caar_tracer_bounds and caar_limit_tracers (HOMME's quasi-monotone limiter, limiter_option 8) on resident data.
    python tools/limiter_bench.py [--configs 86400x72q4,21600x72q35,49152x128q4] [--reps 10]
Prints one JSON line per configuration and input regime:
  inbounds     Qdp(0) within the bounds caar_tracer_bounds computed from it: one pass per problem
  advected     the bounds of Qdp(0), then one fast caar_advect_tracers step (dt = 1 s), limiting Qdp(1)
  adversarial  staircase problems (tests/test_limiter_cpu.staircase, geometric weights): most need >= 10 passes
The limiter changes Qdp and may relax the bounds, so before every timed call Qdp is restored from a device copy
(a device-to-device copy on the handle's stream) and the bounds from pinned host memory; only the kernel is inside the
CUDA events. Reported: min and median ms over --reps calls, GB/s over the algorithmic bytes per problem
(limiter 256 + 32 + 128/qsize + 128/(L qsize), bounds 128 + 128/qsize + 16), the fraction of the device-to-device copy
rate measured in the same process, the byte-bound time at that rate, and the card's name, power limit and SM clocks
from a read-only nvidia-smi query."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
import tinman_sandbox_b200 as tb  # noqa: E402
from rk5_bench import copy_peak_gbps, gpu_info  # noqa: E402
from test_levelop_regimes_cpu import lean_inputs  # noqa: E402
from test_limiter_cpu import staircase, staircase_weights  # noqa: E402

import limiter_oracle as lo  # noqa: E402

POOL = 257
DT = 1.0
GEOM = ("elem_Dinv", "elem_metdet", "elem_rmetdet")


def limiter_bytes(L, q):
    return 256.0 + 32.0 + 128.0 / q + 128.0 / (L * q)


def bounds_bytes(L, q):
    return 128.0 + 128.0 / q + 16.0


def pool_arrays(L, Q, regime, rng):
    """one pool of POOL elements of every array the regime reads, and the pool's bounds [POOL][Q][L][2] (adversarial)"""
    s, vin, _, _ = lean_inputs("randomize", POOL, L, 2026, scalar=False)
    a = {n: s.arrays[n] for n in GEOM}
    sph = rng.uniform(0.5, 2.0, (POOL, 4, 4))
    dp = rng.uniform(0.5, 2.0, (POOL, 3, L, 4, 4)) * 10.0 ** rng.uniform(0, 3, (POOL, 1, L, 1, 1))
    x = rng.uniform(0.0, 1.0, (POOL, Q, 2, L, 4, 4)) * rng.uniform(0.01, 0.2, (POOL, Q, 1, 1, 1, 1))
    bounds = None
    if regime == "adversarial":
        dp[...] = 1.0
        bounds = np.zeros((POOL, Q, L, 2))
        for e in range(POOL):
            cF = staircase_weights(rng, 1)[0]
            sph[e].reshape(16)[lo.FORTRAN] = cF
            n = Q * 2 * L
            xF, _ = staircase(rng, n, np.tile(cF, (n, 1)))
            scale = rng.uniform(0.01, 0.2, (n, 1))
            xe = np.empty((n, 16))
            xe[:, lo.FORTRAN] = xF * scale
            x[e] = xe.reshape(Q, 2, L, 4, 4)
            bounds[e, ..., 1] = scale.reshape(Q, 2, L)[:, 0]
    a["elem_spheremp"], a["elem_state_dp3d"] = sph, dp
    a["elem_state_Qdp"] = x * dp[:, 0][:, None, None]
    return a, vin, bounds


def tiled(h, pool, E):
    for e0 in range(0, E, POOL):
        e1 = min(E, e0 + POOL)
        h.upload_range({n: np.ascontiguousarray(v[:e1 - e0]) for n, v in pool.items()}, e0, e1, names=tuple(pool))


def device_view(ptr, n):
    """torch float64 tensor over n doubles of device memory at ptr (no copy)"""
    import torch

    class Mem:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3}
    return torch.as_tensor(Mem(), device="cuda")


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="86400x72q4,21600x72q35,49152x128q4")
    ap.add_argument("--regimes", default="inbounds,advected,adversarial")
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    info = gpu_info()
    peak = copy_peak_gbps()
    for cfg in args.configs.split(","):
        el, q = cfg.split("q")
        E, L = (int(x) for x in el.split("x"))
        Q = int(q)
        n = E * L * Q
        for regime in args.regimes.split(","):
            rng = np.random.default_rng(11)
            pool, vin, pb = pool_arrays(L, Q, regime, rng)
            h = tb.Caar(E, L, Q)
            s0 = lean_inputs("randomize", 1, L, 1, scalar=False)[0]
            h.set_params(s0.consts, s0.dvv, s0.ps0, s0.hyai)
            stream = torch.cuda.current_stream()
            h.set_stream(stream.cuda_stream)
            tiled(h, pool, E)
            qtl = 0
            if regime == "adversarial":
                bounds = np.ascontiguousarray(np.concatenate([pb] * (-(-E // POOL)))[:E])
            else:
                h.tracer_bounds(0, Q, 0)
                if regime == "advected":
                    h.upload_vstar(np.ascontiguousarray(np.concatenate([vin] * (-(-E // POOL)))[:E]))
                    qtl = h.advect_tracers(0, Q, DT, 1, tb.MODE_FAST)
                bounds = h.download_bounds()
            tb.host_register({"bounds": bounds})
            qdp = device_view(h.device_pointers()["elem_state_Qdp"], E * Q * 2 * L * 16)
            saved = qdp.clone()
            tb_ms, lim_ms = [], []
            for r in range(args.reps + 1):
                qdp.copy_(saved)
                h.upload_bounds(bounds)
                h.timer_start()
                h.limit_tracers(qtl, Q, 0, sync=False)
                t = h.timer_stop()
                h.timer_start()
                h.tracer_bounds(qtl, Q, 0, sync=False)
                u = h.timer_stop()
                if r:   # the first call warms up
                    lim_ms.append(t)
                    tb_ms.append(u)
            h.set_stream(None)
            tb.host_unregister({"bounds": bounds})
            del qdp, saved
            torch.cuda.empty_cache()
            h.close()
            bl, bb = n * limiter_bytes(L, Q), n * bounds_bytes(L, Q)
            rec = {"config": cfg, "regime": regime, "nelem": E, "nlev": L, "qsize": Q, "reps": args.reps}
            for name, ms, by in (("limit", lim_ms, bl), ("bounds", tb_ms, bb)):
                best, med = min(ms), float(np.median(ms))
                rec[name] = {"ms_min": round(best, 4), "ms_median": round(med, 4), "bytes": by,
                             "GBps": round(by / (best * 1e-3) / 1e9, 1),
                             "frac_copy_peak": round(by / (best * 1e-3) / 1e9 / peak, 4),
                             "byte_bound_ms_at_copy_peak": round(by / (peak * 1e9) * 1e3, 3)}
            rec["copy_peak_GBps"] = round(peak, 1)
            rec["gpu"] = info
            print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
