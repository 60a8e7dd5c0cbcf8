#!/usr/bin/env python
"""Times caar_advect_tracers (HOMME's three-stage tracer step, rkstage = 3) on resident data, and each of its launch
kinds alone.
    python tools/advect_bench.py [--configs 86400x72q4,21600x72q35,49152x128q4] [--modes fast,strict] [--steps 20]
Prints one JSON line per configuration and mode:
  ms_per_step         CUDA events around --steps back-to-back steps, best of 3 windows, after a warm-up step
  kind_ms             kernel time of each launch kind from a torch.profiler capture of --steps steps: the stage
                      (levelop_kernel<OP_EULER> in fast mode, euler_step_kernel<true> in strict mode; the mean of the
                      three stages) and the average (combine_kernel<QdpAverage>)
  euler_step_ms       caar_euler_step (into CAAR_X_QTENS) at the same size and dt/2, event-timed in windows that
                      alternate with the step windows: the fast stage runs its body, so the two rates should match
  bytes               algorithmic, per element x level x tracer: a stage 256 + (256 + 1408/L)/qsize (Qdp in and out,
                      vstar and the geometry once per element and level), the average 384 (two levels in, one out),
                      the step 3 stages + the average; rates use each kind's own count
  frac_copy_peak      GB/s over the device-to-device copy rate measured in the same process (torch bf16 copy)
The state is lean: the geometry of tests/test_levelop_regimes_cpu.lean_inputs on a pool of 257 elements, tiled over
the handle, Qdp uniform in [0, 0.2] at both levels, vstar +-40 m/s and dt = 1 s (finite over any number of steps
timed here). The card's name, power limit and SM clocks come from a read-only nvidia-smi query in the same process."""
import argparse
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
import tinman_sandbox_b200 as tb  # noqa: E402
from rk5_bench import copy_peak_gbps, gpu_info  # noqa: E402
from test_levelop_regimes_cpu import lean_inputs  # noqa: E402

DT = 1.0
POOL = 257
QNAMES = ("elem_Dinv", "elem_metdet", "elem_rmetdet", "elem_state_Qdp")
STAGE_KERNELS = ("levelop_kernel", "euler_step_kernel")
AVG_KERNEL = "QdpAverage"


def stage_bytes(L, qsize):
    return 256.0 + (256.0 + 1408.0 / L) / qsize


def make_handle(E, L, qsize):
    s, vin, _, _ = lean_inputs("randomize", POOL, L, 2026, Q=qsize, qn0=0, qsize=qsize, scalar=False)
    rng = np.random.default_rng(7)
    s.arrays["elem_state_Qdp"][...] = rng.uniform(0.0, 0.2, size=s.arrays["elem_state_Qdp"].shape)
    h = tb.Caar(E, L, qsize)
    h.set_params(s.consts, s.dvv, s.ps0, s.hyai)
    reps = max(1, 1024 // POOL)
    tile = {n: np.ascontiguousarray(np.concatenate([s.arrays[n]] * reps)) for n in QNAMES}
    for e0 in range(0, E, POOL * reps):
        e1 = min(E, e0 + POOL * reps)
        h.upload_range({n: np.ascontiguousarray(a[:e1 - e0]) for n, a in tile.items()}, e0, e1, names=QNAMES)
    vstar = np.ascontiguousarray(np.concatenate([vin] * (-(-E // POOL)))[:E])
    h.upload_vstar(vstar)
    return h


def window(h, fn, reps):
    h.timer_start()
    for _ in range(reps):
        fn()
    return h.timer_stop() / reps


def profiled_kinds(h, qsize, mode, steps):
    """(mean stage kernel ms, average kernel ms, kernel names) from torch.profiler over `steps` steps."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.advect_tracers(0, qsize, DT, steps, mode)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    st = [e.time_range.elapsed_us() for e in ev if any(k in e.name for k in STAGE_KERNELS)]
    av = [e.time_range.elapsed_us() for e in ev if AVG_KERNEL in e.name]
    names = sorted({re.sub(r"\(.*", "", e.name.replace("(anonymous namespace)::", "")) for e in ev
                    if any(k in e.name for k in STAGE_KERNELS + (AVG_KERNEL,))})
    if len(st) != 3 * steps or len(av) != steps:
        return None, None, names
    return sum(st) / len(st) / 1e3, sum(av) / len(av) / 1e3, names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="86400x72q4,21600x72q35,49152x128q4")
    ap.add_argument("--modes", default="fast,strict")
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    info = gpu_info()
    peak = copy_peak_gbps()
    for cfg in args.configs.split(","):
        el, q = cfg.split("q")
        E, L = (int(x) for x in el.split("x"))
        Q = int(q)
        h = make_handle(E, L, Q)
        n = E * L * Q
        b_stage, b_avg = n * stage_bytes(L, Q), n * 384.0
        b_step = 3 * b_stage + b_avg
        for mode_name in args.modes.split(","):
            mode = tb.MODE_FAST if mode_name == "fast" else tb.MODE_STRICT
            step = lambda: h.advect_tracers(0, Q, DT, 2, mode, sync=False)   # two steps: qn0 back to 0
            euler = lambda: h.euler_step(0, Q, DT / 2, mode, sync=False)
            step()
            euler()
            h.sync()
            ms_step, ms_euler = 1e30, 1e30
            for _ in range(3):   # alternating windows
                ms_step = min(ms_step, window(h, step, max(1, args.steps // 2)) / 2)
                ms_euler = min(ms_euler, window(h, euler, args.steps))
            stage_ms, avg_ms, names = profiled_kinds(h, Q, mode, args.steps)
            gbps = lambda b, ms: round(b / (ms * 1e-3) / 1e9, 1) if ms else None
            rec = {
                "config": cfg, "nelem": E, "nlev": L, "qsize": Q, "mode": mode_name, "steps": args.steps, "dt": DT,
                "ms_per_step": round(ms_step, 4), "bytes_per_step": b_step, "GBps": gbps(b_step, ms_step),
                "copy_peak_GBps": round(peak, 1), "frac_copy_peak": round(b_step / (ms_step * 1e-3) / 1e9 / peak, 4),
                "byte_bound_ms_at_copy_peak": round(b_step / (peak * 1e9) * 1e3, 3),
                "kind_ms": {"stage": round(stage_ms, 4) if stage_ms else None,
                            "average": round(avg_ms, 4) if avg_ms else None},
                "kind_GBps": {"stage": gbps(b_stage, stage_ms), "average": gbps(b_avg, avg_ms)},
                "euler_step_ms": round(ms_euler, 4), "euler_step_GBps": gbps(b_stage, ms_euler),
                "profiled_kernels": names, "gpu": info,
            }
            print(json.dumps(rec), flush=True)
        h.close()


if __name__ == "__main__":
    main()
