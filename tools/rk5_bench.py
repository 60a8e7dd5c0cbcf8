#!/usr/bin/env python
"""Times caar_run_rk5 (HOMME's tstep_type 5 dynamics step) on resident data, and each of its six launch kinds.
    python tools/rk5_bench.py [--configs 86400x72,49152x128,51840x30,21600x72e] [--modes fast,strict] [--steps 10]
A trailing "e" runs the Eulerian branch (hybi = linspace(0, 1, nlev + 1)). Prints one JSON line per configuration
and mode:
  ms_per_step        CUDA events around --steps back-to-back steps, best of 3 windows
  stage_ms           each launch kind alone: stages 1-5 as caar_run with that stage's levels, dt2 and eta_ave_w,
                     event-timed; the combination from a torch.profiler capture of run_rk5 (kernel time)
  bytes_per_step     algorithmic: stage 1 reads 17 level-fields (n0 == nm1 is read once), stages 2-5 21 each, the
                     combination 12 (read 4 at nm1 and 4 at n0, write 4), plus 1664 B of geometry per element and stage
  frac_copy_peak     GB/s over the device-to-device copy rate measured in the same process (torch bf16 copy)
  aliased_GBps       stages 3-5 (n0 == np1 != nm1) on their own: their bytes over the sum of their alone times
The state is the reference's closed form with spheremp = 1 (with its spheremp of 2 to 8 every stage scales the
state, and it overflows within a few steps); dt = 1 s keeps it finite. Before timing, one step is checked on 64
elements against tests/rk5_oracle.rk5_step on those elements alone: bit for bit in strict mode, 1e-12 per field in
fast mode. Each mode starts from the initial state, and the run stops if the state is not finite after its timed
steps (checksums of every time level). The card's name, power limit and SM clocks come from a read-only nvidia-smi query."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import tinman_sandbox_b200 as tb  # noqa: E402
from tinman_sandbox_b200.testdata import TestData  # noqa: E402
from oracle import harness  # noqa: E402
import rk5_oracle as ro  # noqa: E402

DT = 1.0
LF_STAGE1, LF_STAGE, LF_COMBINE, GEO = 17, 21, 12, 1664


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True, check=False).stdout.strip()
    return dict(zip(q.split(","), (x.strip() for x in out.split(",")))) if out else {}


def copy_peak_gbps():
    import torch
    n = 1 << 30
    x = torch.empty(n, dtype=torch.bfloat16, device="cuda")
    y = torch.empty_like(x)
    y.copy_(x)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e30
    for _ in range(10):
        a.record()
        y.copy_(x)
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b))
    del x, y
    torch.cuda.empty_cache()
    return 2 * n * 2 / (best * 1e-3) / 1e9


def sample_state(h, td, idx):
    """harness.State holding elements idx of the handle's mirrors, with td's scalars and the handle's levels."""
    s = harness.State.empty(len(idx), td.nlev, td.qsize_d, td.ntl)
    for k, e in enumerate(idx):
        got = h.download_range(int(e), int(e) + 1, names=harness.FIELD_NAMES)
        for n in harness.FIELD_NAMES:
            s.arrays[n][k] = got[n][0]
    c = h.control
    s.ctl[:] = (0, len(idx), c.n0, c.np1, c.nm1, c.qn0)
    s.dt2, s.consts[:], s.dvv[...], s.ps0, s.hyai[:] = td.dt2, td.consts, td.dvv, td.ps0, td.hyai
    return s


def parity(h, td, hybi, mode, rng):
    idx = np.sort(rng.choice(td.nelem, 64, replace=False))
    want = sample_state(h, td, idx)
    ro.rk5_step(harness.PortOracle(), want, DT, hybi)
    h.run_rk5(1, DT, mode)
    got = sample_state(h, td, idx)
    if mode == tb.MODE_STRICT:
        return {"bit_exact": all(np.array_equal(got.arrays[n], want.arrays[n]) for n in harness.FIELD_NAMES)}
    rel = max(float(np.max(np.abs(got.arrays[n] - want.arrays[n])) / max(float(np.max(np.abs(want.arrays[n]))), 1e-300))
              for n in harness.MUTATED)
    return {"max_rel_err": rel, "ok": rel <= 1e-12}


def timed(h, fn, reps):
    fn()
    h.sync()
    best = 1e30
    for _ in range(3):
        h.timer_start()
        for _ in range(reps):
            fn()
        best = min(best, h.timer_stop() / reps)
    return best


def stage_alone_ms(h, td, mode, reps):
    """Stages 1-5 each on its own (caar_run with the stage's levels, dt2 and eta_ave_w), ms per launch."""
    c = h.control
    n0, np1, nm1 = c.n0, c.np1, c.nm1
    out = []
    for st in ro.schedule(n0, np1, nm1, DT, float(td.consts[1])):
        if st == "combine":
            continue
        consts = td.consts.copy()
        consts[1] = st[4]
        h.set_params(consts, td.dvv, td.ps0, td.hyai)
        h.set_control(n0=st[0], np1=st[1], nm1=st[2], dt2=st[3])
        out.append(timed(h, lambda: h.compute_and_apply_rhs(1, mode, sync=False), reps))
    h.set_params(td.consts, td.dvv, td.ps0, td.hyai)
    h.set_control(n0=n0, np1=np1, nm1=nm1, dt2=td.dt2)
    return out


def profiled_kernel_ms(h, mode, steps):
    """Kernel time of each of the six launches of a step, from torch.profiler over `steps` steps (None if the capture
    holds no kernels)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.run_rk5(steps, DT, mode)
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                 and ("caar_" in e.name or "combine_kernel" in e.name)), key=lambda e: e.time_range.start)
    if len(ev) != 6 * steps:
        return None, [e.name for e in ev[:8]]
    per = [sum(ev[6 * s + k].time_range.elapsed_us() for s in range(steps)) / steps / 1e3 for k in range(6)]
    return per, sorted({e.name.split("(")[0] for e in ev})


def check_finite(h, E, where):
    """Stops the run when the state is no longer finite: checksums of every time level."""
    for tl in range(3):
        ck = h.checksums(tl, 0, E)
        if not (np.isfinite(ck["sum"]).all() and np.isfinite(ck["sumsq"]).all()):
            raise SystemExit(f"{where}: time level {tl} is not finite")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="86400x72,49152x128,51840x30,21600x72e")
    ap.add_argument("--modes", default="fast,strict")
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    info = gpu_info()
    peak = copy_peak_gbps()
    rng = np.random.default_rng(2026)
    for cfg in args.configs.split(","):
        eulerian = cfg.endswith("e")
        E, L = (int(x) for x in cfg.rstrip("e").split("x"))
        td = TestData(E, L).init_data()
        td.arrays["elem_spheremp"][...] = 1.0
        hybi = np.linspace(0.0, 1.0, L + 1) if eulerian else None
        h = tb.Caar(E, L)
        h.set_params(td.consts, td.dvv, td.ps0, td.hyai)
        if eulerian:
            h.set_vertical_coordinate(0, hybi)
        lf = E * L * 16 * 8
        stage_bytes = [LF_STAGE1 * lf + GEO * E] + [LF_STAGE * lf + GEO * E] * 4   # stages 1-5
        comb_bytes = LF_COMBINE * lf
        step_bytes = sum(stage_bytes) + comb_bytes
        for mode_name in args.modes.split(","):
            mode = tb.MODE_FAST if mode_name == "fast" else tb.MODE_STRICT
            h.set_control(0, E, 0, 1, 2, 0, dt2=td.dt2)
            h.upload(td.arrays)           # each mode starts from the initial state
            par = parity(h, td, hybi, mode, rng)
            ms = timed(h, lambda: h.run_rk5(args.steps, DT, mode, sync=False), 1) / args.steps
            prof, names = profiled_kernel_ms(h, mode, args.steps)
            comb = prof[4] if prof else None   # launch order: stages 1-4, combination, stage 5
            check_finite(h, E, f"{cfg} {mode_name} after the timed steps")
            h.set_control(0, E, 0, 1, 2, 0, dt2=td.dt2)
            h.upload(td.arrays)
            alone = stage_alone_ms(h, td, mode, args.steps)
            check_finite(h, E, f"{cfg} {mode_name} after the stages alone")
            alias_ms = sum(alone[2:5])
            rec = {
                "config": cfg, "nelem": E, "nlev": L, "branch": "eulerian" if eulerian else "lagrangian",
                "mode": mode_name, "kernel": h.describe(mode)[0], "steps": args.steps, "dt": DT,
                "ms_per_step": round(ms, 4),
                "elem_lev_stage_updates_per_s": round(E * L * 5 / (ms * 1e-3), 1),
                "bytes_per_step": step_bytes, "GBps": round(step_bytes / (ms * 1e-3) / 1e9, 1),
                "copy_peak_GBps": round(peak, 1), "frac_copy_peak": round(step_bytes / (ms * 1e-3) / 1e9 / peak, 4),
                "byte_bound_ms": round(step_bytes / (peak * 1e9) * 1e3, 3),
                "stage_ms": {"alone": {f"stage{k + 1}": round(t, 4) for k, t in enumerate(alone)},
                             "combine_kernel": round(comb, 4) if comb is not None else None,
                             "in_step_kernels": [round(t, 4) for t in prof] if prof else None},
                "sum_of_parts_ms": round(sum(alone) + comb, 4) if comb is not None else None,
                "stage_GBps_alone": [round(b / (t * 1e-3) / 1e9, 1) for b, t in zip(stage_bytes, alone)],
                "combine_GBps": round(comb_bytes / (comb * 1e-3) / 1e9, 1) if comb else None,
                "aliased_stages_3to5_ms": round(alias_ms, 4),
                "aliased_GBps": round(sum(stage_bytes[2:5]) / (alias_ms * 1e-3) / 1e9, 1),
                "profiled_kernels": names, "parity_64": par, "gpu": info,
            }
            print(json.dumps(rec), flush=True)
        h.close()


if __name__ == "__main__":
    main()
