#!/usr/bin/env python
"""Times caar_run (resident state, CUDA events on the launching stream).

    python tools/kernel_sweep.py [--nelem 86400] [--nlev 72] [--steps 20] [--warmup 3] [--tag name]
                                 [--host-steps 0] [--chunk 0]

Prints one JSON line per run: updates/s, ms/step, algorithmic GB/s, fraction of the measured copy peak.
A development tool; bench.py is the judged measurement.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nelem", type=int, default=86400)
    ap.add_argument("--nlev", type=int, default=72)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--tag", default="")
    ap.add_argument("--mode", default="fast")
    ap.add_argument("--host-steps", type=int, default=0, help="also time caar_run_host (pinned host arrays)")
    ap.add_argument("--chunk", type=int, nargs="*", default=[0])
    ap.add_argument("--eulerian", action="store_true", help="rsplit == 0 branch")
    ap.add_argument("--random", action="store_true", help="random geometry/fields instead of the closed form")
    ap.add_argument("--variants", nargs="*", default=None, choices=["distinct", "aliased", "dry", "aliased_dry"],  # may repeat
                    help="time the same resident state under several controls, one JSON line each: distinct = n0/np1/nm1 "
                         "= 0/1/2, qn0 = 0 (21 compulsory level-fields); aliased = n0 = np1 = nm1 = 0 (forward Euler / RK "
                         "stage, F/routine_extracted.F90:6-16: the aliased level is read once, 17); dry = qn0 = -1 (no Qdp "
                         "read, 20). spheremp = 1 and dt2 = 1e-9 keep the state finite over the repeated in-place calls")
    args = ap.parse_args()

    import tinman_sandbox_b200 as tb
    from tinman_sandbox_b200.testdata import TestData
    import torch

    E, L = args.nelem, args.nlev
    mode = tb.MODE_FAST if args.mode == "fast" else tb.MODE_STRICT
    pinned = []

    def alloc(shape):
        t = torch.empty(int(np.prod(shape)), dtype=torch.float64, pin_memory=args.host_steps > 0)
        pinned.append(t)
        return t.numpy().reshape(shape)

    td = TestData(E, L, alloc=alloc).init_data()
    if args.random:
        rng = np.random.default_rng(1)
        for n in ("elem_state_dp3d", "elem_state_T", "elem_state_v"):
            td.arrays[n] *= rng.uniform(0.9, 1.1, size=td.arrays[n].shape)
    h = tb.Caar(E, L)
    h.set_params(td.consts, td.dvv, td.ps0, td.hyai)
    dt2 = td.dt2
    if args.variants:
        dt2 = 1e-9
        td.arrays["elem_spheremp"][...] = 1.0
    h.set_control(*[int(x) for x in td.ctl], dt2=dt2)
    if args.eulerian:
        h.set_vertical_coordinate(0, np.linspace(0.0, 1.0, L + 1))
    h.upload(td.arrays)
    peak = 6545.6
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    def sm_clock():  # SM clock and throttle reasons right after a timed loop (NVML); None without pynvml
        try:
            import pynvml
            pynvml.nvmlInit()
            d = pynvml.nvmlDeviceGetHandleByIndex(0)
            return {"sm_mhz": pynvml.nvmlDeviceGetClockInfo(d, pynvml.NVML_CLOCK_SM),
                    "reasons": hex(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(d))}
        except Exception:
            return None

    for variant in (args.variants or ["distinct"]):
        aliased, dry = variant.startswith("aliased"), variant.endswith("dry")
        if args.variants:
            h.set_control(n0=0, np1=0 if aliased else 1, nm1=0 if aliased else 2, qn0=-1 if dry else 0)
        h.compute_and_apply_rhs(args.warmup, mode)
        best = 1e30
        for _ in range(args.repeat):
            h.timer_start()
            h.compute_and_apply_rhs(args.steps, mode, sync=False)
            best = min(best, h.timer_stop() / args.steps)
        clk = sm_clock()
        # compulsory level-fields (SURVEY 8d): 13 read + 8 written; an aliased nm1 = n0 is read once (-4), dry reads no Qdp (-1)
        fields = 21 - (4 if aliased else 0) - (1 if dry else 0)
        balg = fields * 128.0 + 1664.0 / L + (256.0 * (L + 1) / L if args.eulerian else 0.0)
        rate = E * L / (best * 1e-3)
        out = {"tag": args.tag, "nelem": E, "nlev": L, "mode": args.mode,
               "variant": variant, "eulerian": bool(args.eulerian), "B_alg": round(balg, 1),
               "ms_per_step": round(best, 4), "Mupdates_per_s": round(rate / 1e6, 1),
               "GBps": round(rate * balg / 1e9, 1), "frac_measured": round(rate * balg / 1e9 / peak, 4),
               "clock_after": clk}
        print(json.dumps(out), flush=True)
    if args.host_steps > 0:
        h2d, d2h = h.host_traffic(mode)
        for chunk in args.chunk:
            h.compute_and_apply_rhs_host(td.arrays, mode, chunk)
            t0 = time.perf_counter()
            for _ in range(args.host_steps):
                h.compute_and_apply_rhs_host(td.arrays, mode, chunk)
            dt = (time.perf_counter() - t0) / args.host_steps
            print(json.dumps({"tag": args.tag, "host_call": True, "chunk": chunk, "ms_per_step": round(dt * 1e3, 2),
                              "Mupdates_per_s": round(E * L / dt / 1e6, 2), "h2d_GBps": round(h2d / dt / 1e9, 2),
                              "d2h_GBps": round(d2h / dt / 1e9, 2)}), flush=True)
    h.close()


if __name__ == "__main__":
    main()
