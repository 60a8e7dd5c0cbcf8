#!/usr/bin/env python
"""Times the level-local operators (tracer step, weak-form operators) on resident data.
    python tools/levelop_bench.py [--nelem 21600] [--nlev 72] [--qsize 4] [--steps 10] [--ops euler,divwk,lap,lapt]
Prints one JSON line per operator and mode: updates/s, algorithmic GB/s, fraction of the measured copy peak."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tinman_sandbox_b200 as tb  # noqa: E402
from tinman_sandbox_b200.testdata import TestData  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nelem", type=int, default=21600)
    ap.add_argument("--nlev", type=int, default=72)
    ap.add_argument("--qsize", type=int, default=4)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--ops", default="euler,divwk,lap,lapt")
    ap.add_argument("--modes", default="fast,strict")
    args = ap.parse_args()
    E, L, Q = args.nelem, args.nlev, args.qsize
    peak = 6545.6
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    td = TestData(E, L, qsize_d=Q).init_data()
    td.arrays["elem_state_Qdp"][...] = 1.0 + 0.01 * np.arange(16).reshape(4, 4)
    h = tb.Caar(E, L, Q)
    h.set_params(td.consts, td.dvv, td.ps0, td.hyai)
    h.upload(td.arrays)
    h.upload_vstar(np.ascontiguousarray(td.arrays["elem_derived_vn0"] * 3.0))
    h.upload_extra(tb.X_SCALAR_IN, np.ascontiguousarray(td.arrays["elem_derived_phi"]))
    h.upload_extra(tb.X_TENSORVISC, np.ascontiguousarray(td.arrays["elem_D"]))
    geo = 1408.0
    ops = {"euler": ("euler_step", lambda m: h.euler_step(0, Q, 100.0, m, sync=False), Q, 256.0 + (256.0 + geo / L) / Q),
           "divwk": ("divergence_sphere_wk", lambda m: h.sphere_wk(tb.OP_DIVERGENCE_WK, m, sync=False), 1, 384.0 + 640.0 / L),
           "lap": ("laplace_simple", lambda m: h.sphere_wk(tb.OP_LAPLACE_SIMPLE, m, sync=False), 1, 256.0 + 640.0 / L),
           "lapt": ("laplace_tensor", lambda m: h.sphere_wk(tb.OP_LAPLACE_TENSOR, m, sync=False), 1, 256.0 + 1152.0 / L)}
    for key in args.ops.split(","):
        name, fn, mult, balg = ops[key]
        for mode_name in args.modes.split(","):
            mode = tb.MODE_FAST if mode_name == "fast" else tb.MODE_STRICT
            fn(mode)
            h.sync()
            best = 1e30
            for _ in range(3):
                h.timer_start()
                for _ in range(args.steps):
                    fn(mode)
                best = min(best, h.timer_stop() / args.steps)
            rate = E * L * mult / (best * 1e-3)
            print(json.dumps({"op": name, "mode": mode_name, "nelem": E, "nlev": L, "qsize": Q if key == "euler" else None,
                              "ms": round(best, 4), "Mupdates_per_s": round(rate / 1e6, 1),
                              "B_alg": round(balg, 1), "GBps": round(rate * balg / 1e9, 1),
                              "frac_measured": round(rate * balg / 1e9 / peak, 4)}), flush=True)
    h.close()


if __name__ == "__main__":
    main()
