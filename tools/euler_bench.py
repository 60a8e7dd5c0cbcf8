#!/usr/bin/env python
"""Times caar_euler_step (tracer RHS after CAAR) on resident data: updates = elements x levels x tracers.
    python tools/euler_bench.py [--nelem 21600] [--nlev 72] [--qsize 4] [--steps 10]"""
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
    ap.add_argument("--lib", default=None)
    args = ap.parse_args()
    if args.lib:
        from tinman_sandbox_b200 import capi
        path = os.path.abspath(args.lib)
        capi.lib_path = lambda: path
    E, L, Q = args.nelem, args.nlev, args.qsize
    td = TestData(E, L, qsize_d=Q).init_data()
    td.arrays["elem_state_Qdp"][...] = 1.0 + 0.01 * np.arange(16).reshape(4, 4)
    h = tb.Caar(E, L, Q)
    h.set_params(td.consts, td.dvv, td.ps0, td.hyai)
    h.upload(td.arrays)
    h.upload_vstar(np.ascontiguousarray(td.arrays["elem_derived_vn0"] * 3.0))
    for mode, name, kernel in ((tb.MODE_FAST, "fast", "levelop_kernel<OP_EULER>"),
                               (tb.MODE_STRICT, "strict", "euler_step_kernel")):
        h.euler_step(0, Q, 100.0, mode)
        h.timer_start()
        for _ in range(args.steps):
            h.euler_step(0, Q, 100.0, mode, sync=False)
        ms = h.timer_stop() / args.steps
        balg = 256.0 + (256.0 + 1408.0 / L) / Q
        rate = E * L * Q / (ms * 1e-3)
        print(json.dumps({"kernel": kernel, "mode": name, "nelem": E, "nlev": L, "qsize": Q,
                          "ms": round(ms, 4), "Mupdates_per_s": round(rate / 1e6, 1),
                          "GBps": round(rate * balg / 1e9, 1), "frac_measured": round(rate * balg / 1e9 / 6545.6, 4)}))
    h.close()


if __name__ == "__main__":
    main()
