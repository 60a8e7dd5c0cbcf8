#!/usr/bin/env python
"""bench.py — compute_and_apply_rhs element·level updates per second on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the reference's own CPU implementation on the host cores
    python bench.py ... --dump-outputs DIR   # also write the arrays of the last timed step as DIR/<name>.npy

A "step" = one compute_and_apply_rhs over every element this job holds. Workload = BASELINE configs[3]:
ne=120 cubed sphere (86400 elements), np=4, nlev=72, FP64 — per GPU (weak scaling: the element loop has no
inter-element coupling, each rank owns a contiguous element range, no collective in the timed loop; NCCL is
used only for the max-over-ranks time and the final all-reduce of the squared norms).

One JSON line on stdout (rank 0). `value` = whole-job updates/s with state resident in HBM (CUDA events on
the launching stream); `e2e` = the same through the reference-facing host call (pinned host arrays, H2D of
inputs and D2H of results inside the timed region); `roofline` = achieved algorithmic HBM GB/s of the fused
kernel against the measured copy peak; `cpu_baseline` = the reference CPU build on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree (which may be read-only)

METRIC = "compute_and_apply_rhs_elem_lev_updates_per_s"
UNIT = "elem*lev updates/s"
NE120 = 86400
# (elements, nlev) of the BASELINE.json configs, for the workload label
WORKLOADS = {(5400, 72): "ne=30", (86400, 72): "ne=120", (393216, 128): "ne=256", (49152, 128): "ne=256 / 8"}


def b_alg(nlev: int) -> float:
    """Algorithmic (compulsory) HBM bytes per element·level, SURVEY.md §8(d)/DESIGN.md: 13 level-fields read
    + 8 written (21 x 128 B) + 1664 B of per-element 2-D geometry amortised over the levels."""
    return 21 * 128.0 + 1664.0 / nlev


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_per_launch(nelem, nlev, eulerian=False):
    """dram bytes per launch of the fused kernel from the committed ncu --set full capture, scaled to this
    launch's element count (traffic is linear in elements); None until a capture exists."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))["by_nlev_eulerian" if eulerian else "by_nlev"][str(nlev)]
        return float(t["dram_bytes_per_elem"]) * nelem
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe) through NVML
    (the library behind nvidia-smi) from a background thread every few milliseconds — the timed region of the
    default run lasts ~60 ms, too short for `nvidia-smi -lms`."""

    def __init__(self, gpu_index, period_s=0.002):
        import threading
        self.samples, self.reasons, self.max_mhz, self.power = [], set(), None, []
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES if it is a plain list of ordinals
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = gpu_index
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                phys = int(vis.split(",")[gpu_index])
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.period = period_s
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def _run(self):
        nv = self.nv
        names = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
                 ("sw_power_cap", 0x4))
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.dev, nv.NVML_CLOCK_SM)))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                    nv.nvmlDeviceGetCurrentClocksThrottleReasons
                r = int(get(self.dev))
                for n, bit in names:
                    if r & bit:
                        self.reasons.add(n)
                if len(self.samples) % 8 == 1:      # power is slow to read and slow to change
                    self.power.append(nv.nvmlDeviceGetPowerUsage(self.dev) / 1000.0)
            except Exception:
                pass
            self._stop.wait(self.period)

    extended = False

    def count_since_mark(self):
        return len(self.samples) - getattr(self, "t_mark", 0)

    def mark(self):
        """Samples taken from here on belong to the timed region (plus the one in flight: the GPU has been under
        the same load for two steps when this is called, and an NVML query takes longer than a step)."""
        self.t_mark = max(0, len(self.samples) - 1)
        self.reasons.clear()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        if self._thread is None:
            return out
        self._stop.set()
        self._thread.join(timeout=2)
        sm = self.samples[getattr(self, "t_mark", 0):]
        if sm:
            out.update(sm_mhz=statistics.median(sm), reasons=sorted(self.reasons), samples=len(sm),
                       power_w_max=max(self.power) if self.power else None,
                       window="timed region" + (" + the same kernel loop continued until 5 samples" if self.extended else ""))
        return out


def bind_to_gpu_numa_node(gpu_index):
    """Pin this process to the CPUs NVML reports as local to its GPU BEFORE the host arrays are allocated and
    first touched, so that the page-locked arrays of the end-to-end leg live on the GPU's NUMA node (what a
    launcher would do with numactl). Returns the number of CPUs bound to, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        phys = gpu_index
        if vis and all(x.strip().isdigit() for x in vis.split(",")):
            phys = int(vis.split(",")[gpu_index])
        dev = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = pynvml.nvmlDeviceGetCpuAffinity(dev, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def randomize_like_reference_bench(td, seed):
    """Fields U(1/64, 1), D random with |det D| >= 1/64, Dinv = D^-1, metdet = |det D| — the recipe of the reference's
    Kokkos bench (level_vectorized_ppscan/Elements.cpp:101-152), which seeds from std::random_device; here a fixed
    seed (numpy PCG64, so the values are not those of any mt19937_64 run). dp3d stays positive by construction."""
    rng = np.random.default_rng(seed)
    A = td.arrays
    for n, a in A.items():
        if n in ("elem_D", "elem_Dinv", "elem_metdet", "elem_rmetdet"):
            continue
        a[...] = rng.uniform(1.0 / 64, 1.0, size=a.shape)
    D = rng.uniform(1.0 / 64, 1.0, size=A["elem_D"].shape)
    det = D[..., 0, 0] * D[..., 1, 1] - D[..., 0, 1] * D[..., 1, 0]
    bad = np.abs(det) < 1.0 / 64
    D[bad] = np.array([[1.0, 0.25], [0.125, 0.75]])
    det = D[..., 0, 0] * D[..., 1, 1] - D[..., 0, 1] * D[..., 1, 0]
    A["elem_D"][...] = D
    A["elem_Dinv"][..., 0, 0] = D[..., 1, 1] / det
    A["elem_Dinv"][..., 0, 1] = -D[..., 0, 1] / det
    A["elem_Dinv"][..., 1, 0] = -D[..., 1, 0] / det
    A["elem_Dinv"][..., 1, 1] = D[..., 0, 0] / det
    A["elem_metdet"][...] = np.abs(det)
    A["elem_rmetdet"][...] = 1.0 / np.abs(det)


def cpu_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_reference_rate(nlev, target_s=15.0, threads=None, calls=None):
    """The reference's own CPU implementation (oracle/_ref when built from /root/reference, else the C port)
    on `threads` host threads over a bounded sample: 256 elements per thread, enough calls for ~target_s."""
    from oracle import harness
    orc = harness.best_oracle(nlev)
    threads = threads or cpu_threads()
    E = 256 * threads
    s = orc.init(E, nlev)
    t1 = orc.run(s, 1, threads)                       # also warms the pages
    if calls is None:
        calls = max(1, min(5000, int(target_s / max(t1, 1e-6))))
    t = orc.run(s, calls, threads)
    rate = E * nlev * calls / t
    sample = (f"{E} elements (256 per thread) x {calls} calls, nlev={nlev}, closed-form init, "
              f"{threads} threads on disjoint [nets,nete) ranges, wall clock {t:.2f}s")
    return rate, orc.kind, threads, sample, t / calls


def run_reference_arm(args):
    """The reference's own CPU implementation (oracle/_ref: the unmodified pointers_only sources) on every host
    thread, one unmodified routine per disjoint [nets,nete) range, over the FULL per-GPU workload of the b200 arm
    (--nelem elements, default ne=120: 86400) — one call per step, like PO/main.cpp:113-121."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = cpu_threads()
    from oracle import harness
    orc = harness.best_oracle(args.nlev)
    E = args.nelem
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 1 << 62
    need = E * (186112.0 / 72 * args.nlev)
    sampled = need > 0.6 * avail
    if sampled:                                   # never on the pool's boxes; keeps the arm alive on a small host
        E = max(threads, int(0.5 * avail / (186112.0 / 72 * args.nlev)) // threads * threads)
    s = orc.init(E, args.nlev)
    for _ in range(max(1, args.warmup)):
        orc.run(s, 1, threads)
    steps = args.steps
    t0 = time.perf_counter()
    total = 0.0
    for _ in range(steps):
        total += orc.run(s, 1, threads)
    wall = time.perf_counter() - t0
    rate = E * args.nlev * steps / total
    sample = (f"{E} elements x 1 call per step, nlev={args.nlev}, closed-form init, {threads} threads on disjoint "
              f"[nets,nete) ranges" + ("; SUB-SAMPLED: the host cannot hold the full arrays" if sampled else
                                       "; the full per-GPU workload of the b200 arm"))
    if args.gpus > 1:
        sample += (f"; the b200 arm at {args.gpus} GPUs holds {args.gpus} x {args.nelem} elements — the CPU rate is "
                   f"per unit of work and does not depend on the element count")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic (reference closed-form init)",
        "config": {"workload": f"{WORKLOADS.get((args.nelem, args.nlev), 'cubed sphere')}: {args.nelem} elements per GPU, "
                               f"np=4, nlev={args.nlev}, FP64, n0/np1/nm1 distinct, qn0=0",
                   "elements_per_gpu": args.nelem, "nlev": args.nlev, "sampled": sampled, "elements_timed": E},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": orc.kind, "sample": sample,
                         "cpu_model": cpu_model()},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---- correctness attached to the speed records -------------------------------------------------------------------
def sample_windows(E, seed):
    """first / middle / last 16 elements + 16 random single elements of a rank's slice (fewer on tiny slices)"""
    if E <= 64:
        return [(0, E)]
    rng = np.random.default_rng(seed)
    mid = E // 2
    w = [(0, 16), (mid - 8, mid + 8), (E - 16, E)]
    w += [(int(e), int(e) + 1) for e in sorted(rng.choice(np.arange(16, E - 16), size=16, replace=False))]
    return w


def oracle_states(td, windows, nlev):
    """harness.State copies of the window elements of td (the inputs as they are in the host arrays right now)"""
    from oracle import harness
    out = []
    for (a, b) in windows:
        st = harness.State(b - a, nlev)
        st.arrays = {n: td.arrays[n][a:b].copy() for n in harness.FIELD_NAMES}
        st.ctl = np.array([0, b - a] + [int(x) for x in td.ctl[2:6]], dtype=np.int32)
        st.dt2, st.consts, st.dvv, st.ps0, st.hyai = td.dt2, td.consts.copy(), td.dvv.copy(), td.ps0, td.hyai.copy()
        out.append(st)
    return out


def max_rel_err(got, want, names):
    worst = 0.0
    for n in names:
        den = max(float(np.max(np.abs(want[n]))), 1e-300)
        worst = max(worst, float(np.max(np.abs(got[n] - want[n]))) / den)
    return worst


def max_pointwise_rel_err(got, want, names):
    """max over points of |a-b| / |b| (points with |b| below 1e-30 of the field maximum skipped): reported, not gated —
    a cancelling field like omega_p shows a scan-carry regression here long before it reaches 1e-12 of the maximum."""
    worst, where = 0.0, None
    for n in names:
        b = want[n]
        floor = 1e-30 * max(float(np.max(np.abs(b))), 1e-300)
        mask = np.abs(b) > floor
        if not mask.any():
            continue
        e = float(np.max(np.abs(got[n][mask] - b[mask]) / np.abs(b[mask])))
        if e > worst:
            worst, where = e, n
    return worst, where


DUMP_BYTES = 64_000_000
DUMP_SEED = 20261020


def dump_elements(E, L):
    """The elements --dump-outputs writes: all E when the seven mutated arrays of all of them fit DUMP_BYTES, else a
    sample drawn with a fixed seed, in index order. Depends on (E, L) only, so two runs with the same arguments dump
    the same elements."""
    from tinman_sandbox_b200 import MUTATED_FIELDS, field_shape
    per_elem = 8 * sum(int(np.prod(field_shape(n, 1, L))) for n in MUTATED_FIELDS)
    n = (DUMP_BYTES - 4096) // per_elem                 # 4096: room for the .npy headers
    if E <= n:
        return np.arange(E)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(E, size=n, replace=False))


def dump_outputs(h, E, L, out_dir):
    """DIR/<name>.npy (float64) for each array the routine mutates, every time level, as a caller downloading from the
    handle receives them, restricted to dump_elements(E, L)."""
    from tinman_sandbox_b200 import MUTATED_FIELDS
    elems = dump_elements(E, L)
    runs = np.split(elems, np.flatnonzero(np.diff(elems) != 1) + 1)     # contiguous runs: one download each
    parts = [h.download_range(int(r[0]), int(r[-1]) + 1, names=MUTATED_FIELDS) for r in runs]
    os.makedirs(out_dir, exist_ok=True)
    for n in MUTATED_FIELDS:
        np.save(os.path.join(out_dir, n + ".npy"), np.concatenate([p[n] for p in parts]))


def link_probe(dev, h2d_bytes, d2h_bytes, total=1 << 29, sync=None):
    """What this GPU's host link does right now, in this process (pinned buffers, two streams, best of 4): host->device
    alone, device->host alone, both at once with equal sizes (duplex), and both at once IN THE PROPORTION OF ONE e2e
    STEP (h2d_bytes : d2h_bytes) — the time of that last probe, scaled to the step's bytes, is the link-bound time of a
    step and the denominator of the end-to-end number."""
    import torch
    n_in = int(total * h2d_bytes / float(h2d_bytes + d2h_bytes)) // 4096 * 4096
    n_out = int(total * d2h_bytes / float(h2d_bytes + d2h_bytes)) // 4096 * 4096
    nmax = max(n_in, n_out, total // 2)
    hin = torch.empty(nmax, dtype=torch.uint8, pin_memory=True)
    hout = torch.empty(nmax, dtype=torch.uint8, pin_memory=True)
    din = torch.empty(nmax, dtype=torch.uint8, device=dev)
    dout = torch.empty(nmax, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    res = {}
    half = total // 2
    for name, bi, bo in (("h2d", half, 0), ("d2h", 0, half), ("duplex", half, half), ("step_mix", n_in, n_out)):
        best = 1e30
        for _ in range(4):
            torch.cuda.synchronize(dev)
            if sync is not None:
                sync()                               # every rank runs the SAME probe at the same time
            t0 = time.perf_counter()
            if bi:
                with torch.cuda.stream(s1):
                    din[:bi].copy_(hin[:bi], non_blocking=True)
            if bo:
                with torch.cuda.stream(s2):
                    hout[:bo].copy_(dout[:bo], non_blocking=True)
            torch.cuda.synchronize(dev)
            best = min(best, time.perf_counter() - t0)
        res[name] = max(bi, bo) / best / 1e9 if name != "step_mix" else best
    res["step_mix_h2d_bytes"] = n_in
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nelem", type=int, default=NE120, help="elements per GPU (default ne=120: 86400)")
    ap.add_argument("--nlev", type=int, default=72)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --nelem elements per GPU (default); strong: --nelem elements in total, cut into "
                         "contiguous blocks per rank (BASELINE configs[3]/[4] strong-scaling variants)")
    ap.add_argument("--mode", default="fast", choices=["fast", "strict"])
    ap.add_argument("--data", default="closed-form", choices=["closed-form", "random"],
                    help="closed-form: the reference's init (PO/data_structures.cpp:38-92); random: U(1/64,1) fields and a "
                         "random D with |det| >= 1/64, Dinv = D^-1 (the recipe of LV/Elements.cpp:101-152, fixed seed)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-chunk", type=int, default=0, help="elements per pipeline chunk (0 = automatic)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-target-s", type=float, default=15.0)
    ap.add_argument("--eulerian", action="store_true",
                    help="rsplit == 0: the Eulerian vertical coordinate (SURVEY 8f rank 3) instead of the reference's "
                         "vertically Lagrangian path; hybi = linspace(0,1); the checker is then the CPU restatement")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled oracle check after the timed loops")
    ap.add_argument("--no-clock-topup", action="store_true",
                    help="do not continue the kernel loop after a short timed region to collect 5 clock samples (keeps the "
                         "number of calls, hence the accumulators and their checksums, deterministic)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the arrays the routine mutates, as they stand after the last timed "
                         "step, to DIR/<name>.npy (float64, rank 0's slice; a fixed sample of elements when the slice "
                         f"would take more than {DUMP_BYTES // 10**6} MB). Inputs depend only on the arguments, so runs "
                         "of two builds can be compared array by array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = max(args.warmup, 1)

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    import tinman_sandbox_b200 as tb
    from tinman_sandbox_b200.testdata import TestData

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    L = args.nlev
    if args.scaling == "strong":
        from tinman_sandbox_b200.partition import element_range
        lo, hi = element_range(rank, world, args.nelem)
        E, elem_offset, E_total = hi - lo, lo, args.nelem
    else:
        E, elem_offset, E_total = args.nelem, rank * args.nelem, world * args.nelem
    mode = tb.MODE_FAST if args.mode == "fast" else tb.MODE_STRICT

    # ---- synthetic inputs: the reference's closed-form init for this rank's element range, in pinned memory
    pinned = []

    def alloc(shape):
        n = int(np.prod(shape))
        try:
            t = torch.empty(n, dtype=torch.float64, pin_memory=True)
        except Exception:
            t = torch.empty(n, dtype=torch.float64)
        pinned.append(t)
        return t.numpy().reshape(shape)

    # page-locking world x 16 GB must not exhaust the box: fall back to pageable host arrays (and say so) if it would
    try:
        import psutil
        host_total = psutil.virtual_memory().total
    except Exception:
        host_total = 0
    host_need = world * E * (186112.0 / 72 * L)
    pin_ok = host_total == 0 or host_need < 0.6 * host_total
    if not pin_ok:
        def alloc(shape):  # noqa: F811
            return np.zeros(shape, dtype=np.float64)
    td = TestData(E, L, alloc=alloc).init_data(elem_offset=elem_offset)
    if args.data == "random":
        randomize_like_reference_bench(td, seed=20261018 + rank)
    h = tb.Caar(E, L, device=local_rank)
    h.set_params(td.consts, td.dvv, td.ps0, td.hyai)
    h.set_control(*[int(x) for x in td.ctl], dt2=td.dt2)
    hybi = np.linspace(0.0, 1.0, L + 1)
    if args.eulerian:
        h.set_vertical_coordinate(0, hybi)
    h.upload(td.arrays)

    def oracle_run(orc_, st_, calls, threads):
        return orc_.run_eulerian(st_, hybi, calls, threads) if args.eulerian else orc_.run(st_, calls, threads)

    # ---- resident-state throughput: W warm-up steps, then exactly K steps between CUDA events
    h.compute_and_apply_rhs(args.warmup, mode)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    h.compute_and_apply_rhs(2, mode)       # the sampler thread is running: put the GPU under load, then mark
    barrier()
    if sampler:
        sampler.mark()
    launches0 = h.launch_count()
    h.timer_start()
    h.compute_and_apply_rhs(args.steps, mode, sync=False)
    ms = h.timer_stop()
    barrier()
    launches = h.launch_count() - launches0
    calls_done = args.warmup + 2 + args.steps
    if args.dump_outputs and rank == 0:       # before anything below runs more calls
        dump_outputs(h, E, L, args.dump_outputs)
    # A timed region shorter than ~5 NVML samples (small or strong-scaled slices): keep the SAME load running, outside
    # the timed region, until the sampler has at least 5 — and say so; never print a clocks record with fewer.
    if sampler and sampler.count_since_mark() < 5 and not args.no_clock_topup:
        t_end = time.perf_counter() + 2.0
        batch = max(args.steps, int(0.02 / max(ms / args.steps * 1e-3, 1e-6)))   # >= 20 ms of the same kernel per sync
        extra_cap = 500                       # the accumulators are compared with the oracle after the same number of calls
        while sampler.count_since_mark() < 5 and time.perf_counter() < t_end and extra_cap > 0:
            batch = min(batch, extra_cap)
            h.compute_and_apply_rhs(batch, mode)
            calls_done += batch
            extra_cap -= batch
        sampler.extended = True
    barrier()
    clocks = sampler.stop() if sampler else None
    if clocks and clocks.get("samples", 0) < 5:
        clocks = {"sm_mhz": None, "sm_max_mhz": clocks.get("sm_max_mhz"), "reasons": [], "samples": clocks.get("samples", 0),
                  "rejected": "fewer than 5 NVML samples under load"}
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    ms_per_step = ms_max / args.steps
    value = E_total * L * args.steps / (ms_max * 1e-3)

    # ---- the collectives of the job, all AFTER the timed loop (NCCL over NVLink): squared norms of v, T, dp3d(np1)
    # (print_results_2norm, PO/compute_and_apply_rhs.cpp:372-399), checksums of all seven mutated arrays and the two
    # energy norms (caar_checksums), summed over ranks; the bit-pattern sums travel as 64-bit integers.
    ss_local = h.sumsq(int(td.ctl[3]))
    ss = torch.from_numpy(ss_local).to(dev)
    cs = h.checksums(int(td.ctl[3]))
    cs_f = torch.from_numpy(np.concatenate([cs["sum"], cs["sumsq"], cs["energy"]])).to(dev)
    cs_b = torch.from_numpy(cs["bits"].view(np.int64).copy()).to(dev)
    if world > 1:
        dist.all_reduce(ss, op=dist.ReduceOp.SUM)
        dist.all_reduce(cs_f, op=dist.ReduceOp.SUM)
        dist.all_reduce(cs_b, op=dist.ReduceOp.SUM)
    norms = torch.sqrt(ss).cpu().numpy().tolist()
    cs_f = cs_f.cpu().numpy()
    checksums = {"fields": list(tb.CHECKSUM_FIELDS), "sum": cs_f[:7].tolist(), "sumsq": cs_f[7:14].tolist(),
                 "energy": {"kinetic": float(cs_f[14]), "internal": float(cs_f[15])},
                 "bits": [format(int(x) & 0xFFFFFFFFFFFFFFFF, "016x") for x in cs_b.cpu().numpy()],
                 "time_level": int(td.ctl[3]), "calls": calls_done}

    # ---- parity of THIS run: a sample of this rank's slice against the CPU oracle after the same number of calls
    parity = None
    if not args.no_parity:
        from oracle import harness
        orc = harness.PortOracle() if args.eulerian else harness.best_oracle(L)   # the reference has no rsplit == 0 branch
        wins = sample_windows(E, seed=1000 + rank)
        states = oracle_states(td, wins, L)          # td still holds the inputs: nothing has written the host arrays
        worst, nchk, pw, pw_field = 0.0, 0, 0.0, None
        for (a, b), st in zip(wins, states):
            oracle_run(orc, st, calls_done, 1)
            got = h.download_range(a, b, names=harness.MUTATED)
            worst = max(worst, max_rel_err(got, st.arrays, harness.MUTATED))
            e_pw, f_pw = max_pointwise_rel_err(got, st.arrays, harness.MUTATED)
            if e_pw > pw:
                pw, pw_field = e_pw, f_pw
            nchk += b - a
        parity = {"max_rel_err": worst, "max_pointwise_rel_err": pw, "max_pointwise_field": pw_field,
                  "elements_checked": nchk, "calls": calls_done, "oracle": orc.kind,
                  "tolerance": 0.0 if mode == tb.MODE_STRICT else 1e-12,
                  "what": "first/middle/last 16 + 16 random elements of every rank's slice, all 7 mutated arrays, "
                          "max|a-b|/max|b| per field and window, max over ranks"}

    # ---- end to end through the reference-facing host semantics: host arrays in, host arrays out, per step
    e2e = None
    if not args.no_e2e:
        # every step: caar_run_host = copy-in of the slices the routine reads (pinned host arrays), the kernel,
        # copy-out of the slices it writes, pipelined over element chunks; results are in the host arrays
        h2d, d2h = h.host_traffic(mode)
        e2e_states = None
        if parity is not None:
            e2e_wins = sample_windows(E, seed=2000 + rank)
            e2e_states = oracle_states(td, e2e_wins, L)
        barrier()                                    # every rank probes its link at the same time
        link = link_probe(dev, h2d, d2h, sync=barrier if world > 1 else None)
        h.compute_and_apply_rhs_host(td.arrays, mode, args.e2e_chunk)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            h.compute_and_apply_rhs_host(td.arrays, mode, args.e2e_chunk)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t_e = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        dt = float(t_e.item())
        if e2e_states is not None:                   # the host arrays now hold 1 + e2e_steps calls: check them too
            from oracle import harness
            worst = 0.0
            for (a, b), st in zip(e2e_wins, e2e_states):
                oracle_run(orc, st, 1 + args.e2e_steps, 1)
                worst = max(worst, max_rel_err({n: td.arrays[n][a:b] for n in harness.MUTATED}, st.arrays, harness.MUTATED))
            parity["e2e_max_rel_err"] = worst
            parity["e2e_calls"] = 1 + args.e2e_steps
        # link-bound time of one step = time of the proportional probe scaled to the step's bytes
        t_link = link["step_mix"] * (h2d / float(link["step_mix_h2d_bytes"]))
        lk = torch.tensor([link["h2d"], link["d2h"], link["duplex"]], dtype=torch.float64, device=dev)
        tl_ = torch.tensor([t_link], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(lk, op=dist.ReduceOp.MIN)       # the slowest rank's link bounds the job
            dist.all_reduce(tl_, op=dist.ReduceOp.MAX)
        lk = lk.cpu().numpy()
        t_link = float(tl_.item())
        h2d_rate = h2d * args.e2e_steps / dt / 1e9
        e2e = {"value": E_total * L * args.e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps,
               "ms_per_step": 1e3 * dt / args.e2e_steps,
               "pcie_gbs": {"h2d": h2d_rate, "d2h": d2h * args.e2e_steps / dt / 1e9},
               "link": {"h2d_gbs": float(lk[0]), "d2h_gbs": float(lk[1]), "duplex_peak_gbs": float(lk[2]),
                        "step_ms_at_link_speed": 1e3 * t_link, "frac": t_link / (dt / args.e2e_steps),
                        "bound": "host link (PCIe) and, with several GPUs, the host's memory system behind it",
                        "how": "pinned copies in this process just before the timed e2e steps, one GPU per rank and all "
                               "ranks at once: each direction alone, both with equal sizes (duplex, GB/s per direction, min "
                               "over ranks), and both in the byte proportion of one e2e step; step_ms_at_link_speed = that "
                               "last probe scaled to the step's bytes (max over ranks); frac = it / the measured step"},
               "how": "caar_run_host per step: host arrays in, host arrays out (%s), copy-in | kernel | "
                      "copy-out pipelined over element chunks; PCIe-bound" %
                      ("pinned" if pin_ok else "PAGEABLE: pinning would take >60% of host RAM")}
    # ---- the protocol the reference driver's loop needs (PO/main.cpp:99-131): init -> [upload once] -> K calls ->
    # [download once] -> norms. An extra number beside e2e (which pays the copies at EVERY call).
    resident = None
    if not args.no_e2e:
        barrier()
        t0 = time.perf_counter()
        h.upload(td.arrays)
        t1 = time.perf_counter()
        h.compute_and_apply_rhs(args.steps, mode)
        t2 = time.perf_counter()
        h.download(td.arrays)
        t3 = time.perf_counter()
        tt = torch.tensor([t3 - t0, t1 - t0, t2 - t1, t3 - t2], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        tt = tt.cpu().numpy()
        resident = {"value": E_total * L * args.steps / float(tt[0]), "unit": UNIT, "steps": args.steps,
                    "upload_s": float(tt[1]), "compute_s": float(tt[2]), "download_s": float(tt[3]),
                    "how": "caar_upload of all 16 arrays once, %d caar_run calls, caar_download of the 7 mutated arrays "
                           "once; wall clock, max over ranks" % args.steps}

    # ---- the printed norms against the reference: one CPU call over this rank's whole slice (T, v, dp3d at np1 do not
    # depend on the number of calls: the reference loop does not rotate time levels, PO/main.cpp:118)
    if parity is not None:
        from oracle import harness
        os.sched_setaffinity(0, all_cpus)
        st = harness.State(E, L)
        st.arrays = td.arrays
        st.ctl = np.array([0, E] + [int(x) for x in td.ctl[2:6]], dtype=np.int32)
        st.dt2, st.consts, st.dvv, st.ps0, st.hyai = td.dt2, td.consts, td.dvv, td.ps0, td.hyai
        oracle_run(orc, st, 1, max(1, cpu_threads() // max(1, world)))
        want = np.array(orc.norms(st)) ** 2
        nerr = torch.tensor([float(np.max(np.abs(ss_local - want) / want))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(nerr, op=dist.ReduceOp.MAX)
        parity["norms_rel_err"] = float(nerr.item())
        pm = torch.tensor([parity["max_rel_err"], parity.get("e2e_max_rel_err", 0.0)], dtype=torch.float64, device=dev)
        pn = torch.tensor([parity["elements_checked"]], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(pm, op=dist.ReduceOp.MAX)
            dist.all_reduce(pn, op=dist.ReduceOp.SUM)
        parity["max_rel_err"] = float(pm[0].item())
        if "e2e_max_rel_err" in parity:
            parity["e2e_max_rel_err"] = float(pm[1].item())
        parity["elements_checked"] = int(pn.item())
        parity["ok"] = bool(parity["max_rel_err"] <= parity["tolerance"] and
                            parity.get("e2e_max_rel_err", 0.0) <= parity["tolerance"] and
                            parity["norms_rel_err"] <= 1e-13)
    h.close()

    # ---- roofline of the dominant (only) kernel of a step
    peak, peak_src = measured_peak_gbs()
    alg_bytes = (b_alg(L) + (256.0 * (L + 1) / L if args.eulerian else 0.0)) * E * L   # + the eta_dot_dpdn read-modify-write
    achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic_per_launch(E, L, args.eulerian), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "frac_of_nominal_8000": achieved / 8000.0,
                "kernel": ("caar_fused_kernel" if mode == tb.MODE_FAST else "caar_strict_kernel") +
                          (" (Eulerian instance, rsplit == 0)" if args.eulerian else ""),
                "note": "the measured peak is a 50/50 read/write copy; this kernel's traffic is 62 % reads, and the "
                        "library's own saxpby (67 % reads) streams 6.6-6.8 TB/s on the same GPUs (profiles/README.md)"}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)       # the CPU baseline uses every host core, not only the GPU's node
        rate, kind, cores, sample, _ = cpu_reference_rate(L, target_s=args.cpu_target_s)
        # BASELINE.md §5 asks for two CPU numbers: the reference as shipped (single-threaded) and all host cores
        rate1, _, _, sample1, _ = cpu_reference_rate(L, target_s=min(5.0, args.cpu_target_s), threads=1)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                        "cpu_model": cpu_model(),
                        "one_core": {"value": rate1, "unit": UNIT, "sample": sample1}}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64",
            "data": "synthetic (reference closed-form init)" if args.data == "closed-form" else
                    "synthetic (random U(1/64,1) fields, random D with |det|>=1/64: LV/Elements.cpp:101-152 recipe)",
            "config": {"workload": f"{WORKLOADS.get((E_total // (world if args.scaling == 'weak' else 1), L), 'cubed sphere')}: "
                                   f"{E} elements per GPU ({E_total} in total), np=4, nlev={L}, FP64, "
                                   f"n0/np1/nm1 distinct, qn0=0",
                       "elements_per_gpu": E, "nlev": L, "mode": args.mode, "host_cpus_bound": numa,
                       "vertical_coordinate": "Eulerian (rsplit == 0)" if args.eulerian else "Lagrangian (the reference's path)",
                       "l2": "inputs (%.1f GB per GPU) far larger than the 126 MB L2; no flush needed" %
                             (sum(a.nbytes for a in td.arrays.values()) / 1e9)},
            "e2e": e2e, "gpu_launches": int(launches * world), "roofline": roofline,
            "cpu_baseline": cpu_baseline, "clocks": clocks, "norms_np1": norms, "checksums": checksums,
            "parity": parity, "resident_protocol": resident,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
