"""bench.py contract checks that need no GPU: the reference arm (the reference's own CPU code on the host cores)
prints one JSON line with the agreed keys, and non-zero ranks stay silent."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                           "--warmup", "1", "--nelem", "512"], capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_json_line():
    p = _run()
    assert p.returncode == 0, p.stderr
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "compute_and_apply_rhs_elem_lev_updates_per_s"
    assert d["unit"] == "elem*lev updates/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["value"] > 0 and d["steps"] == 1 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["sampled"] is False and d["config"]["elements_timed"] == 512


def test_reference_arm_other_ranks_are_silent():
    p = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_sample_is_fixed_and_fits_the_budget():
    """--dump-outputs writes every element of a small slice and a fixed, sorted sample of a large one, within 64 MB."""
    import numpy as np
    import bench
    import tinman_sandbox_b200 as tb
    for E, L in ((10, 72), (300, 72), (5400, 72), (86400, 72), (49152, 128), (393216, 128), (86400, 26)):
        e = bench.dump_elements(E, L)
        per_elem = 8 * sum(int(np.prod(tb.field_shape(n, 1, L))) for n in tb.MUTATED_FIELDS)
        assert len(e) * per_elem <= 64_000_000 - 4096, (E, L)
        assert e[0] >= 0 and e[-1] < E and np.all(np.diff(e) > 0), (E, L)
        assert np.array_equal(e, bench.dump_elements(E, L))
        if E * per_elem <= 60_000_000:
            assert np.array_equal(e, np.arange(E))
        else:
            assert len(e) > 100


def test_steps_must_be_positive():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert p.returncode != 0 and "--steps" in p.stderr
