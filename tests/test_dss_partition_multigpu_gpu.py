"""partition.halo_exchange across two ranks of a torch.distributed job over NCCL (skipped on a one-GPU box): each rank
holds one block of a permuted ne = 4 sphere on its own GPU, assembles dp3d, v, T and Qdp with the exchanged DSS and
widens its limiter bounds with the exchanged neighbor_minmax, and writes its slice to a temporary directory. The
slices concatenate to exactly the result of one handle that holds the whole mesh."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import tinman_sandbox_b200 as tb
import dss_oracle as do

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E, L, QD, NTL, QS = 96, 30, 3, 2, 2
PS = [0, 37, 96]
NAMES = tuple(tb.DSS_FIELDS)

WORKER = r'''
import os, sys
root, out = sys.argv[1], sys.argv[2]
sys.path[:0] = [root, os.path.join(root, "tests")]
import numpy as np
import torch
import torch.distributed as dist
import tinman_sandbox_b200 as tb
from tinman_sandbox_b200 import partition
import test_dss_partition_multigpu_gpu as t

dist.init_process_group("nccl")
r = dist.get_rank()
torch.cuda.set_device(r)
gid, inp, bounds = t.inputs()
e0, e1 = t.PS[r], t.PS[r + 1]
h = tb.Caar(e1 - e0, t.L, t.QD, t.NTL, device=r)
h.upload({n: np.ascontiguousarray(a[e0:e1]) for n, a in inp.items()}, names=tuple(inp))
h.upload_bounds(np.ascontiguousarray(bounds[e0:e1]))
h.set_partition(gid, t.PS, r)
partition.halo_exchange(h, tb.HALO_DSS, t.NAMES, t.QS, tl=1, qtl=1, weighting=tb.DSS_PROJECT)
partition.halo_exchange(h, tb.HALO_MINMAX, (), t.QS)
h.sync()
res = {n: np.empty(tb.field_shape(n, e1 - e0, t.L, t.QD, t.NTL)) for n in t.NAMES}
h.download(res, names=t.NAMES)
res["bounds"] = h.download_bounds()
np.savez(os.path.join(out, f"rank{r}.npz"), **res)
h.close()
dist.destroy_process_group()
'''


def inputs():
    rng = np.random.default_rng(77)
    gid = do.cubed_sphere_gid(4, rng)
    inp = {"elem_spheremp": rng.uniform(0.5, 2.0, (E, 4, 4))}
    for n in NAMES:
        inp[n] = rng.uniform(1.0, 3.0, tb.field_shape(n, E, L, QD, NTL))
    bounds = np.sort(rng.standard_normal((E, QD, L, 2)), -1)
    return gid, inp, bounds


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_two_ranks_concatenate_to_one_handle(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    worker = tmp_path / "worker.py"
    worker.write_text(WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), str(worker), ROOT, str(tmp_path)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    ranks = [np.load(tmp_path / f"rank{r}.npz") for r in range(2)]
    gid, inp, bounds = inputs()
    h = tb.Caar(E, L, QD, NTL)
    h.upload(inp, names=tuple(inp))
    h.upload_bounds(np.ascontiguousarray(bounds))
    h.set_connectivity(gid)
    h.dss(NAMES, tl=1, qtl=1, qsize=QS, weighting=tb.DSS_PROJECT)
    h.neighbor_minmax(QS)
    want = {n: np.empty(tb.field_shape(n, E, L, QD, NTL)) for n in NAMES}
    h.download(want, names=NAMES)
    want["bounds"] = h.download_bounds()
    h.close()
    for n in want:
        got = np.concatenate([r[n] for r in ranks])
        assert np.array_equal(got.view(np.uint64), want[n].view(np.uint64)), n
