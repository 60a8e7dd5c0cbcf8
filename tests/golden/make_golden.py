#!/usr/bin/env python
"""tests/golden/make_golden.py — regenerates the committed golden fixtures. All but the last need the
reference's sources (REF below); the fixtures it writes travel with the repo.

  fortran_golden.npz        Ttest / v1test / v2test, the reference's own known-answer vectors
                            (compute_and_apply_rhs_test/fortran/test_mod.F90:8-296, 299-591, 594-886):
                            T, v(:,:,1,:), v(:,:,2,:) at time level np1 of element 1 after
                            compute_and_apply_rhs, 1152 = np*np*nlev values each, stored in Fortran
                            order (i fastest, then j, then k) exactly as main.F90:241-252 reads them.
                            The Fortran driver initialises Dvv from SINGLE-precision literals
                            (main.F90:79-90), so the vectors correspond to Dvv = (double)(float)Dvv.
  pointers_only_stdout.txt  stdout of the unmodified reference driver (pointers_only/main.cpp) built by
                            oracle/Makefile, default config (10 elements, 1 call): the printed-norm KAT.
  ref_outputs_E3.npz        every array the reference routine mutates, for 3 elements of the closed-form
                            init after 1 and after 2 calls (oracle/_ref/libcaar_ref_L72.so), so the GPU
                            tests can check against the REAL reference even if oracle/_ref is absent.
  full_size_digests.json    `make_golden.py --full-size`: sha256 of every mutated array of every window of
                            test_parity_gpu.py::test_full_size_runs_against_the_compiled_reference after 2
                            calls, computed by the CPU restatement (oracle/caar_oracle.c, bit-identical to the
                            reference: tests/test_oracle.py), plus a digest of the inputs. Needs no reference
                            checkout; the closed-form elements 0-2 are checked against ref_outputs_E3.npz first.
"""
import json
import os
import re
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference/compute_and_apply_rhs_test"


def parse_fortran_vectors(path):
    txt = open(path).read()
    out = {}
    for name in ("Ttest", "v1test", "v2test"):
        m = re.search(name + r"\(np\*np\*nlev\)\s*=\s*\(/(.*?)/\)", txt, re.S)
        body = m.group(1)
        vals = re.findall(r"[-+]?\d+\.\d*(?:[dDeE][-+]?\d+)?", body)
        arr = np.array([float(v.replace("d", "e").replace("D", "e")) for v in vals])
        assert arr.size == 4 * 4 * 72, (name, arr.size)
        out[name] = arr
    return out


def main():
    from oracle import harness
    harness.build_ref()
    vec = parse_fortran_vectors(os.path.join(REF, "fortran", "test_mod.F90"))
    np.savez(os.path.join(HERE, "fortran_golden.npz"), **vec)
    exe = os.path.join(ROOT, "oracle", "_ref", "pointers_only")
    txt = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    txt = "\n".join(l for l in txt.splitlines() if "total time" not in l) + "\n"
    open(os.path.join(HERE, "pointers_only_stdout.txt"), "w").write(txt)
    ro = harness.RefOracle(72)
    s = ro.init(3)
    out = {}
    for call in (1, 2):
        ro.run(s, 1, 1)
        for n in harness.MUTATED:
            a = s.arrays[n]
            if n in ("elem_state_dp3d", "elem_state_v", "elem_state_T"):
                a = a[:, int(s.ctl[3])]
            out[f"call{call}_{n}"] = a.copy()
    np.savez_compressed(os.path.join(HERE, "ref_outputs_E3.npz"), **out)
    print("wrote", os.listdir(HERE))


def full_size_digests():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_parity_gpu as T
    from oracle import harness
    orc = harness.PortOracle()
    ref = np.load(os.path.join(HERE, "ref_outputs_E3.npz"))
    out = {}
    for E, L in ((86400, 72), (49152, 128)):
        _, wins, states = T.full_size_inputs(E, L)
        entry = {"inputs": T.inputs_digest(states), "windows": []}
        for (a, b), s in zip(wins, states):
            orc.run(s, 2, 1)
            entry["windows"].append([[a, b], {n: T.digest(s.arrays[n]) for n in harness.MUTATED}])
            if (E, L, a) == (86400, 72, 0):        # closed-form: its first elements are those of ref_outputs_E3
                for n in harness.MUTATED:
                    x = s.arrays[n][:3, int(s.ctl[3])] if n.startswith("elem_state") else s.arrays[n][:3]
                    assert np.array_equal(x, ref[f"call2_{n}"]), n
        out[f"{E}x{L}"] = entry
    with open(os.path.join(HERE, "full_size_digests.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    if "--full-size" in sys.argv:
        full_size_digests()
    else:
        main()
