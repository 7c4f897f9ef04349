"""Device memory over the life of a handle.

1. A handle frees everything it allocated: a child process takes an engine of 5·10⁴ beads through
   every path that allocates device memory (both exact pair kernels, the cut-off kernels and the cluster
   surrogate, minimisation, MD, the dense and sparse contact maps, the distance map, the mean pair
   distance, the Hilbert points, timed evaluation with the L2 flush), destroys it, and does so three
   times.  Its per-process device memory (nvidia-smi, a read-only query) after the third cycle is that
   after the first: the dense maps alone are 128 and 256 MB, so a buffer left behind would show.
2. Buffers that grow on one handle give the bits of a fresh handle at every size, growing and
   shrinking again."""
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from common import make_case, to_engine

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 50_000

CHILD = r"""
import json, os, subprocess, sys
import numpy as np
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from common import make_case, to_engine

def used_mib():
    out = subprocess.run(["nvidia-smi", "--query-compute-apps=pid,used_memory", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout
    for line in out.splitlines():
        pid, mem = [f.strip() for f in line.split(",")]
        if int(pid) == os.getpid():
            return float(mem.split()[0])
    return None

case = make_case(N, n_chrom=4, seed=11)
bins = (np.arange(N) * 4096 // N).astype(np.int32)
used = []
for cycle in range(3):
    eng = to_engine(case)
    for kernel in (0, 1):                      # Newton-3, gather
        eng.set_pair_kernel(kernel)
        eng.energy_forces()
    eng.set_cutoff(0.3)
    for kernel in (0, 2, 1):                   # Morton warp kernel, CTA-level variant, cell list
        eng.set_pair_kernel(kernel)
        eng.energy_forces()
    eng.set_pair_kernel(0)
    eng.set_chb_surrogate(True)
    eng.energy_forces()
    eng.set_chb_surrogate(False)
    eng.set_cutoff(0.0)
    eng.minimize(tol=10.0, max_iter=20)
    eng.md_configure("langevin", seed=1)
    eng.set_velocities_to_temperature(310.0, seed=2)
    eng.md_run(20)
    eng.contacts(0.2, bins, 4096)
    eng.contacts_sparse(0.2, np.arange(N, dtype=np.int32), N)
    eng.distance_map(bins, 4096)
    eng.mean_pair_distance()
    eng.hilbert_points(6)
    eng.evaluate_timed(2, flush_l2=True)
    eng.close()
    used.append(used_mib())
print(json.dumps(used))
"""


def test_handle_frees_its_device_memory():
    if shutil.which("nvidia-smi") is None:
        pytest.skip("nvidia-smi is not available")
    code = f"ROOT = {ROOT!r}\nN = {N}\n" + CHILD
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout + res.stderr
    used = json.loads(res.stdout.strip().splitlines()[-1])
    if used[0] is None:
        pytest.skip("nvidia-smi does not list this process (separate PID namespace)")
    assert used[2] - used[0] <= 2.0, f"device memory after cycles 1, 2, 3: {used} MiB"


def test_growing_buffers_match_a_fresh_handle():
    case = make_case(20_000, n_chrom=3, seed=5)
    n = case["n"]
    eng = to_engine(case)
    for n_bins in (64, 4096, 64):
        bins = (np.arange(n) * n_bins // n).astype(np.int32)
        with to_engine(case) as ref:
            for got, want in zip(eng.contacts(0.2, bins, n_bins), ref.contacts(0.2, bins, n_bins)):
                assert np.array_equal(got, want)
            for got, want in zip(eng.distance_map(bins, n_bins), ref.distance_map(bins, n_bins)):
                assert np.array_equal(got, want)
    bead_bins = np.arange(n, dtype=np.int32)
    pairs = []
    for rc in (0.12, 0.2, 0.3, 0.12):  # binned contacts (sort keys) grow twice, then shrink below the capacity
        got = eng.contacts_sparse(rc, bead_bins, n)
        with to_engine(case) as ref:
            want = ref.contacts_sparse(rc, bead_bins, n)
        for g, w in zip(got[:3], want[:3]):
            assert g.dtype == w.dtype and np.array_equal(g, w)
        assert got[3] == want[3]
        pairs.append(got[3])
    assert pairs[0] < pairs[1] < pairs[2]
    eng.close()
