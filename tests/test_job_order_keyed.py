"""Host-only check of the keyed job order of the allocate action (csrc/kai_job_order.cuh): on seeded two- and
three-level queue trees it pops the same job sequence as the replica job-order tree (csrc/kai_seq.cuh), and its
eligibility check refuses the snapshots where the two could differ.  Compiled with nvcc as host code."""
import os
import shutil
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")
def test_keyed_order_equals_replica_and_rejects_ties():
    src = os.path.join(ROOT, "tests", "native", "job_order_check.cu")
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "check")
        subprocess.check_call(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                               "-Xcompiler", "-ffp-contract=off", "-x", "cu", "-o", exe, src],
                              stdout=subprocess.DEVNULL)
        out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.startswith("OK")
