"""OT-target global fits (PairSynthesizer(targets="ot")) on N GPUs of one node (torchrun, one process per GPU): sharded
granules with one rank holding none, and S2-grid row bands of one target.  Skipped when the box has fewer GPUs; the
single-GPU forms run in tests/test_gpu_ot_pair.py.  Two ranks sharing one GPU over gloo run the same protocol (count
all-reduce, -0.0 sample assembly, a rank with no unit, stitched bands) on any box with a GPU."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_ot_pair_on_n_gpus(nproc):
    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr",
           "127.0.0.1", "--master-port", str(29680 + nproc), os.path.join(ROOT, "tests", "ot_pair_worker.py")]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert f"multi-gpu ot pair OK {nproc}" in proc.stdout


def test_ot_pair_two_ranks_sharing_one_gpu():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29679", os.path.join(ROOT, "tests", "ot_pair_worker.py"), "--shared-gpu"]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert "multi-gpu ot pair OK 2" in proc.stdout
