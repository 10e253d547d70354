"""PairSynthesizer.matched_fine after a global fit on N GPUs of one node (torchrun, one process per GPU): granules on
their S2 targets dealt to the ranks with one rank holding none, synthesize_sharded with stretch_scope="fit", then the
10 m step with group=.  Skipped when the box has fewer GPUs; the single-GPU forms run in tests/test_gpu_fine_grid.py."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_matched_fine_on_n_gpus(nproc):
    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr",
           "127.0.0.1", "--master-port", str(29680 + nproc), os.path.join(ROOT, "tests", "fine_grid_worker.py")]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert f"multi-gpu fine grid OK {nproc}" in proc.stdout
