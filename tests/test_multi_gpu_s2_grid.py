"""BASELINE.json configs[3] (one global fit over granules on their own S2 targets) and configs[4] (a mosaic on the S2
grid in row bands with per-band ortho and raw staging) on N GPUs of one node (torchrun, one process per GPU).  Skipped
when the box has fewer GPUs; the single-GPU forms run in tests/test_gpu_s2_grid_slabs.py."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_s2_grid_configs_on_n_gpus(nproc):
    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr",
           "127.0.0.1", "--master-port", str(29640 + nproc), os.path.join(ROOT, "tests", "s2_grid_worker.py")]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert f"multi-gpu s2 grid OK {nproc}" in proc.stdout
