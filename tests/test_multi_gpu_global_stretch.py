"""The percentile stretch over a global fit (stretch_scope="fit") in BASELINE.json configs[3] and configs[4] on N GPUs
of one node (torchrun, one process per GPU; tests/global_stretch_worker.py).  Skipped when the box has fewer GPUs; the
single-GPU forms run in tests/test_gpu_union_select.py."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_global_stretch_on_n_gpus(nproc):
    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr",
           "127.0.0.1", "--master-port", str(29580 + nproc), os.path.join(ROOT, "tests", "global_stretch_worker.py")]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert f"global stretch OK {nproc}" in proc.stdout
